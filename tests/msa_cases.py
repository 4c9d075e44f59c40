"""Synthetic A3M alignments shared by the alignment -> HMM tests (CPU scanner test and GPU parity tests)."""
import os

CASES = [  # (match columns, sequences after the master, seed, generator options)
    (50, 20, 1, {}),
    (8, 5, 2, {}),                                    # fewer than NCOLMIN columns: global weights everywhere
    (120, 300, 3, dict(with_ss=True)),
    (200, 60, 4, dict(with_comment=True)),
    (80, 40, 5, dict(consensus_first=True)),          # compressed databases: consensus row outside the profile
    (30, 0, 6, {}),                                   # single sequence
    (300, 150, 7, dict(ident=0.9, dup_frac=0.6)),     # most rows removed by the 90 % identity filter
    (15, 3, 8, dict(with_ss=True, with_comment=True)),
    (60, 1, 9, {}),
    (431, 58, 10, dict(ident=0.3)),
    (700, 90, 11, dict(ident=0.6, with_ss=True)),
    (90, 25, 12, dict(with_ss=True, ss_conf=False)),  # ss_pred without ss_conf: confidence 5 everywhere
]


# hand-written corner cases (CPU tests): a single sequence with fewer than six match states falls back to "-M first"
# (src/hhalignment.cpp:861-880): lower-case letters become match states, '-' columns do not
TINY = [b">master\nZ-iwHkv\n", b"#NAME some description\n>master\nlKV\n", b">ss_pred\nHHEC-\n>ss_conf\n12345\n>m\nAc-dE\n",
        b">m\r\nACDEFGHIKL\r\n>s1 x\r\nAC-EFGHIKL\r\n>s2\r\n.ACDEFGaaHIKL\r\n"]


def texts():
    from hhsuite_b200 import synth
    out = [synth.a3m_text(L, n, seed, **kw).encode() for (L, n, seed, kw) in CASES]
    from tests.util import ref_data
    out.append(ref_data("query.a3m"))
    return out


CA3M_CASES = [(50, 20, 21, {}), (120, 200, 22, dict(ident=0.8, dup_frac=0.5)), (300, 40, 23, {}),
              (260, 30, 25, dict(ident=0.4)), (9, 6, 26, {})]


def ca3m_database(directory):
    """A small compressed alignment database (<dir>/db_ca3m|_sequence|_header .ffdata/.ffindex) made from synthetic
    alignments.  Returns (prefix, names in index order)."""
    from hhsuite_b200 import ffindex, synth
    prefix = os.path.join(str(directory), "db")
    recs, seqs, heads = [], [], []
    for (L, n, seed, kw) in CA3M_CASES:
        a = synth.a3m_text(L, n, seed, name=f"al{seed}", **kw)
        ca, sq, hd = synth.a3m_to_ca3m(a, seq_index_base=len(seqs))
        recs.append((f"al{seed}", ca)); seqs += sq; heads += hd
    names = [f"s{i:06d}" for i in range(len(seqs))]
    ffindex.write_ffindex(prefix + "_ca3m.ffdata", recs)
    ffindex.write_ffindex(prefix + "_sequence.ffdata", list(zip(names, seqs)))
    ffindex.write_ffindex(prefix + "_header.ffdata", list(zip(names, heads)))
    return prefix
