"""CPU tests of the HHM-text loader (SURVEY 8a rows a10/a11): the oracle's restatement of HMM::Read +
PrepareTemplateHMM against the reference (goldens, and the compiled reference when present), and the product's
host tokeniser against the oracle's."""
import numpy as np
import pytest

from tests.util import bits, golden


def _params(G):
    from oracle.binding import PrepParams
    v = G["prep_params"]
    return PrepParams(*[float(x) for x in v[:7]], int(v[7]), *[float(x) for x in v[8:]])


@pytest.mark.parametrize("name,gp,gtr,gpav", [("hhm_ss60_text", "hhm_ss60_praw", "hhm_ss60_tr", "hhm_ss60_pav"),
                                               ("hhm_t150_text", "nm_t150_praw", "nm_t150_tr", "nm_t150_pav")])
def test_oracle_prepare_equals_reference_goldens(oracle, name, gp, gtr, gpav):
    G = golden()
    text = G[name].tobytes()
    rec = oracle.hhm_parse(text)
    out = oracle.hhm_prepare(rec, oracle.null_to_pb(rec["null"]), G["R"], _params(G))
    assert out["L"] == G[gp].shape[0] - 2
    assert np.array_equal(bits(out["p"]), bits(G[gp]))
    assert np.array_equal(bits(out["tr"]), bits(G[gtr]))
    assert np.array_equal(bits(out["pav"]), bits(G[gpav]))
    if name == "hhm_ss60_text":
        assert rec["has_ss"] and np.array_equal(out["ss"][1:-1], G["hhm_ss60_ss"][1:-1])


def test_oracle_fast_log2_table_equals_reference(oracle):
    G = golden()
    x = ((np.arange(1024, dtype=np.uint32) << 13) | np.uint32(0x3F800000)).view(np.float32)
    mine = np.array([oracle.fast_log2(float(v)) for v in x], np.float32)
    assert np.array_equal(bits(mine), bits(G["fastlog2_lg2"]))


@pytest.mark.parametrize("seed", [1, 2, 3, 4])
def test_oracle_prepare_equals_compiled_reference(oracle, refshim, tmp_path, seed):
    from hhsuite_b200 import synth
    rng = np.random.default_rng(seed)
    refshim.load_query_hhm(str(_query_path()))
    R, pp = refshim.R(), refshim.prep_params()
    for k in range(4):
        L = int(rng.integers(1, 500))
        ss = bool(rng.integers(0, 2))
        f = tmp_path / f"t{k}.hhm"
        f.write_text(synth.hhm_text(L, 1000 * seed + k, f"t{k}", with_ss=ss))
        rec = oracle.hhm_parse(f.read_bytes())
        out = oracle.hhm_prepare(rec, oracle.null_to_pb(rec["null"]), R, pp)
        ref = refshim.prepare_template_hhm_raw(str(f))
        ref_ss = refshim.prepare_template_hhm(str(f))["ss"]
        assert out["L"] == ref["L"] == L
        assert np.array_equal(bits(out["p"]), bits(ref["p_raw"]))
        assert np.array_equal(bits(out["tr"]), bits(ref["tr"]))
        assert np.array_equal(bits(out["pav"]), bits(ref["pav"]))
        if ss:      # a fresh reference HMM leaves ss_pred/ss_conf unset otherwise
            assert np.array_equal(out["ss"][1:-1], ref_ss[1:-1])
        else:
            assert not out["ss"].any()


def _query_path():
    from tests.util import ref_data_path
    return ref_data_path("query.hhm")


def test_product_tokeniser_equals_oracle(oracle):
    """hhg_hhm_parse (the host half of hhg_db_create_hhm; no GPU needed) against the oracle's parser."""
    from hhsuite_b200 import capi, synth
    G = golden()
    texts = [G["hhm_ss60_text"].tobytes(), G["hhm_t150_text"].tobytes(), open(_query_path(), "rb").read()]
    texts += [synth.hhm_text(L, 70 + k, f"x{k}", with_ss=ss).encode()
              for k, (L, ss) in enumerate([(1, False), (2, True), (333, False), (800, True)])]
    texts.append(texts[0] + b"\0trailing garbage that an ffindex neighbour would be")
    for t in texts:
        a, b = capi.hhm_parse(t), oracle.hhm_parse(t)
        L = a["L"]
        assert L == b["L"] and a["has_ss"] == b["has_ss"] and a["has_pc"] == b["has_pc"]
        assert a["neff_hmm"] == b["neff_hmm"]
        assert np.array_equal(a["f"], b["f"][1:L + 1]) and np.array_equal(a["tr"], b["tr"])
        nb = b["neff"].copy()
        nb[1:, 0] = np.where(nb[1:, 0] == 0, 1000, nb[1:, 0])      # Neff_M == 0 -> 1 is folded into the integers
        assert np.array_equal(a["neff"], nb)
        assert np.array_equal(a["ss"], b["ss"][1:-1]) and np.array_equal(a["null"], b["null"])


def test_product_tokeniser_rejects_malformed_records():
    from hhsuite_b200 import capi
    G = golden()
    good = G["hhm_ss60_text"].tobytes()
    with pytest.raises(capi.HhgError, match="LENG"):
        capi.hhm_scan(b"this is not an HHM record\n")
    cut = good[:good.index(b"\nHMM ") + 2000]                    # truncated inside the column block
    with pytest.raises(capi.HhgError, match="fewer columns|short|missing|fewer than"):
        capi.hhm_parse(cut)
    nonull = good.replace(b"\nNULL ", b"\nXULL ")
    with pytest.raises(capi.HhgError, match="NULL"):
        capi.hhm_parse(nonull)
    more = good.replace(b"LENG  60", b"LENG  59")
    assert more != good
    with pytest.raises(capi.HhgError, match="more columns"):
        capi.hhm_parse(more)


def test_ffindex_roundtrip(tmp_path):
    from hhsuite_b200 import ffindex
    recs = [("zeta", b"abc\ndef"), ("alpha", b"x"), ("mid", b"")]
    ffindex.write_ffindex(str(tmp_path / "db_hhm.ffdata"), recs)
    ff = ffindex.FFIndex(str(tmp_path / "db_hhm.ffdata"))
    assert ff.names == ["alpha", "mid", "zeta"] and len(ff) == 3
    got = {n: ff.record(k) for k, n in enumerate(ff.names)}
    assert got == {n: b + b"\0" for n, b in recs}
    ff.close()


def test_cs219_ffindex_arrays(tmp_path):
    """init_prefilter's view of a binary cs219 database: length = entry length - 1, pointers into the data file."""
    from hhsuite_b200 import ffindex
    rng = np.random.default_rng(4)
    seqs = {f"s{k:03d}": rng.integers(0, 219, int(L), dtype=np.uint8).tobytes() for k, L in enumerate([5, 1, 300, 77])}
    ffindex.write_ffindex(str(tmp_path / "db_cs219.ffdata"), list(seqs.items()))
    ff = ffindex.FFIndex(str(tmp_path / "db_cs219.ffdata"))
    L, off, seq = ffindex.cs219_arrays(ff)
    assert L.tolist() == [len(seqs[n]) for n in ff.names]
    for k, n in enumerate(ff.names):
        assert seq[off[k]:off[k] + L[k]].tobytes() == seqs[n] and seq[off[k] + L[k]] == 0
    ff.close()
    ffindex.write_ffindex(str(tmp_path / "old_cs219.ffdata"), [("a", b">a\nABCDEF")])
    ff = ffindex.FFIndex(str(tmp_path / "old_cs219.ffdata"))
    with pytest.raises(ValueError, match="old text format"):
        ffindex.cs219_arrays(ff)
    ff.close()


def test_tokeniser_fuzz_never_crashes_and_agrees_with_oracle(oracle):
    """Truncated / corrupted / spliced HHM records (what a damaged ffindex entry looks like): the product tokeniser
    must either refuse the record or return exactly the integers the oracle's parser reads."""
    from hhsuite_b200 import capi, synth
    G = golden()
    rng = np.random.default_rng(0)
    base = [synth.hhm_text(L, 900 + k, f"f{k}", with_ss=bool(k % 2)).encode() for k, L in enumerate([3, 17, 60])]
    base.append(G["hhm_ss60_text"].tobytes())
    accepted = rejected = 0
    for it in range(800):
        t = bytearray(base[it % len(base)])
        mode = it % 5
        if mode == 0:
            t = t[:int(rng.integers(0, len(t)))]
        elif mode == 1:
            for _ in range(int(rng.integers(1, 20))):
                t[int(rng.integers(0, len(t)))] = int(rng.integers(0, 256))
        elif mode == 2:
            lines = bytes(t).split(b"\n"); del lines[int(rng.integers(0, len(lines)))]; t = bytearray(b"\n".join(lines))
        elif mode == 3:
            lines = bytes(t).split(b"\n"); k = int(rng.integers(0, len(lines))); lines.insert(k, lines[k])
            t = bytearray(b"\n".join(lines))
        else:
            k = int(rng.integers(0, len(t)))
            t[k:k] = bytes(rng.integers(0, 256, int(rng.integers(1, 50)), dtype=np.uint8))
        t = bytes(t)
        if not t:
            continue
        try:
            a = capi.hhm_parse(t)
        except capi.HhgError:
            rejected += 1
            continue
        accepted += 1
        try:
            b = oracle.hhm_parse(t, maxL=a["L"] + 5)
        except ValueError:
            continue
        if b["L"] == a["L"]:
            assert np.array_equal(a["f"], b["f"][1:a["L"] + 1]) and np.array_equal(a["tr"], b["tr"]), it
    assert accepted > 100 and rejected > 100
