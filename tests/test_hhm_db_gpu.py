"""GPU tests of the HHM-text database loader (hhg_db_create_hhm: SURVEY 8a rows a10 + a11, 8f-1).
The column records it leaves in HBM must be bit-identical to (1) the oracle's restatement of HMM::Read +
PrepareTemplateHMM, (2) the reference's goldens, (3) the compiled reference when it is shipped; a search over the
loaded shard must equal a search over a shard built from the reference's own prepared arrays."""
import os

import numpy as np
import pytest

from tests.util import ROOT, bits, golden, ref_data_path

pytestmark = pytest.mark.gpu


def _pp(G):
    from hhsuite_b200.capi import PrepParams
    v = G["prep_params"]
    return PrepParams(*[float(x) for x in v[:7]], int(v[7]), *[float(x) for x in v[8:]])


def _opp(G):
    from oracle.binding import PrepParams
    v = G["prep_params"]
    return PrepParams(*[float(x) for x in v[:7]], int(v[7]), *[float(x) for x in v[8:]])


def _pack(texts):
    data = b"".join(t + b"\0" for t in texts)
    ln = np.array([len(t) + 1 for t in texts], np.int64)
    off = np.concatenate([[0], np.cumsum(ln)[:-1]]).astype(np.int64)
    return data, off, ln


def _expected_records(p, tr, ss, any_ss):
    """ColRec layout of include/hhg.h from reference-layout p[(L+2),20], tr[(L+1),7], ss[L+2]."""
    from hhsuite_b200.capi import COLREC_DTYPE
    L = p.shape[0] - 2
    r = np.zeros(L, COLREC_DTYPE)
    r["p"] = p[1:L + 1]
    r["m2m"], r["m2d"], r["d2m"], r["d2d"], r["i2m"] = tr[:L, 0], tr[:L, 2], tr[:L, 5], tr[:L, 6], tr[:L, 3]
    r["i2i"], r["m2i"] = tr[1:L + 1, 4], tr[1:L + 1, 1]
    r["ss"] = ss[1:L + 1] if any_ss else 0
    return r


def _texts(G, extra_seed=0, n_extra=9):
    from hhsuite_b200 import synth
    rng = np.random.default_rng(900 + extra_seed)
    texts = [G["hhm_ss60_text"].tobytes(), G["hhm_t150_text"].tobytes()]
    for k in range(n_extra):
        L = int(rng.integers(1, 420))
        texts.append(synth.hhm_text(L, 5000 + 31 * extra_seed + k, f"r{k}", with_ss=bool(k % 3 == 0)).encode())
    texts.append(synth.hhm_text(1, 4242, "one").encode())
    return texts


def test_loaded_records_equal_oracle_and_goldens(hhg, gpu_ctx, oracle):
    G = golden()
    texts = _texts(G)
    data, off, ln = _pack(texts)
    db = hhg.TargetDB.from_hhm(gpu_ctx, data, off, ln, G["R"], _pp(G))
    cols = db.read_cols(0)
    pav = db.read_pav()
    assert db.n == len(texts) and len(cols) == int(db.Lh.sum())
    pos = 0
    for k, t in enumerate(texts):
        rec = oracle.hhm_parse(t)
        out = oracle.hhm_prepare(rec, oracle.null_to_pb(rec["null"]), G["R"], _opp(G))
        L = out["L"]
        assert db.Lh[k] == L
        want = _expected_records(out["p"], out["tr"], out["ss"], True)
        got = cols[pos:pos + L]
        assert got.tobytes() == want.tobytes(), f"record {k} (L={L}) differs from the oracle"
        assert np.array_equal(bits(pav[k]), bits(out["pav"])), k
        pos += L
    # the two records whose reference outputs are committed as goldens
    w = _expected_records(G["hhm_ss60_praw"], G["hhm_ss60_tr"], G["hhm_ss60_ss"], True)
    assert cols[:60].tobytes() == w.tobytes() and np.array_equal(bits(pav[0]), bits(G["hhm_ss60_pav"]))
    w = _expected_records(G["nm_t150_praw"], G["nm_t150_tr"], np.zeros(152, np.uint8), True)
    assert cols[60:210].tobytes() == w.tobytes() and np.array_equal(bits(pav[1]), bits(G["nm_t150_pav"]))
    db.close()


def test_loaded_records_equal_compiled_reference(hhg, gpu_ctx, refshim, tmp_path):
    G = golden()
    qpath = ref_data_path("query.hhm")
    refshim.load_query_hhm(qpath)
    texts = _texts(G, extra_seed=1, n_extra=5) + [open(qpath, "rb").read()]
    data, off, ln = _pack(texts)
    db = hhg.TargetDB.from_hhm(gpu_ctx, data, off, ln, refshim.R(), None)     # default parameters
    cols, pav = db.read_cols(0), db.read_pav()
    pos = 0
    for k, t in enumerate(texts):
        f = tmp_path / f"t{k}.hhm"
        f.write_bytes(t)
        ref = refshim.prepare_template_hhm_raw(str(f))
        # a fresh reference HMM leaves ss_pred/ss_conf unset when the record has no ss_pred sequence
        ss = refshim.prepare_template_hhm(str(f))["ss"] if hhg.capi.hhm_scan(t)[1] else np.zeros(ref["L"] + 2, np.uint8)
        L = ref["L"]
        want = _expected_records(ref["p_raw"], ref["tr"], ss, True)
        assert cols[pos:pos + L].tobytes() == want.tobytes(), k
        assert np.array_equal(bits(pav[k]), bits(ref["pav"])), k
        pos += L
    db.close()


@pytest.mark.parametrize("columnscore", [1, 2])
def test_search_over_loaded_shard_equals_reference_prepared_shard(hhg, gpu_ctx, columnscore):
    """data/query.hhm (golden query) vs the HHM text of synth150: hits through text loader + device null model ==
    hits over the reference-prepared profile == the golden Viterbi result."""
    G = golden()
    gpu_ctx.set_query(G["q_p"], G["q_tr"])
    data, off, ln = _pack([G["hhm_t150_text"].tobytes()])
    db = hhg.TargetDB.from_hhm(gpu_ctx, data, off, ln, G["R"], _pp(G))
    with pytest.raises(hhg.HhgError):
        hhg.viterbi_search(gpu_ctx, db)                 # null model not applied yet
    db.apply_null_model(q_pav=G["q_pav"], pb=G["pb"], columnscore=columnscore)
    h1, p1 = hhg.viterbi_search(gpu_ctx, db)
    db_ref = hhg.TargetDB.from_profiles(gpu_ctx, [(G[f"nm_t150_p_cs{columnscore}"], G["nm_t150_tr"], None)])
    h2, p2 = hhg.viterbi_search(gpu_ctx, db_ref)
    assert h1.tobytes() == h2.tobytes() and np.array_equal(p1, p2)
    if columnscore == 1:                                 # the default pipeline = golden config 1
        assert bits(h1["score"][0]) == bits(G["t150_score"][0]) and bits(h1["hit_score"][0]) == bits(G["t150_score"][1])
        assert (h1["i2"][0], h1["j2"][0], h1["nsteps"][0]) == tuple(G["t150_res"][:3])
    # prepared records can be read back too
    assert len(db.read_cols(1)) == 150
    db.close(); db_ref.close()


def test_packed_format_roundtrip_and_chunks(hhg, gpu_ctx, monkeypatch):
    """read_cols/read_pav -> from_packed reproduces the shard; many records exercise the multi-threaded tokeniser."""
    from hhsuite_b200 import synth
    G = golden()
    rng = np.random.default_rng(5)
    uniq = [synth.hhm_text(int(rng.integers(20, 300)), 8000 + k, f"u{k}", with_ss=False).encode() for k in range(12)]
    texts = [uniq[int(rng.integers(0, 12))] for _ in range(700)]
    data, off, ln = _pack(texts)
    db = hhg.TargetDB.from_hhm(gpu_ctx, data, off, ln, G["R"], _pp(G))
    cols, pav = db.read_cols(0), db.read_pav()
    # identical text -> identical records wherever it sits
    first = {}
    pos = 0
    for k, t in enumerate(texts):
        L = int(db.Lh[k])
        blob = cols[pos:pos + L].tobytes() + pav[k].tobytes()
        assert first.setdefault(t, blob) == blob, k
        pos += L
    db2 = hhg.TargetDB.from_packed(gpu_ctx, db.Lh, cols, pav)
    assert db2.read_cols(0).tobytes() == cols.tobytes() and np.array_equal(db2.read_pav(), pav)
    gpu_ctx.set_query(G["q_p"], G["q_tr"])
    for d in (db, db2):
        d.apply_null_model(q_pav=G["q_pav"], columnscore=1)
    h1, _ = hhg.viterbi_search(gpu_ctx, db)
    h2, _ = hhg.viterbi_search(gpu_ctx, db2)
    assert h1.tobytes() == h2.tobytes()
    db.close(); db2.close()


def test_loader_errors(hhg, gpu_ctx):
    from hhsuite_b200.capi import PrepParams
    G = golden()
    good = G["hhm_ss60_text"].tobytes()
    bad = good.replace(b"LENG  60", b"LENG  61")
    data, off, ln = _pack([good, bad])
    with pytest.raises(hhg.HhgError, match="record 1"):
        hhg.TargetDB.from_hhm(gpu_ctx, data, off, ln, G["R"], _pp(G))
    pp = PrepParams.defaults()
    pp.pcm = 4                                            # there is no such mode (src/hhhmm.cpp:1885-1918: 0..3)
    data, off, ln = _pack([good])
    with pytest.raises(hhg.HhgError, match="mode 4"):
        hhg.TargetDB.from_hhm(gpu_ctx, data, off, ln, G["R"], pp)


def test_dropin_with_text_loader(tmp_path):
    """The reference's own ViterbiRunner (reading the HHM files itself) against the GPU adapter whose templates were
    loaded by hhg_db_create_hhm from the same files: every Hit identical."""
    import subprocess
    from hhsuite_b200 import synth
    binp = os.path.join(ROOT, "oracle", "_ref", "hh_dropin_check")
    qpath = os.path.join(ROOT, "oracle", "_ref", "data", "query.hhm")
    if not (os.path.exists(binp) and os.path.exists(qpath)):
        pytest.skip("oracle/_ref/hh_dropin_check not built/shipped")
    files = []
    for k, L in enumerate([150, 60, 431, 300, 33, 200, 97, 120, 250, 75]):
        f = tmp_path / f"t{k}.hhm"
        f.write_text(synth.hhm_text(L, 100 + k, f"t{k}"))
        files.append(str(f))
    r = subprocess.run([binp, "--hhm-loader", qpath, qpath] + files, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "all hits identical" in r.stdout and "hhg_db_create_hhm" in r.stdout, r.stdout + r.stderr
    # SS variant
    q = tmp_path / "q.hhm"
    q.write_text(synth.hhm_text(180, 7, "qss", with_ss=True))
    files = []
    for k, L in enumerate([180, 90, 140, 260, 45, 180, 75, 200, 66]):
        f = tmp_path / f"s{k}.hhm"
        f.write_text(synth.hhm_text(L, 7 if k in (0, 5) else 300 + k, f"s{k}", with_ss=True))
        files.append(str(f))
    r = subprocess.run([binp, "--hhm-loader", str(q)] + files, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "all hits identical" in r.stdout, r.stdout + r.stderr


def test_query_from_hhm_equals_reference_prepare_query(hhg, gpu_ctx, refshim, tmp_path):
    """hhg_query_from_hhm = HMM::Read + PrepareQueryHMM with par.nocontxt (src/hhfunc.cpp:121-160): p (all rows incl. 0
    and L+1), the complete transition rows, ss, pav and Neff_HMM bit-identical to the reference's query."""
    from hhsuite_b200 import synth
    cases = [ref_data_path("query.hhm")]
    for k, (L, ss) in enumerate([(1, False), (57, True), (300, False)]):
        f = tmp_path / f"q{k}.hhm"
        f.write_text(synth.hhm_text(L, 70 + k, f"q{k}", with_ss=ss))
        cases.append(str(f))
    for path in cases:
        ref = refshim.load_query_hhm(path)
        rec = open(path, "rb").read() + b"\0"
        got = hhg.capi.query_from_hhm(gpu_ctx, rec, refshim.R())
        assert got["L"] == ref["L"]
        assert np.array_equal(got["p"].view(np.uint32), ref["p"].view(np.uint32)), path
        assert np.array_equal(got["tr"].view(np.uint32), ref["tr"].view(np.uint32)), path
        assert np.array_equal(got["pav"].view(np.uint32), ref["pav"].view(np.uint32))
        if got["has_ss"]:
            assert np.array_equal(got["ss"][1:-1], ref["ss"][1:-1])
        assert np.float32(got["neff"]).view(np.uint32) == np.float32(ref["neff"]).view(np.uint32)


@pytest.mark.parametrize("pc", [(2, 1.0, 1.5, 0.5), (2, 0.9, 2.0, 1.7), (3, 1.0, 12.0, 0.3), (1, 0.35, 1.5, 1.0), (0, 1.0, 1.5, 1.0)],
                         ids=["pcm2-pcc0.5", "pcm2-pcc1.7", "pcm3", "pcm1", "pcm0"])
def test_every_pseudocount_mode_equals_compiled_reference(hhg, gpu_ctx, refshim, tmp_path, pc):
    """HMM::AddAminoAcidPseudocounts modes 0..3 (src/hhhmm.cpp:1874-1921) incl. mode 2 with pcc != 1, whose pow() is the C
    library's powf (tau computed per column on the host with the same libm) and the constant-diversity mode 3."""
    G = golden()
    qpath = ref_data_path("query.hhm")
    refshim.load_query_hhm(qpath)
    texts = _texts(G, extra_seed=2, n_extra=4)
    data, off, ln = _pack(texts)
    pp = hhg.capi.PrepParams.defaults()
    pp.pcm, pp.pca, pp.pcb, pp.pcc = pc
    refshim.set_pc(*pc)
    try:
        db = hhg.TargetDB.from_hhm(gpu_ctx, data, off, ln, refshim.R(), pp)
        cols, pav = db.read_cols(0), db.read_pav()
        pos = 0
        for k, t in enumerate(texts):
            f = tmp_path / f"t{k}.hhm"
            f.write_bytes(t)
            ref = refshim.prepare_template_hhm_raw(str(f))
            L = ref["L"]
            got_p = np.stack([cols["p"][pos + j] for j in range(L)])
            assert np.array_equal(got_p.view(np.uint32), ref["p_raw"][1:L + 1].view(np.uint32)), (k, pc)
            assert np.array_equal(bits(pav[k]), bits(ref["pav"])), k
            pos += L
        db.close()
    finally:
        refshim.set_pc(2, 1.0, 1.5, 1.0)
