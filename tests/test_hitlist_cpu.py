"""Hit-list statistics of the library (hhg_hitlist_*: host side, SURVEY 8a row a13) against the compiled reference's
HitList::CalculatePvalues / CalculateHHblitsEvalues / SortList and against committed goldens generated from it
(tests/golden/make_golden.py).  Bar: every double and float bit-identical, same order."""
import ctypes as C
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "hitlist_v1.npz")

STATS = np.dtype([("Pval", np.float64), ("logPval", np.float64), ("Eval", np.float64), ("logEval", np.float64),
                  ("score_aass", np.float32), ("Probab", np.float32), ("lamda", np.float32), ("mu", np.float32)])


def product_stats(score, score_ss, L, neff, qL, qneff, N, loc, ssm, ssw, ssm2=None, files=None, hhblits=None):
    import hhsuite_b200 as hh
    lib = hh.capi.load()
    n = len(score)
    out = np.zeros(n, STATS)
    f32 = lambda a: np.ascontiguousarray(a, np.float32)   # noqa: E731
    i32 = lambda a: None if a is None else np.ascontiguousarray(a, np.int32)   # noqa: E731
    p = hh.capi._p
    s, ss, Lt, ne, s2 = f32(score), f32(score_ss), i32(L), f32(neff), i32(ssm2)
    lib.hhg_hitlist_pvalues.argtypes = [C.c_int, hh.capi.c_f32p, hh.capi.c_f32p, hh.capi.c_i32p, hh.capi.c_f32p,
                                        hh.capi.c_i32p, C.c_int, C.c_float, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p]
    assert lib.hhg_hitlist_pvalues(n, p(s, hh.capi.c_f32p), p(ss, hh.capi.c_f32p), p(Lt, hh.capi.c_i32p),
                                   p(ne, hh.capi.c_f32p), p(s2, hh.capi.c_i32p), qL, qneff, N, loc, ssm, ssw,
                                   out.ctypes.data_as(C.c_void_p)) == 0
    if hhblits:
        lib.hhg_hitlist_hhblits_evalues.argtypes = [C.c_int, C.c_void_p, hh.capi.c_f32p, C.c_float, C.c_int, C.c_float,
                                                    C.c_float, C.c_float, C.c_double]
        assert lib.hhg_hitlist_hhblits_evalues(n, out.ctypes.data_as(C.c_void_p), p(ne, hh.capi.c_f32p), qneff,
                                               hhblits["dbsize"], 0.4, 0.02, 0.1, hhblits["thresh"]) == 0
    order = np.zeros(n, np.int32)
    farr = None if files is None else (C.c_char_p * n)(*[f.encode() for f in files])
    lib.hhg_hitlist_order.argtypes = [C.c_int, C.c_void_p, C.c_void_p, hh.capi.c_i32p]
    assert lib.hhg_hitlist_order(n, out.ctypes.data_as(C.c_void_p), farr, p(order, hh.capi.c_i32p)) == 0
    return out, order


def cases():
    rng = np.random.default_rng(77)
    n = 400
    score = np.concatenate([rng.uniform(-5, 60, n - 40), rng.uniform(60, 1500, 30), rng.uniform(-30, 0, 10)]).astype(np.float32)
    score_ss = rng.uniform(-3, 12, n).astype(np.float32)
    L = rng.integers(20, 2500, n).astype(np.int32)
    neff = rng.uniform(1.0, 14.0, n).astype(np.float32)
    ssm2 = rng.integers(0, 2, n).astype(np.int32)
    files = [f"dir/t{int(k) % 97:03d}" for k in rng.integers(0, 10 ** 6, n)]
    score[5] = score[6]; score_ss[5] = score_ss[6]; L[5] = L[6]; neff[5] = neff[6]; ssm2[5] = ssm2[6]   # tie: file decides
    files[5], files[6] = "zz", "aa"
    out = []
    for (qL, qneff, N, loc, ssm, ssw, hb) in [(431, 6.3, 5000, 1, 2, 0.11, None), (60, 1.0, 1, 1, 0, 0.0, None),
                                               (1500, 11.7, 1000000, 1, 2, 0.11, dict(dbsize=1000000, thresh=1000.0)),
                                               (300, 4.0, 20000, 0, 2, 0.11, None), (300, 4.0, 20000, 0, 0, 0.0, None),
                                               (400, 9.9, 0, 1, 4, 0.2, dict(dbsize=52000, thresh=0.1))]:
        out.append(dict(score=score, score_ss=score_ss, L=L, neff=neff, ssm2=ssm2, files=files, qL=qL, qneff=qneff, N=N,
                        loc=loc, ssm=ssm, ssw=ssw, hb=hb))
    return out


def _check(st, order, ref, files):
    for f in ("Pval", "logPval", "Eval", "logEval"):
        assert np.array_equal(st[f].view(np.uint64), np.asarray(ref[f]).view(np.uint64)), f
    for f in ("score_aass", "Probab"):
        assert np.array_equal(st[f].view(np.uint32), np.asarray(ref[f], np.float32).view(np.uint32)), f
    # same order wherever the reference's key is strict (its quicksort leaves exact duplicates in arbitrary order)
    ro = np.asarray(ref["order"])
    key = lambda o: [(float(st["score_aass"][k]), files[k]) for k in o]   # noqa: E731
    assert key(order) == key(ro)


def test_hitlist_stats_match_compiled_reference(refshim):
    for c in cases():
        ref = refshim.hitlist_stats(c["score"], c["score_ss"], c["L"], c["neff"], c["qL"], c["qneff"], c["N"], c["loc"],
                                    c["ssm"], c["ssw"], c["ssm2"], c["files"], hhblits=c["hb"] is not None,
                                    dbsize=(c["hb"] or {}).get("dbsize", 1), pf_evalue_thresh=(c["hb"] or {}).get("thresh", 1.0))
        st, order = product_stats(c["score"], c["score_ss"], c["L"], c["neff"], c["qL"], c["qneff"], c["N"], c["loc"],
                                  c["ssm"], c["ssw"], c["ssm2"], c["files"], c["hb"])
        _check(st, order, ref, c["files"])


@pytest.mark.skipif(not os.path.exists(GOLD), reason="golden file missing")
def test_hitlist_stats_match_goldens():
    G = np.load(GOLD)
    for i, c in enumerate(cases()):
        st, order = product_stats(c["score"], c["score_ss"], c["L"], c["neff"], c["qL"], c["qneff"], c["N"], c["loc"],
                                  c["ssm"], c["ssw"], c["ssm2"], c["files"], c["hb"])
        ref = {f: G[f"c{i}_{f}"] for f in ("Pval", "logPval", "Eval", "logEval", "score_aass", "Probab", "order")}
        _check(st, order, ref, c["files"])


def test_early_stop_sum_matches_compiled_reference(refshim):
    """ViterbiRunner::calculateEarlyStop (float arithmetic, src/hhviterbirunner.cpp:213-247): same float bits."""
    import hhsuite_b200 as hh
    rng = np.random.default_rng(3)
    for n, qL, qneff, pf, dbsize in [(2000, 400, 7.3, True, 1000000), (2000, 60, 1.0, False, 52000), (137, 1500, 12.0, True, 20000)]:
        score = rng.uniform(-5, 40, n).astype(np.float32)
        score[:5] = rng.uniform(100, 900, 5)
        L = rng.integers(20, 2000, n).astype(np.int32)
        neff = rng.uniform(1, 13, n).astype(np.float32)
        a = hh.capi.early_stop_sum(score, L, neff, qL, qneff, pf, dbsize)
        b = refshim.early_stop(score, L, neff, qL, qneff, pf, dbsize)
        assert np.float32(a).view(np.uint32) == np.float32(b).view(np.uint32), (a, b)


def test_cs219_library_parser_matches_reference(refshim):
    """hhg_cs219_parse (Prefilter ctor: ContextLibrary read + TransformToLin, src/hhprefilter.cpp:28-47) on the
    reference's own cs219.lib: every float equal to what the compiled reference holds and to the golden copy."""
    import hhsuite_b200 as hh
    from tests.util import golden, ref_data
    lib = hh.capi.cs219_parse(ref_data("cs219.lib"))
    assert lib.shape == (219, 20)
    assert np.array_equal(lib.view(np.uint32), refshim.cs219().view(np.uint32))
    assert np.array_equal(lib.view(np.uint32), np.ascontiguousarray(golden()["cs219_lin"], np.float32).view(np.uint32))
