"""CPU tests of the context-specific (CRF) query pseudocounts: the parser of the `.crf` text and the host tail
(log-sum-exp over the states, admixture, normalisation) against the compiled reference's CrfPseudocounts engine.
The context scores the CUDA kernel produces are restated here with numpy in the same summation order."""
import numpy as np
import pytest

from tests.util import CRF_SAMPLE, bits, ref_data, ref_data_path


def _scores(crf, f, neff_m):
    L = f.shape[0] - 2
    K, W = crf.n_states, crf.window
    c = (W - 1) // 2
    Wt = np.zeros((W, 20, K)); bias = np.zeros(K)
    for k in range(K):
        w, b = crf.state(k)
        Wt[:, :, k] = w; bias[k] = b
    counts = (f[1:L + 1] * neff_m[1:L + 1, None]).astype(np.float32).astype(np.float64)
    score = np.zeros((L, K))
    for i in range(L):
        sc = np.zeros(K)
        for ci in range(max(0, i - c), min(L, i + c + 1)):
            for a in range(20):
                sc = sc + Wt[ci - i + c, a, :] * counts[ci, a]
        score[i] = bias + sc
    return score


def test_crf_parser_and_tail_equal_reference(refshim):
    from hhsuite_b200 import capi, synth
    crf = capi.Crf(None, ref_data(CRF_SAMPLE))
    assert refshim.set_contxt(ref_data_path(CRF_SAMPLE)) == 100
    assert (crf.n_states, crf.window) == (100, 13)
    pc = crf.pc()
    for k in (0, 1, 50, 99):
        n, rpc, rb, rw = refshim.crf_state(k)
        w, b = crf.state(k)
        assert n == 100 and b == rb and np.array_equal(w.view(np.uint64), rw.view(np.uint64))
        assert np.array_equal(pc[k].view(np.uint64), rpc.view(np.uint64))       # long-double sum + log of UpdatePseudocounts
    rng = np.random.default_rng(3)
    L = 24
    f = rng.dirichlet(np.full(20, 0.3), L + 2).astype(np.float32)
    f[3] = 0; f[3, 7] = 1.0                                                        # a fully conserved column
    neff_m = np.concatenate([[99.999], rng.uniform(1.0, 9.0, L)]).astype(np.float32)
    neff_m[5] = 1.0
    score = _scores(crf, f, neff_m)
    for engine, adm in ((0, capi.Admix.hhm()), (1, capi.Admix.prefilter())):
        got = crf.tail_host(score, f, neff_m, adm)
        ref, _ = refshim.context_pc(f, neff_m, 4.2, engine=engine)
        assert np.array_equal(bits(got[1:L + 1]), bits(ref[1:L + 1])), engine
    crf.close()


def test_crf_parser_errors():
    from hhsuite_b200 import capi
    with pytest.raises(capi.HhgError):
        capi.Crf(None, b"NOT A CRF\n")
    with pytest.raises(capi.HhgError):
        capi.Crf(None, b"CRF\nSIZE\t2\nLENG\t3\nCrfState\nBIAS\t-1.0\nLENG\t3\nALPH\t20\nWEIGHTS\n1\t" + b"\t".join([b"1"] * 20) + b"\n//\n")
