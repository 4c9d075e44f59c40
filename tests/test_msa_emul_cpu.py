"""The product's alignment -> HMM kernels (hh-suite_b200/csrc/hhg_msa.cuh, unmodified source) executed on the CPU by
the multi-warp host emulation in tests/emul/cuda_emul_mw.h and compared bit for bit with the compiled reference's
Alignment::Filter + FrequenciesAndTransitions.  This is how the kernels are checked in the authoring container before
GPU minutes are spent (it caught a warp-divergent early exit ahead of a shuffle that hangs real hardware)."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

from tests import msa_cases
from tests.util import ROOT, bits

EMUL_DIR = os.path.join(ROOT, "tests", "emul")
LIB = os.path.join(EMUL_DIR, "libmsaemul.so")


@pytest.fixture(scope="module")
def emul():
    srcs = [os.path.join(EMUL_DIR, "msa_emul.cpp"), os.path.join(EMUL_DIR, "cuda_emul_mw.h"),
            os.path.join(ROOT, "hh-suite_b200", "csrc", "hhg_msa.cuh"), os.path.join(ROOT, "hh-suite_b200", "csrc", "hhg_math.cuh"),
            os.path.join(ROOT, "hh-suite_b200", "csrc", "hhg_crf.cuh")]
    if not os.path.exists(LIB) or any(os.path.getmtime(s) > os.path.getmtime(LIB) for s in srcs):
        subprocess.check_call(["g++", "-O1", "-std=c++20", "-ffp-contract=off", "-fPIC", "-shared", "-pthread", "-DHHG_EMUL",
                               "-o", LIB, srcs[0]])
    L = C.CDLL(LIB)
    L.emul_msa_to_hmm.argtypes = [C.c_char_p, C.c_longlong, C.c_void_p, C.c_float] + [C.c_void_p] * 4 + [C.c_int] + [C.c_void_p] * 7
    return L


def _tables():
    """fast_log2's lg2 / diff tables as the library builds them (double log, src/util-inl.h:117-123)."""
    lg2 = np.zeros(1025, np.float32); dif = np.zeros(1025, np.float32)
    prev = np.float32(0)
    for i in range(1, 1025):
        lg2[i] = np.float32(math.log(1024 + i) * 1.442695041 - 10.0)
        dif[i - 1] = np.float32(float(np.float32(lg2[i] - prev)) * 1.2352E-4)
        prev = lg2[i]
    return lg2, dif


def _run(L, refshim, t, filt=(90, 0, 0, -20.0, 100), wg=0, threads=64, M=1, Mgaps=50):
    lg2, dif = _tables()
    ip = np.array([65535, 32765, 20001, filt[0], filt[1], filt[2], filt[4], wg, M, Mgaps], np.int32)
    Lc, Nc = 1000, 1000
    dims = np.zeros(4, np.int32); keep = np.zeros(Nc, np.int8); wgv = np.zeros(Nc, np.float32)
    f = np.zeros((Lc + 2) * 20, np.float32); tr = np.zeros((Lc + 1) * 7, np.float32)
    neff = np.zeros(3 * (Lc + 1), np.float32); nh = np.zeros(1, np.float32)
    S = np.ascontiguousarray(refshim.S(), np.float32); pb = refshim.pb()
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    rc = L.emul_msa_to_hmm(t, len(t), p(ip), C.c_float(filt[3]), p(S), p(pb), p(lg2), p(dif), threads, p(dims), p(keep),
                           p(wgv), p(f), p(tr), p(neff), p(nh))
    assert rc == 0 and dims[3] == 0
    Lm, N = int(dims[0]), int(dims[1])
    return dict(L=Lm, N_in=N, N_filtered=int(dims[2]), keep=keep[:N], wg=wgv[:N], f=f[:(Lm + 2) * 20].reshape(Lm + 2, 20),
                tr=tr[:(Lm + 1) * 7].reshape(Lm + 1, 7), neff_m=neff[:Lm + 1], neff_i=neff[Lm + 1:2 * (Lm + 1)],
                neff_d=neff[2 * (Lm + 1):3 * (Lm + 1)], neff_hmm=float(nh[0]))


def _cmp(got, ref, tag):
    assert (got["L"], got["N_in"], got["N_filtered"]) == (ref["L"], ref["N_in"], ref["N_filtered"]), tag
    assert np.array_equal(got["keep"], ref["keep"]), tag
    if ref["N_filtered"] > 1:
        assert np.array_equal(bits(got["wg"]), bits(ref["wg"])), tag
    for key in ("f", "tr", "neff_m", "neff_i", "neff_d"):
        assert np.array_equal(bits(got[key]), bits(ref[key])), (tag, key)
    assert bits(np.float32(got["neff_hmm"])) == bits(np.float32(ref["neff_hmm"])), tag


@pytest.mark.parametrize("case", [0, 1, 4, 5, 7, 8])
def test_emulated_kernels_equal_compiled_reference(emul, refshim, tmp_path, case):
    t = msa_cases.texts()[case]
    path = tmp_path / "m.a3m"
    path.write_bytes(t)
    _cmp(_run(emul, refshim, t), refshim.msa_to_hmm(str(path)), f"case {case}")


@pytest.mark.parametrize("filt,wg", [((70, 0, 30, -20.0, 0), 0), ((90, 0, 0, 0.2, 0), 0), ((50, 30, 20, 0.0, 20), 0),
                                     ((15, 0, 0, -20.0, 5), 0), ((90, 0, 0, -20.0, 100), 1)])
def test_emulated_filter_options_and_global_weights(emul, refshim, tmp_path, filt, wg):
    for case in (0, 4):
        t = msa_cases.texts()[case]
        path = tmp_path / "m.a3m"
        path.write_bytes(t)
        _cmp(_run(emul, refshim, t, filt=filt, wg=wg), refshim.msa_to_hmm(str(path), filt=filt, wg=wg), f"case {case} {filt} wg={wg}")


def test_emulated_context_score_kernel(emul, refshim):
    """k_crf_scores on the CPU emulator + the library's host tail == the compiled reference's CRF pseudocounts."""
    from hhsuite_b200 import capi
    from tests.util import CRF_SAMPLE, ref_data, ref_data_path
    crf = capi.Crf(None, ref_data(CRF_SAMPLE))
    assert refshim.set_contxt(ref_data_path(CRF_SAMPLE)) == crf.n_states
    K, W = crf.n_states, crf.window
    Wt = np.zeros((W, 20, K)); bias = np.zeros(K)
    for k in range(K):
        w, b = crf.state(k)
        Wt[:, :, k] = w; bias[k] = b
    rng = np.random.default_rng(9)
    L = 9
    f = rng.dirichlet(np.full(20, 0.4), L + 2).astype(np.float32)
    neff_m = np.concatenate([[99.999], rng.uniform(1.0, 8.0, L)]).astype(np.float32)
    counts = np.ascontiguousarray((f[1:L + 1] * neff_m[1:L + 1, None]).astype(np.float32).astype(np.float64))
    score = np.zeros((L, K))
    wt = np.ascontiguousarray(Wt)
    emul.emul_crf_scores.argtypes = [C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 4
    emul.emul_crf_scores(L, K, W, wt.ctypes.data, bias.ctypes.data, counts.ctypes.data, score.ctypes.data)
    got = crf.tail_host(score, f, neff_m, capi.Admix.hhm())
    ref, _ = refshim.context_pc(f, neff_m, 3.0, engine=0)
    assert np.array_equal(bits(got[1:L + 1]), bits(ref[1:L + 1]))
    crf.close()


def test_emulated_kernels_on_corner_cases(emul, refshim, tmp_path):
    for k, t in enumerate(msa_cases.TINY):
        path = tmp_path / f"t{k}.a3m"
        path.write_bytes(t)
        for wg in (0, 1):
            _cmp(_run(emul, refshim, t, wg=wg), refshim.msa_to_hmm(str(path), wg=wg), f"tiny {k} wg={wg}")


FASTA = (b">ss_pred\nHHHEEECCCHHH\n>m\nACDEFGHIKLMN\n>s1\nAC-EFGHI-LMN\n>s2\n--DEFaHIKLM-\n>s3\nACDE.GHIKL--\n>s4\n-CDEFGHIKLMN\n",
         b">m\nMKV-LAAGIV\n>s1\nMRV-LSAGLV\n")


@pytest.mark.parametrize("M,Mgaps", [(2, 50), (2, 20), (3, 50)])
def test_emulated_kernels_with_other_match_state_rules(emul, refshim, tmp_path, M, Mgaps):
    """-M <percent> / -M first (Compress cases 2 and 3) for alignments that are not A3M; incl. the two-sequence case in
    which the reference keeps the residue counts of ALL input columns."""
    try:
        refshim.set_M(M, Mgaps)
        for k, t in enumerate(FASTA):
            path = tmp_path / f"f{k}.fas"
            path.write_bytes(t)
            _cmp(_run(emul, refshim, t, M=M, Mgaps=Mgaps), refshim.msa_to_hmm(str(path)), f"fasta {k} M={M}/{Mgaps}")
    finally:
        refshim.set_M(1, 50)
