"""ctypes bindings for the TEST-ONLY oracle libraries (never imported by the product package).

  Oracle()   -> oracle/liboracle.so        (C restatement, oracle/hh_oracle.c; always buildable)
  RefShim()  -> oracle/_ref/libhhref_shim.so (the compiled, unmodified reference; built in the
                authoring container from /root/reference, shipped prebuilt to the GPU box)
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
c_f32p = C.POINTER(C.c_float)
c_i32p = C.POINTER(C.c_int)
c_u8p = C.POINTER(C.c_uint8)


def _p(a, t):
    return None if a is None else a.ctypes.data_as(t)


def build_oracle():
    subprocess.check_call(["make", "-C", HERE, "-s"])


class PrepParams(C.Structure):
    """hho_prep_params / hhg_prep_params: Parameters::gap* and pc_hhm_nocontext_* (src/hhdecl.cpp:64-80)."""
    _fields_ = [("gapb", C.c_float), ("gapd", C.c_float), ("gape", C.c_float), ("gapf", C.c_float),
                ("gapg", C.c_float), ("gaph", C.c_float), ("gapi", C.c_float), ("pcm", C.c_int),
                ("pca", C.c_float), ("pcb", C.c_float), ("pcc", C.c_float)]

    @classmethod
    def defaults(cls):
        return cls(1.0, 0.15, 1.0, 0.6, 0.6, 0.6, 0.6, 2, 1.0, 1.5, 1.0)


# alphabetical HHM column order -> internal amino-acid numbers (s2a, src/hhdecl.h:61)
S2A = np.array([0, 4, 3, 6, 13, 7, 8, 9, 11, 10, 12, 2, 14, 5, 1, 15, 16, 19, 17, 18])


class Oracle:
    def __init__(self):
        path = os.path.join(HERE, "liboracle.so")
        if not os.path.exists(path):
            build_oracle()
        self.lib = L = C.CDLL(path)
        L.hho_viterbi_align.restype = C.c_int
        L.hho_viterbi_align.argtypes = [C.c_int, c_f32p, c_f32p, c_u8p, C.c_int, c_f32p, c_f32p, c_u8p,
                                        c_f32p, C.c_float, c_u8p, C.c_int, C.c_float, C.c_float,
                                        C.c_float, c_f32p, c_i32p, c_i32p, c_u8p]
        L.hho_backtrace.restype = C.c_int
        L.hho_backtrace.argtypes = [C.c_int, c_u8p, C.c_int, C.c_int, c_i32p, c_i32p, c_u8p, c_i32p]
        L.hho_exclude_alignment.restype = None
        L.hho_exclude_alignment.argtypes = [C.c_int, C.c_int, c_i32p, c_i32p, C.c_int, c_u8p]
        L.hho_prefilter_query_profile.restype = None
        L.hho_prefilter_query_profile.argtypes = [C.c_int, c_f32p, c_f32p, c_f32p, C.c_int, C.c_int, c_u8p]
        L.hho_ungapped_score.restype = C.c_int
        L.hho_ungapped_score.argtypes = [C.c_int, c_u8p, c_u8p, C.c_int, C.c_int]
        L.hho_ungapped_corrected.restype = C.c_int
        L.hho_ungapped_corrected.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int]
        L.hho_flog2.restype = C.c_float
        L.hho_flog2.argtypes = [C.c_float]
        L.hho_fpow2.restype = C.c_float
        L.hho_fpow2.argtypes = [C.c_float]
        L.hho_fast_log2.restype = C.c_float
        L.hho_fast_log2.argtypes = [C.c_float]
        L.hho_hhm_parse.restype = C.c_int
        L.hho_hhm_parse.argtypes = [C.c_char_p, C.c_long, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_int),
                                    C.POINTER(C.c_int), c_i32p, c_i32p, c_i32p, c_i32p, c_u8p, c_u8p,
                                    C.POINTER(C.c_int)]
        L.hho_hhm_prepare.restype = C.c_int
        L.hho_hhm_prepare.argtypes = [C.c_int, c_i32p, c_i32p, c_i32p, c_f32p, C.c_float, C.c_int,
                                      C.POINTER(PrepParams), c_f32p, c_f32p, c_f32p, c_f32p]
        L.hho_log2lin.restype = C.c_float
        L.hho_log2lin.argtypes = [C.c_float]
        L.hho_mac_realign.restype = C.c_int
        L.hho_mac_realign.argtypes = [C.c_int, c_f32p, c_f32p, C.c_int, c_f32p, c_f32p, C.c_int, C.c_float, C.c_float,
                                      C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, c_i32p, c_i32p, C.c_int, c_i32p,
                                      c_i32p, c_i32p, c_i32p, c_f32p, C.POINTER(C.c_double), c_i32p, c_i32p, c_u8p,
                                      c_f32p, c_f32p]
        L.hho_sw_striped_byte.restype = C.c_int
        L.hho_sw_striped_byte.argtypes = [C.c_int, c_u8p, c_u8p, C.c_int, C.c_int, C.c_int, C.c_int]

    def hhm_parse(self, text, maxL=4000):
        """HMM::Read restatement: the integers of one HHM record."""
        if isinstance(text, str):
            text = text.encode()
        f = np.zeros(((maxL + 2), 20), np.int32); tr = np.zeros((maxL + 1, 7), np.int32)
        ne = np.zeros((maxL + 1, 3), np.int32); null = np.zeros(20, np.int32)
        sp = np.zeros(maxL + 2, np.uint8); sc = np.zeros(maxL + 2, np.uint8)
        neff = C.c_float(); has_pc = C.c_int(); has_null = C.c_int(); nss = C.c_int()
        L = self.lib.hho_hhm_parse(text, len(text), maxL, C.byref(neff), C.byref(has_pc), C.byref(has_null),
                                   _p(null, c_i32p), _p(f, c_i32p), _p(tr, c_i32p), _p(ne, c_i32p),
                                   _p(sp, c_u8p), _p(sc, c_u8p), C.byref(nss))
        if L < 0:
            raise ValueError(f"hho_hhm_parse: {L}")
        return dict(L=L, neff_hmm=neff.value, has_pc=has_pc.value, null=null if has_null.value else None,
                    f=f[:L + 2].copy(), tr=tr[:L + 1].copy(), neff=ne[:L + 1].copy(),
                    ss=(sp[:L + 2] * 11 + sc[:L + 2]).astype(np.uint8), has_ss=nss.value >= 0)

    def null_to_pb(self, null_mb):
        """pb[s2a[a]] = fpow2(-x/1000), src/hhhmm.cpp:543."""
        pb = np.zeros(20, np.float32)
        for a in range(20):
            pb[S2A[a]] = self.lib.hho_fpow2(float(np.float32(-int(null_mb[a])) / np.float32(1000)))
        return pb

    def hhm_prepare(self, rec, pb, R, params=None):
        """Query-independent part of PrepareTemplateHMM on a parsed record -> p (pre-null-model), tr, pav."""
        pp = params or PrepParams.defaults()
        L = rec["L"]
        f = np.ascontiguousarray(rec["f"], np.int32); tr_mb = np.ascontiguousarray(rec["tr"], np.int32)
        ne = np.ascontiguousarray(rec["neff"], np.int32)
        pb = np.ascontiguousarray(pb, np.float32); R = np.ascontiguousarray(R, np.float32)
        p = np.zeros((L + 2, 20), np.float32); tr = np.zeros((L + 1, 7), np.float32); pav = np.zeros(20, np.float32)
        rc = self.lib.hho_hhm_prepare(L, _p(f, c_i32p), _p(tr_mb, c_i32p), _p(ne, c_i32p), _p(pb, c_f32p),
                                      rec["neff_hmm"], rec["has_pc"], C.byref(pp), _p(R, c_f32p),
                                      _p(p, c_f32p), _p(tr, c_f32p), _p(pav, c_f32p))
        if rc != 0:
            raise ValueError(f"hho_hhm_prepare: {rc}")
        return dict(L=L, p=p, tr=tr, pav=pav, ss=rec["ss"])

    def fast_log2(self, x):
        return self.lib.hho_fast_log2(float(x))

    def log2lin(self, tr):
        """HMM::Log2LinTransitionProbs(1.0), src/hhhmm.cpp:2305-2313."""
        tr = np.asarray(tr, np.float32)
        out = np.array([self.lib.hho_log2lin(float(v)) for v in tr.reshape(-1)], np.float32)
        return out.reshape(tr.shape)

    def mac_realign(self, q_p, q_tr_lin, t_p, t_tr_lin, vit, excl=(), local=True, shift=-0.03, mact=0.35):
        """PosteriorDecoder::realign restated (no SS term).  vit = (i1, i2, j1, j2, nsteps, i_steps, j_steps)."""
        Lq = q_p.shape[0] - 2; Lt = t_p.shape[0] - 2
        q_p = np.ascontiguousarray(q_p, np.float32); q_tr_lin = np.ascontiguousarray(q_tr_lin, np.float32)
        t_p = np.ascontiguousarray(t_p, np.float32); t_tr_lin = np.ascontiguousarray(t_tr_lin, np.float32)
        i1, i2, j1, j2, n, vi, vj = vit
        vi = np.ascontiguousarray(vi, np.int32); vj = np.ascontiguousarray(vj, np.int32)
        eo = np.zeros(len(excl) + 1, np.int32)
        for k, (a, b) in enumerate(excl):
            eo[k + 1] = eo[k] + len(a)
        ei = np.ascontiguousarray(np.concatenate([np.asarray(a, np.int32) for a, _ in excl]) if excl else np.zeros(1, np.int32))
        ej = np.ascontiguousarray(np.concatenate([np.asarray(b, np.int32) for _, b in excl]) if excl else np.zeros(1, np.int32))
        cap = Lq + Lt + 4
        res = np.zeros(6, np.int32); sp = np.zeros(1, np.float32); pf = C.c_double()
        oi = np.zeros(cap, np.int32); oj = np.zeros(cap, np.int32); ost = np.zeros(cap, np.uint8)
        ops = np.zeros(cap, np.float32); post = np.zeros((Lq + 1, Lt + 1), np.float32)
        nn = self.lib.hho_mac_realign(Lq, _p(q_p, c_f32p), _p(q_tr_lin, c_f32p), Lt, _p(t_p, c_f32p), _p(t_tr_lin, c_f32p),
                                      1 if local else 0, shift, mact, i1, i2, j1, j2, n, _p(vi, c_i32p), _p(vj, c_i32p),
                                      len(excl), _p(eo, c_i32p), _p(ei, c_i32p), _p(ej, c_i32p), _p(res, c_i32p),
                                      _p(sp, c_f32p), C.byref(pf), _p(oi, c_i32p), _p(oj, c_i32p), _p(ost, c_u8p),
                                      _p(ops, c_f32p), _p(post, c_f32p))
        if nn < 0:
            raise RuntimeError(f"hho_mac_realign: {nn}")
        return dict(i1=int(res[0]), i2=int(res[1]), j1=int(res[2]), j2=int(res[3]), nsteps=int(res[4]),
                    matched_cols=int(res[5]), sum_of_probs=float(sp[0]), Pforward=pf.value, i=oi[:nn + 1].copy(),
                    j=oj[:nn + 1].copy(), states=ost[:nn + 1].copy(), P_posterior=ops[:nn + 1].copy(), post=post)

    def viterbi(self, q_p, q_tr, t_p, t_tr, q_ss=None, t_ss=None, S33=None, ssw=0.11, celloff=None,
                local=True, egq=0.0, egt=0.0, shift=-0.03, want_bt=True):
        Lq = q_p.shape[0] - 2
        Lt = t_p.shape[0] - 2
        q_p = np.ascontiguousarray(q_p, np.float32); q_tr = np.ascontiguousarray(q_tr, np.float32)
        t_p = np.ascontiguousarray(t_p, np.float32); t_tr = np.ascontiguousarray(t_tr, np.float32)
        bt = np.zeros((Lq + 1, Lt + 1), np.uint8) if want_bt else None
        sc = C.c_float(); i2 = C.c_int(); j2 = C.c_int()
        use_ss = S33 is not None
        self.lib.hho_viterbi_align(Lq, _p(q_p, c_f32p), _p(q_tr, c_f32p), _p(q_ss, c_u8p) if use_ss else None,
                                   Lt, _p(t_p, c_f32p), _p(t_tr, c_f32p), _p(t_ss, c_u8p) if use_ss else None,
                                   _p(S33, c_f32p) if use_ss else None, ssw, _p(celloff, c_u8p),
                                   1 if local else 0, egq, egt, shift, C.byref(sc), C.byref(i2),
                                   C.byref(j2), _p(bt, c_u8p))
        return sc.value, i2.value, j2.value, bt

    def backtrace(self, bt, i2, j2):
        Lt = bt.shape[1] - 1
        n = i2 + j2 + 2
        i_s = np.zeros(n, np.int32); j_s = np.zeros(n, np.int32); st = np.zeros(n, np.uint8)
        mc = C.c_int()
        k = self.lib.hho_backtrace(Lt, _p(bt, c_u8p), i2, j2, _p(i_s, c_i32p), _p(j_s, c_i32p),
                                   _p(st, c_u8p), C.byref(mc))
        return k, i_s[:k + 1], j_s[:k + 1], st[:k + 1], mc.value

    def exclude_alignment(self, celloff, i_steps, j_steps, nsteps):
        Lq, Lt = celloff.shape[0] - 1, celloff.shape[1] - 1
        i_s = np.ascontiguousarray(i_steps, np.int32); j_s = np.ascontiguousarray(j_steps, np.int32)
        self.lib.hho_exclude_alignment(Lq, Lt, _p(i_s, c_i32p), _p(j_s, c_i32p), nsteps, _p(celloff, c_u8p))

    def prefilter_query_profile(self, q_p, q_pav, lib219, offset=50, bit_factor=4):
        Lq = q_p.shape[0] - 2
        prof = np.zeros((220, Lq), np.uint8)
        q_p = np.ascontiguousarray(q_p, np.float32)
        q_pav = np.ascontiguousarray(q_pav, np.float32)
        lib219 = np.ascontiguousarray(lib219, np.float32)
        self.lib.hho_prefilter_query_profile(Lq, _p(q_p, c_f32p), _p(q_pav, c_f32p), _p(lib219, c_f32p),
                                             offset, bit_factor, _p(prof, c_u8p))
        return prof

    def ungapped(self, prof, seq, offset=50):
        seq = np.ascontiguousarray(seq, np.uint8)
        return self.lib.hho_ungapped_score(prof.shape[1], _p(prof, c_u8p), _p(seq, c_u8p), len(seq), offset)


    def sw_byte(self, prof, seq, gap_open=24, gap_extend=4, bias=50):
        seq = np.ascontiguousarray(seq, np.uint8)
        prof = np.ascontiguousarray(prof, np.uint8)
        return self.lib.hho_sw_striped_byte(prof.shape[1], _p(prof, c_u8p), _p(seq, c_u8p), len(seq), gap_open,
                                            gap_extend, bias)

    def flog2(self, x):
        return self.lib.hho_flog2(float(x))

    def fpow2(self, x):
        return self.lib.hho_fpow2(float(x))


class RefShim:
    """The compiled reference. Raises FileNotFoundError when oracle/_ref was not built/shipped."""

    def __init__(self, nocontxt=True, maxres=4096):
        path = os.path.join(HERE, "_ref", "libhhref_shim.so")
        if not os.path.exists(path):
            raise FileNotFoundError(path)
        self.lib = L = C.CDLL(path)
        L.hhref_init.argtypes = [C.c_int, C.c_int]
        L.hhref_par_shift.restype = C.c_float
        L.hhref_par_ssw.restype = C.c_float
        L.hhref_par_corr.restype = C.c_float
        L.hhref_load_query_hhm.argtypes = [C.c_char_p]
        L.hhref_get_query.argtypes = [c_f32p, c_f32p, c_f32p, c_u8p, c_u8p, c_u8p, c_f32p]
        L.hhref_set_query.argtypes = [C.c_int, c_f32p, c_f32p, c_f32p, c_u8p, c_u8p]
        L.hhref_prepare_template_hhm.argtypes = [C.c_char_p, c_f32p, c_f32p, c_f32p, c_u8p, c_u8p, c_u8p,
                                                 c_f32p, C.c_int]
        L.hhref_prepare_template_hhm_raw.argtypes = [C.c_char_p, C.c_int, c_f32p, c_f32p, c_f32p, c_f32p, C.c_int]
        L.hhref_fast_log2.restype = C.c_float
        L.hhref_fast_log2.argtypes = [C.c_float]
        L.hhref_score_cols.restype = C.c_float
        L.hhref_score_cols.argtypes = [c_f32p, c_f32p]
        L.hhref_viterbi_align.argtypes = [C.c_int, c_i32p, C.POINTER(c_f32p), C.POINTER(c_f32p),
                                          C.POINTER(c_u8p), C.POINTER(c_u8p), C.POINTER(c_u8p), C.c_int,
                                          C.c_int, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float,
                                          c_f32p, c_i32p, c_i32p, C.POINTER(c_u8p)]
        L.hhref_backtrace.argtypes = [C.c_int, c_i32p, c_i32p, C.c_char_p, c_i32p]
        L.hhref_score_for_backtrace.argtypes = [C.c_int, c_f32p, c_f32p]
        L.hhref_viterbi_bench.restype = C.c_double
        L.hhref_viterbi_bench.argtypes = [C.c_int, c_i32p, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong),
                                          c_f32p, c_f32p, C.c_int, C.c_int, C.c_int,
                                          C.POINTER(C.c_double), c_f32p]
        L.hhref_get_cs219.argtypes = [c_f32p]
        L.hhref_get_S33.argtypes = [c_f32p]
        L.hhref_get_pb.argtypes = [c_f32p]
        L.hhref_get_R.argtypes = [c_f32p]
        L.hhref_mac_realign.argtypes = [C.c_int, c_f32p, c_f32p, C.c_int, C.c_float, C.c_float, C.c_float, C.c_int,
                                        C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, c_i32p, c_i32p,
                                        C.c_int, c_i32p, c_i32p, c_i32p,
                                        c_i32p, c_f32p, C.POINTER(C.c_double), c_i32p, c_i32p, C.c_char_p,
                                        c_f32p, c_f32p, c_f32p, c_f32p]
        L.hhref_get_prep_params.argtypes = [c_f32p]
        L.hhref_stripe_query_profile.argtypes = [C.c_int, C.c_int, c_u8p]
        L.hhref_ungapped_score.argtypes = [c_u8p, C.c_int, c_u8p, C.c_int, C.c_int]
        L.hhref_sw_striped_byte.argtypes = [c_u8p, C.c_int, c_u8p, C.c_int, C.c_int, C.c_int, C.c_int]
        L.hhref_ungapped_bench.restype = C.c_double
        L.hhref_ungapped_bench.argtypes = [c_u8p, C.c_int, C.c_int, c_u8p, C.POINTER(C.c_longlong), c_i32p,
                                           C.c_int, C.c_int, c_i32p]
        L.hhref_init(1 if nocontxt else 0, maxres)
        self.maxres = maxres
        self.V = L.hhref_vecsize()
        self.Lq = 0
        self._warm_fast_log2()

    def _warm_fast_log2(self):
        """Reference quirk: fast_log2's static table (src/util-inl.h:108-121) is filled by whichever
        translation unit calls it first, and `log(float(..))` resolves to the double-precision C log in
        hhhmm.cpp but to the float overload in hhviterbi.cpp -- two slightly different tables.  Every real
        run of the reference reads the query HMM first (HMM::Read / PrepareQueryHMM), so the table that
        matters is the hhhmm.cpp one; reproduce that order here before anything else touches fast_log2."""
        import importlib.util
        import tempfile
        spec = importlib.util.spec_from_file_location(
            "_hh_synth", os.path.join(os.path.dirname(HERE), "hh-suite_b200", "synth.py"))
        synth = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(synth)
        with tempfile.NamedTemporaryFile("w", suffix=".hhm", delete=False) as f:
            f.write(synth.hhm_text(24, 0, "warm"))
            path = f.name
        try:
            self.lib.hhref_load_query_hhm(path.encode())
        finally:
            os.unlink(path)

    # -- parameters
    def defaults(self):
        return dict(shift=self.lib.hhref_par_shift(), ssw=self.lib.hhref_par_ssw(),
                    corr=self.lib.hhref_par_corr())

    def S33(self):
        out = np.zeros(44 * 44, np.float32)
        self.lib.hhref_get_S33(_p(out, c_f32p))
        return out

    def R(self):
        out = np.zeros(400, np.float32)
        self.lib.hhref_get_R(_p(out, c_f32p))
        return out.reshape(20, 20)

    def S(self):
        out = np.zeros(400, np.float32)
        self.lib.hhref_get_S(_p(out, c_f32p))
        return out.reshape(20, 20)

    def pb(self):
        out = np.zeros(20, np.float32)
        self.lib.hhref_get_pb(_p(out, c_f32p))
        return out

    def prep_params(self):
        v = np.zeros(11, np.float32)
        self.lib.hhref_get_prep_params(_p(v, c_f32p))
        return PrepParams(*[float(x) for x in v[:7]], int(v[7]), *[float(x) for x in v[8:]])

    # -- query
    def set_pc(self, mode, a, b, c):
        """par.pc_hhm_nocontext_mode/_a/_b/_c (-pcm -pca -pcb -pcc) for the following template / query preparations."""
        self.lib.hhref_set_pc.argtypes = [C.c_int, C.c_float, C.c_float, C.c_float]
        self.lib.hhref_set_pc(mode, a, b, c)

    def load_query_hhm(self, path):
        L = self.lib.hhref_load_query_hhm(path.encode())
        if L < 0:
            raise IOError(path)
        self.Lq = L
        return self.get_query()

    def get_query(self):
        L = self.Lq
        p = np.zeros((L + 2, 20), np.float32); tr = np.zeros((L + 1, 7), np.float32)
        pav = np.zeros(20, np.float32)
        sp = np.zeros(L + 2, np.uint8); sc = np.zeros(L + 2, np.uint8); sd = np.zeros(L + 2, np.uint8)
        neff = C.c_float()
        self.lib.hhref_get_query(_p(p, c_f32p), _p(tr, c_f32p), _p(pav, c_f32p), _p(sp, c_u8p),
                                 _p(sc, c_u8p), _p(sd, c_u8p), C.byref(neff))
        return dict(L=L, p=p, tr=tr, pav=pav, ss_pred=sp, ss_conf=sc, ss=(sp * 11 + sc).astype(np.uint8),
                    neff=neff.value)

    def set_query(self, p, tr, pav=None, ss=None):
        L = p.shape[0] - 2
        p = np.ascontiguousarray(p, np.float32); tr = np.ascontiguousarray(tr, np.float32)
        sp = sc = None
        if ss is not None:
            sp = np.ascontiguousarray(ss // 11, np.uint8); sc = np.ascontiguousarray(ss % 11, np.uint8)
        if pav is not None:
            pav = np.ascontiguousarray(pav, np.float32)
        r = self.lib.hhref_set_query(L, _p(p, c_f32p), _p(tr, c_f32p), _p(pav, c_f32p), _p(sp, c_u8p),
                                     _p(sc, c_u8p))
        assert r == L
        self.Lq = L

    def prepare_template_hhm(self, path, maxL=4000):
        p = np.zeros((maxL + 2, 20), np.float32); tr = np.zeros((maxL + 1, 7), np.float32)
        pav = np.zeros(20, np.float32)
        sp = np.zeros(maxL + 2, np.uint8); sc = np.zeros(maxL + 2, np.uint8); sd = np.zeros(maxL + 2, np.uint8)
        neff = C.c_float()
        L = self.lib.hhref_prepare_template_hhm(path.encode(), _p(p, c_f32p), _p(tr, c_f32p), _p(pav, c_f32p),
                                                _p(sp, c_u8p), _p(sc, c_u8p), _p(sd, c_u8p),
                                                C.byref(neff), maxL)
        if L < 0:
            raise IOError(path)
        return dict(L=L, p=p[:L + 2].copy(), tr=tr[:L + 1].copy(), pav=pav,
                    ss=(sp[:L + 2] * 11 + sc[:L + 2]).astype(np.uint8), neff=neff.value)

    def prepare_template_hhm_raw(self, path, columnscore=1, maxL=4000):
        p_raw = np.zeros((maxL + 2, 20), np.float32); p_prep = np.zeros((maxL + 2, 20), np.float32)
        tr = np.zeros((maxL + 1, 7), np.float32); pav = np.zeros(20, np.float32)
        L = self.lib.hhref_prepare_template_hhm_raw(path.encode(), columnscore, _p(p_raw, c_f32p),
                                                    _p(p_prep, c_f32p), _p(tr, c_f32p), _p(pav, c_f32p), maxL)
        if L < 0:
            raise IOError(path)
        return dict(L=L, p_raw=p_raw[:L + 2].copy(), p=p_prep[:L + 2].copy(), tr=tr[:L + 1].copy(), pav=pav)

    def crf_text(self):
        """The context_data.crf bytes embedded in the reference build (what InitializePseudocountsEngine reads)."""
        n = C.c_longlong()
        self.lib.hhref_crf_text.restype = C.c_void_p
        self.lib.hhref_crf_text.argtypes = [C.POINTER(C.c_longlong)]
        ptr = self.lib.hhref_crf_text(C.byref(n))
        return C.string_at(ptr, n.value)

    def set_contxt(self, path):
        """par.clusterfile (-contxt): the .crf library of the following crf_state / context_pc calls."""
        self.lib.hhref_set_contxt.argtypes = [C.c_char_p]
        return self.lib.hhref_set_contxt(path.encode())

    def crf_state(self, k):
        pc = np.zeros(20, np.float64); w = np.zeros(13 * 20, np.float64); b = C.c_double()
        self.lib.hhref_crf_state.argtypes = [C.c_int, C.c_void_p, C.POINTER(C.c_double), C.c_void_p]
        n = self.lib.hhref_crf_state(k, pc.ctypes.data, C.byref(b), w.ctypes.data)
        return n, pc, b.value, w.reshape(13, 20)

    def context_pc(self, f, neff_m, neff_hmm, engine=0):
        """HMM::AddContextSpecificPseudocounts + CalculateAminoAcidBackground by the compiled reference.
        engine 0: query HMM (HHsearch admixture), 1: prefilter profile (CS-BLAST admixture)."""
        f = np.ascontiguousarray(f, np.float32); neff_m = np.ascontiguousarray(neff_m, np.float32)
        L = f.shape[0] - 2
        p = np.zeros((L + 2, 20), np.float32); pav = np.zeros(20, np.float32)
        self.lib.hhref_context_pc.argtypes = [C.c_int, c_f32p, c_f32p, C.c_float, C.c_int, c_f32p, c_f32p]
        self.lib.hhref_context_pc(L, _p(f, c_f32p), _p(neff_m, c_f32p), float(neff_hmm), engine, _p(p, c_f32p), _p(pav, c_f32p))
        return p, pav

    def set_mac_exclstr(self, q="", t=""):
        """par.exclstr / par.template_exclstr (-excl / -template_excl) for the following mac_realign calls."""
        self.lib.hhref_set_mac_exclstr.argtypes = [C.c_char_p, C.c_char_p]
        self.lib.hhref_set_mac_exclstr(q.encode(), t.encode())

    def mac_realign(self, t_p, t_tr, vit, excl=(), local=True, shift=-0.03, mact=0.35, corr=0.1, min_overlap=0,
                    want_post=True):
        """PosteriorDecoder::realign for one hit of the loaded query.  vit = (i1, i2, j1, j2, nsteps, i_steps,
        j_steps) of the Viterbi alignment (step arrays 1-based like Hit.i/Hit.j); excl = list of (alt_i, alt_j)
        of previous MAC alignments of this template."""
        Lq = self.Lq
        Lt = t_p.shape[0] - 2
        t_p = np.ascontiguousarray(t_p, np.float32); t_tr = np.ascontiguousarray(t_tr, np.float32)
        i1, i2, j1, j2, n, vi, vj = vit
        vi = np.ascontiguousarray(vi, np.int32); vj = np.ascontiguousarray(vj, np.int32)
        eo = np.zeros(len(excl) + 1, np.int32)
        for k, (a, b) in enumerate(excl):
            eo[k + 1] = eo[k] + len(a)
        ei = np.ascontiguousarray(np.concatenate([np.asarray(a, np.int32) for a, _ in excl]) if excl else np.zeros(1, np.int32))
        ej = np.ascontiguousarray(np.concatenate([np.asarray(b, np.int32) for _, b in excl]) if excl else np.zeros(1, np.int32))
        cap = Lq + Lt + 4
        res = np.zeros(6, np.int32); fres = np.zeros(2, np.float32); pf = C.c_double()
        oi = np.zeros(cap, np.int32); oj = np.zeros(cap, np.int32); ost = C.create_string_buffer(cap)
        ops = np.zeros(cap, np.float32)
        post = np.zeros((Lq + 1, Lt + 1), np.float32) if want_post else None
        ttl = np.zeros((Lt + 1, 7), np.float32); qtl = np.zeros((Lq + 1, 7), np.float32)
        nn = self.lib.hhref_mac_realign(Lt, _p(t_p, c_f32p), _p(t_tr, c_f32p), 1 if local else 0, shift, mact, corr,
                                        min_overlap, i1, i2, j1, j2, n, _p(vi, c_i32p), _p(vj, c_i32p),
                                        len(excl), _p(eo, c_i32p), _p(ei, c_i32p), _p(ej, c_i32p),
                                        _p(res, c_i32p), _p(fres, c_f32p), C.byref(pf), _p(oi, c_i32p), _p(oj, c_i32p),
                                        ost, _p(ops, c_f32p), _p(post, c_f32p), _p(ttl, c_f32p), _p(qtl, c_f32p))
        if nn < 0:
            raise RuntimeError(f"hhref_mac_realign: {nn}")
        st = np.frombuffer(ost.raw, np.uint8)[:nn + 1].copy()
        return dict(i1=int(res[0]), i2=int(res[1]), j1=int(res[2]), j2=int(res[3]), nsteps=int(res[4]),
                    matched_cols=int(res[5]), sum_of_probs=float(fres[0]), Pforward=pf.value, i=oi[:nn + 1].copy(),
                    j=oj[:nn + 1].copy(), states=st, P_posterior=ops[:nn + 1].copy(), post=post, t_tr_lin=ttl,
                    q_tr_lin=qtl)

    def fast_log2_table(self):
        """lg2[0..1024] of the reference's fast_log2 (x in [1,2): a=0, c=0 -> returns lg2[b] exactly)."""
        x = ((np.arange(1024, dtype=np.uint32) << 13) | np.uint32(0x3F800000)).view(np.float32)
        t = np.array([self.lib.hhref_fast_log2(float(v)) for v in x], np.float32)
        return t

    def fast_log2(self, x):
        return self.lib.hhref_fast_log2(float(x))

    def score_cols(self, qi, tj):
        qi = np.ascontiguousarray(qi, np.float32); tj = np.ascontiguousarray(tj, np.float32)
        return self.lib.hhref_score_cols(_p(qi, c_f32p), _p(tj, c_f32p))

    # -- the kernel
    def viterbi(self, targets, use_ss=False, celloff=None, local=True, egq=0.0, egt=0.0, shift=-0.03,
                ssw=0.11, corr=0.1):
        """targets: list (<= V) of (p, tr, ss|None). Returns list of (score, i2, j2, bt)."""
        n = len(targets)
        assert 1 <= n <= self.V
        Lq = self.Lq
        Lt = np.array([t[0].shape[0] - 2 for t in targets], np.int32)
        ps = [np.ascontiguousarray(t[0], np.float32) for t in targets]
        trs = [np.ascontiguousarray(t[1], np.float32) for t in targets]
        P = (c_f32p * n)(*[_p(a, c_f32p) for a in ps])
        T = (c_f32p * n)(*[_p(a, c_f32p) for a in trs])
        SP = SCF = None
        keep = []
        if use_ss:
            sp = [np.ascontiguousarray(t[2] // 11, np.uint8) for t in targets]
            sc = [np.ascontiguousarray(t[2] % 11, np.uint8) for t in targets]
            keep += sp + sc
            SP = (c_u8p * n)(*[_p(a, c_u8p) for a in sp])
            SCF = (c_u8p * n)(*[_p(a, c_u8p) for a in sc])
        CO = None
        if celloff is not None:
            co = [None if c is None else np.ascontiguousarray(c, np.uint8) for c in celloff]
            keep += co
            CO = (c_u8p * n)(*[_p(a, c_u8p) for a in co])
        bts = [np.zeros((Lq + 1, int(l) + 1), np.uint8) for l in Lt]
        BT = (c_u8p * n)(*[_p(a, c_u8p) for a in bts])
        score = np.zeros(n, np.float32); i2 = np.zeros(n, np.int32); j2 = np.zeros(n, np.int32)
        r = self.lib.hhref_viterbi_align(n, _p(Lt, c_i32p), P, T, SP, SCF, CO, 1 if use_ss else 0,
                                         1 if local else 0, egq, egt, shift, ssw, corr,
                                         _p(score, c_f32p), _p(i2, c_i32p), _p(j2, c_i32p), BT)
        assert r == 0, r
        self._last = (score, i2, j2)
        return [(float(score[k]), int(i2[k]), int(j2[k]), bts[k]) for k in range(n)]

    def backtrace(self, elem):
        score, i2, j2 = self._last
        n = int(i2[elem] + j2[elem] + 2)
        i_s = np.zeros(n, np.int32); j_s = np.zeros(n, np.int32)
        st = C.create_string_buffer(n)
        mc = C.c_int()
        k = self.lib.hhref_backtrace(elem, _p(i_s, c_i32p), _p(j_s, c_i32p), st, C.byref(mc))
        states = np.frombuffer(st.raw, np.uint8)[:k + 1].copy()
        return k, i_s[:k + 1], j_s[:k + 1], states, mc.value

    def hit_score(self, elem):
        s = C.c_float(); ss = C.c_float()
        self.lib.hhref_score_for_backtrace(elem, C.byref(s), C.byref(ss))
        return s.value, ss.value

    def viterbi_bench(self, db, threads, with_backtrace=True, repeats=1, want_scores=False):
        """db: dict from synth.prepared_db. Returns (seconds, cells, scores|None)."""
        N = len(db["L"])
        L = np.ascontiguousarray(db["L"], np.int32)
        po = np.ascontiguousarray(db["p_off"] * 20, np.int64)
        to = np.ascontiguousarray(db["tr_off"] * 7, np.int64)
        cells = C.c_double()
        sc = np.zeros(N, np.float32) if want_scores else None
        sec = self.lib.hhref_viterbi_bench(N, _p(L, c_i32p), po.ctypes.data_as(C.POINTER(C.c_longlong)),
                                           to.ctypes.data_as(C.POINTER(C.c_longlong)),
                                           _p(db["p"], c_f32p), _p(db["tr"], c_f32p), threads,
                                           1 if with_backtrace else 0, repeats, C.byref(cells),
                                           _p(sc, c_f32p))
        return sec, cells.value, sc

    # -- hit-list statistics
    def hitlist_stats(self, score, score_ss, L, neff, qL, qneff, N_searched, loc=1, ssm=2, ssw=0.11, ssm2=None, files=None,
                      hhblits=False, dbsize=1, alphaa=0.4, alphab=0.02, alphac=0.1, pf_evalue_thresh=1000.0):
        """HitList::CalculatePvalues (+ CalculateHHblitsEvalues) of the compiled reference on synthetic hits."""
        n = len(score)
        score = np.ascontiguousarray(score, np.float32); score_ss = np.ascontiguousarray(score_ss, np.float32)
        L = np.ascontiguousarray(L, np.int32); neff = np.ascontiguousarray(neff, np.float32)
        s2 = None if ssm2 is None else np.ascontiguousarray(ssm2, np.int32)
        farr = None
        if files is not None:
            farr = (C.c_char_p * n)(*[f.encode() for f in files])
        out = dict(Pval=np.zeros(n), logPval=np.zeros(n), Eval=np.zeros(n), logEval=np.zeros(n),
                   score_aass=np.zeros(n, np.float32), Probab=np.zeros(n, np.float32), order=np.zeros(n, np.int32))
        dp = C.POINTER(C.c_double)
        self.lib.hhref_hitlist_stats.argtypes = [C.c_int, c_f32p, c_f32p, c_i32p, c_f32p, c_i32p, C.c_void_p, C.c_int,
                                                 C.c_float, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int,
                                                 C.c_float, C.c_float, C.c_float, C.c_double, dp, dp, dp, dp, c_f32p,
                                                 c_f32p, c_i32p]
        m = self.lib.hhref_hitlist_stats(n, _p(score, c_f32p), _p(score_ss, c_f32p), _p(L, c_i32p), _p(neff, c_f32p),
                                         _p(s2, c_i32p), farr, qL, qneff, N_searched, loc, ssm, ssw, 1 if hhblits else 0,
                                         dbsize, alphaa, alphab, alphac, pf_evalue_thresh,
                                         out["Pval"].ctypes.data_as(dp), out["logPval"].ctypes.data_as(dp),
                                         out["Eval"].ctypes.data_as(dp), out["logEval"].ctypes.data_as(dp),
                                         _p(out["score_aass"], c_f32p), _p(out["Probab"], c_f32p), _p(out["order"], c_i32p))
        assert m == n
        return out

    def _msa_call(self, fn, lead_args, filt, wg, prep, capL, capN):
        dims = np.zeros(8, np.int32)
        X = np.zeros(capN * (capL + 2), np.uint8); I = np.zeros(capN * (capL + 2), np.uint16)
        keep = np.zeros(capN, np.int8); wgv = np.zeros(capN, np.float32)
        nres = np.zeros(capN, np.int32); ksort = np.zeros(capN, np.int32)
        f = np.zeros((capL + 2) * 20, np.float32); tr = np.zeros((capL + 1) * 7, np.float32)
        neff = np.zeros(3 * (capL + 1), np.float32); nh = np.zeros(1, np.float32)
        ssp = np.zeros(capL + 2, np.uint8); ssc = np.zeros(capL + 2, np.uint8)
        p = np.zeros((capL + 2) * 20, np.float32); trp = np.zeros((capL + 1) * 7, np.float32); pav = np.zeros(20, np.float32)
        fl = None if filt is None else np.asarray(filt, np.float32)
        fn.restype = C.c_int
        fn.argtypes = [C.c_char_p] * len(lead_args) + [c_f32p, C.c_int, C.c_int, C.c_int, C.c_int, c_i32p, c_u8p,
                                                        C.POINTER(C.c_uint16), C.POINTER(C.c_int8), c_f32p, c_i32p, c_i32p,
                                                        c_f32p, c_f32p, c_f32p, c_f32p, c_u8p, c_u8p, c_f32p, c_f32p, c_f32p]
        L = fn(*[a.encode() for a in lead_args], _p(fl, c_f32p), int(wg), int(bool(prep)), capL, capN, _p(dims, c_i32p),
               _p(X, c_u8p), I.ctypes.data_as(C.POINTER(C.c_uint16)), keep.ctypes.data_as(C.POINTER(C.c_int8)),
               _p(wgv, c_f32p), _p(nres, c_i32p), _p(ksort, c_i32p), _p(f, c_f32p), _p(tr, c_f32p), _p(neff, c_f32p),
               _p(nh, c_f32p), _p(ssp, c_u8p), _p(ssc, c_u8p), _p(p, c_f32p), _p(trp, c_f32p), _p(pav, c_f32p))
        if L < 0:
            raise IOError(f"reference alignment reader {lead_args} = {L} (dims {dims.tolist()})")
        N = int(dims[1])
        out = dict(L=L, N_in=N, N_filtered=int(dims[2]), kfirst=int(dims[3]), kss_pred=int(dims[4]), kss_conf=int(dims[5]),
                   X=X[:N * (L + 2)].reshape(N, L + 2).copy(), I=I[:N * (L + 2)].reshape(N, L + 2).copy(),
                   keep=keep[:N].copy(), wg=wgv[:N].copy(), nres=nres[:N].copy(), ksort=ksort[:N].copy(),
                   f=f[:(L + 2) * 20].reshape(L + 2, 20).copy(), tr=tr[:(L + 1) * 7].reshape(L + 1, 7).copy(),
                   neff_m=neff[:L + 1].copy(), neff_i=neff[L + 1:2 * (L + 1)].copy(), neff_d=neff[2 * (L + 1):3 * (L + 1)].copy(),
                   neff_hmm=float(nh[0]), ss_pred=ssp[:L + 2].copy(), ss_conf=ssc[:L + 2].copy())
        if prep:
            out.update(p=p[:(L + 2) * 20].reshape(L + 2, 20).copy(), tr_prep=trp[:(L + 1) * 7].reshape(L + 1, 7).copy(),
                       pav=pav.copy())
        return out

    def msa_to_hmm(self, path, filt=None, wg=0, prep=False, capL=4000, capN=20000):
        """The A3M template branch of HHEntry::getTemplateHMM (src/hhdatabase.cpp:441-449) run by the compiled reference:
        Read, Compress, Filter, FrequenciesAndTransitions (+ PrepareTemplateHMM's query-independent steps with prep).
        filt = (max_seqid, coverage, qid, qsc, Ndiff) or None for the reference defaults."""
        return self._msa_call(self.lib.hhref_msa_to_hmm, [path], filt, wg, prep, capL, capN)

    def ca3m_to_hmm(self, prefix, entry_name, filt=None, wg=0, prep=False, capL=4000, capN=20000):
        """The compressed branch (src/hhdatabase.cpp:303-326): entry of <prefix>_ca3m.ff*, decoded by
        Alignment::ReadCompressed with <prefix>_sequence.ff* / <prefix>_header.ff*."""
        return self._msa_call(self.lib.hhref_ca3m_to_hmm, [prefix, entry_name], filt, wg, prep, capL, capN)

    def set_M(self, M=1, Mgaps=50):
        """par.M_template / par.Mgaps (-M a2m | <percent> | first) for the following msa_to_hmm calls."""
        self.lib.hhref_set_M.argtypes = [C.c_int, C.c_int]
        self.lib.hhref_set_M(M, Mgaps)

    def rcp_table(self, n):
        out = np.zeros(n, np.float32)
        self.lib.hhref_rcp_table.argtypes = [C.c_int, c_f32p]
        self.lib.hhref_rcp_table(n, _p(out, c_f32p))
        return out

    def early_stop(self, score, L, neff, qL, qneff, prefilter=True, dbsize=1, alphaa=0.4, alphab=0.02, alphac=0.1,
                   thresh=1000.0):
        score = np.ascontiguousarray(score, np.float32); L = np.ascontiguousarray(L, np.int32)
        neff = np.ascontiguousarray(neff, np.float32)
        self.lib.hhref_early_stop.argtypes = [C.c_int, c_f32p, c_i32p, c_f32p, C.c_int, C.c_float, C.c_int, C.c_int,
                                              C.c_float, C.c_float, C.c_float, C.c_double]
        self.lib.hhref_early_stop.restype = C.c_float
        return float(self.lib.hhref_early_stop(len(score), _p(score, c_f32p), _p(L, c_i32p), _p(neff, c_f32p), qL, qneff,
                                               1 if prefilter else 0, dbsize, alphaa, alphab, alphac, thresh))

    # -- prefilter
    def cs219(self):
        out = np.zeros((219, 20), np.float32)
        k = self.lib.hhref_get_cs219(_p(out, c_f32p))
        assert k == 219
        return out

    def stripe_query_profile(self, offset=50, bit_factor=4):
        qc = np.zeros(220 * (self.Lq + 64), np.uint8)
        W = self.lib.hhref_stripe_query_profile(offset, bit_factor, _p(qc, c_u8p))
        return qc, W

    def ungapped(self, qc, seq, offset=50):
        seq = np.ascontiguousarray(seq, np.uint8)
        return self.lib.hhref_ungapped_score(_p(qc, c_u8p), self.Lq, _p(seq, c_u8p), len(seq), offset)

    def sw_byte(self, qc, seq, gap_open=24, gap_extend=4, offset=50):
        seq = np.ascontiguousarray(seq, np.uint8)
        return self.lib.hhref_sw_striped_byte(_p(qc, c_u8p), self.Lq, _p(seq, c_u8p), len(seq), gap_open,
                                              gap_extend, offset)

    def ungapped_bench(self, qc, db, threads, offset=50):
        N = len(db["L"])
        sc = np.zeros(N, np.int32)
        L = np.ascontiguousarray(db["L"], np.int32)
        off = np.ascontiguousarray(db["off"], np.int64)
        sec = self.lib.hhref_ungapped_bench(_p(qc, c_u8p), self.Lq, N, _p(db["seq"], c_u8p),
                                            off.ctypes.data_as(C.POINTER(C.c_longlong)), _p(L, c_i32p),
                                            offset, threads, _p(sc, c_i32p))
        return sec, sc
