"""Adversarial inputs for the Viterbi forward pass and backtrace, shared by the CPU and GPU tests (not product code),
and a float32 numpy restatement of the forward pass that counts the decisions those inputs make the kernel take.

Random profiles (synth.prepared_profile) have continuous, distinct values, so two DP candidates are never equal and
the tie rules of the kernel are never exercised.  The families below are built to produce exact ties and special
float values.  Every profile is in the include/hhg.h layout that synth returns: p[(L+2),20], tr[(L+1),7] (log2,
order M2M,M2I,M2D,I2M,I2I,D2M,D2D), ss[L+2].

  F1 lattice   every dot product is a power of two or zero, transitions in {0,-1,-2,-3,NEG}: integer DP values
  F2 periodic  query and target repeat one motif with constant transitions; and matching segments placed so that
               the tied best cells lie in different rows of one strip and in different strips, the later row at the
               earlier column
  F3 hhm       continuous emissions drawn from a small pool of columns, transitions -k/1000 as HHM files store them
  F4 special   -0.0 emission columns, signed-zero transitions, zero / subnormal / overflowing dot products, chains
               saturated at -FLT_MAX or -inf, cell-off masks over every cell and over every global-mode end cell
  F5 padding   short lanes whose last column is a strong match, in one warp job with a long lane: the padding
               (which repeats that column) would outscore every real cell if it were not masked
  F6 lengths   query lengths around the strip heights 8, 12 and 16, and the C-ABI's limit 32767

census() restates the forward pass (oracle/hh_oracle.c, hho_viterbi_align) in float32 numpy and counts, per target,
the cells where the maximum of {STOP, c1..c5} is attained more than once, the ties a1 == a2 of the four gap-state
comparisons, the tied best cells, and the padded cells that would beat the real best.  Each case states the minimum
counts it is built to produce (Case.expect), so that a change to a generator that stops producing ties fails.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

from hhsuite_b200 import synth

NEG = np.float32(synth.NEG)
FMAX = np.float32(np.finfo(np.float32).max)
M2M, M2I, M2D, I2M, I2I, D2M, D2D = range(7)
STRIP_ROWS = (8, 12, 16)


@dataclass
class Case:
    name: str
    q: tuple                       # (p, tr, ss)
    targets: list                  # [(p, tr, ss)]
    local: bool = True
    egq: float = 0.0
    egt: float = 0.0
    shift: float = -0.03
    q_ranges: tuple = ()           # excluded query rows, 1-based inclusive (-excl)
    t_ranges: tuple = ()           # excluded template columns (-template_excl)
    expect: dict = field(default_factory=dict)   # minimum census counts, summed over the targets

    @property
    def Lq(self):
        return self.q[0].shape[0] - 2

    def par(self):
        """Keyword arguments of Context.set_query and Oracle.viterbi."""
        return dict(local=self.local, egq=self.egq, egt=self.egt, shift=self.shift)

    def celloff(self, k):
        """The u8[(Lq+1),(Lt+1)] cell-off mask of the excluded regions for target k, or None."""
        if not self.q_ranges and not self.t_ranges:
            return None
        Lt = self.targets[k][0].shape[0] - 2
        m = np.zeros((self.Lq + 1, Lt + 1), np.uint8)
        for a, b in self.q_ranges:
            m[a:min(b, self.Lq) + 1, 1:] = 1
        for a, b in self.t_ranges:
            m[1:, a:min(b, Lt) + 1] = 1
        return m

    def with_(self, **kw):
        d = dict(self.__dict__)
        d.update(kw)
        return Case(**d)


# ------------------------------------------------------------------------------------------------ profile builders

def _ss(L, rng):
    ss = np.zeros(L + 2, np.uint8)
    ss[1:L + 1] = (rng.integers(1, 4, L) * 11 + rng.integers(1, 11, L)).astype(np.uint8)
    return ss


def profile(P, TR, rng):
    """Prepared profile from L emission rows and L+1 transition rows (rows 0 and L+1 of p hold 1.0)."""
    P = np.asarray(P, np.float32)
    L = P.shape[0]
    p = np.ones((L + 2, 20), np.float32)
    p[1:L + 1] = P
    tr = np.ascontiguousarray(TR, np.float32)
    assert tr.shape == (L + 1, 7)
    return p, tr, _ss(L, rng)


def onehot(letters, values=2.0):
    """Emission rows with `values` on residue letters[i] and 0 elsewhere."""
    letters = np.asarray(letters)
    P = np.zeros((len(letters), 20), np.float32)
    P[np.arange(len(letters)), letters] = values
    return P


def const_tr(L, m2m=0.0, m2i=-3.0, m2d=-3.0, i2m=-1.0, i2i=-2.0, d2m=-1.0, d2d=-2.0):
    return np.tile(np.float32([m2m, m2i, m2d, i2m, i2i, d2m, d2d]), (L + 1, 1))


def lattice_tr(L, rng, values=(0.0, -1.0, -2.0, -3.0, float(NEG)), prob=(.35, .2, .2, .15, .1)):
    return rng.choice(np.float32(values), size=(L + 1, 7), p=prob).astype(np.float32)


def lattice_em(L, rng, alphabet=3):
    return onehot(rng.integers(0, alphabet, L), np.exp2(rng.integers(-2, 3, L)).astype(np.float32))


def synth_query(L, seed):
    qp, qtr, qss, qpav, qcols = synth.query_profile(L, seed)
    return qp, qtr, qss


def pav(q):
    """Mean emission row of a prepared profile (the refshim's query pav)."""
    return np.ascontiguousarray(q[0][1:-1].mean(axis=0), np.float32)


# ------------------------------------------------------------------------------------------------------ families

def f1_lattice(seed, shift):
    rng = np.random.default_rng(seed)
    Lq = 37
    q = profile(lattice_em(Lq, rng), lattice_tr(Lq, rng), rng)
    tg = [profile(lattice_em(L, rng), lattice_tr(L, rng), rng) for L in (1, 5, 16, 29, 37, 48, 64, 90)]
    return Case(f"F1-lattice-s{seed}-shift{shift:g}", q, tg, shift=shift,
                expect=dict(mm_tie=50, gd_tie=20, im_tie=20, dg_tie=20, mi_tie=20, best_tie=2))


def f2_periodic(R, period):
    """Query of 3R+2 rows and targets of R-3 and 3R+7 columns repeating one motif: the best cells tie over the
    last column's rows R-3..3R+2 (across strips) and the last row's columns (one row)."""
    rng = np.random.default_rng(100 * R + period)
    motif = np.arange(period)
    Lq = 3 * R + 2
    q = profile(onehot(np.resize(motif, Lq)), const_tr(Lq), rng)
    tg = []
    for L, phase in ((R - 3, 0), (3 * R + 7, 0), (2 * R + 1, period - 1)):
        tg.append(profile(onehot(np.resize(np.roll(motif, -phase), L)), const_tr(L), rng))
    return Case(f"F2-periodic-R{R}-p{period}", q, tg, shift=0.0,
                expect={"best_tie": 10, f"best_rows_in_strip@R{R}": 1, f"best_cross_strip@R{R}": 1})


def f2_segments(R, shift):
    """Matching segments of three cells: query rows 1-3 (X) and 4-6 (W) lie in strip 0, rows R+2..R+4 (Y) in strip
    1; the target holds Y at columns 2-4, W at 8-10 and X at 14-16.  The three segment ends tie exactly; row-major
    first occurrence picks (3,16), but a column-major sweep meets (6,10) first inside strip 0 and (R+4,4) first
    overall.  A second target repeats X at columns 2-4 and 10-12: a tie within one row."""
    rng = np.random.default_rng(7 * R)
    Lq = R + 9
    ql = np.full(Lq, 6)
    ql[0:3], ql[3:6], ql[R + 1:R + 4] = 0, 1, 2
    q = profile(onehot(ql), const_tr(Lq), rng)
    tl = np.full(20, 5)
    tl[1:4], tl[7:10], tl[13:16] = 2, 1, 0
    t2 = np.full(15, 5)
    t2[1:4], t2[9:12] = 0, 0
    tg = [profile(onehot(tl), const_tr(20), rng), profile(onehot(t2), const_tr(15), rng)]
    return Case(f"F2-segments-R{R}-shift{shift:g}", q, tg, shift=shift,
                expect={"best_tie": 3, f"best_rows_in_strip@R{R}": 1, f"best_cross_strip@R{R}": 1,
                        f"best_inverted_in_strip@R{R}": 1, f"best_inverted_cross_strip@R{R}": 1})


def f3_hhm(seed):
    """Continuous emissions from a pool of 5 columns and transitions -k/1000 ('*' = NEG), as HHM records store them."""
    rng = np.random.default_rng(seed)
    pool = rng.dirichlet(np.ones(20) * 0.5, 5).astype(np.float32) * np.float32(4.0)
    ks = np.array([0, 415, 1000, 1415, 2000, 3000])

    def tr(L):
        t = (np.float32(-1) * rng.choice(ks, size=(L + 1, 7)).astype(np.float32)) / np.float32(1000)
        t[rng.random((L + 1, 7)) < 0.05] = NEG
        return t.astype(np.float32)
    Lq = 48
    q = profile(pool[rng.integers(0, 5, Lq)], tr(Lq), rng)
    tg = [profile(pool[rng.integers(0, 5, L)], tr(L), rng) for L in (3, 20, 47, 48, 64, 77, 100, 120)]
    return Case(f"F3-hhm-s{seed}", q, tg, expect=dict(mm_tie=5, gd_tie=20, im_tie=20, mi_tie=20))


def _synth_targets(rng, lens, qcols=None):
    return [synth.prepared_profile(int(L), rng, qcols if (qcols is not None and k % 2 == 0) else None, noise=0.3)
            for k, L in enumerate(lens)]


def f4_special():
    """The special-value cases (a list)."""
    out = []
    # -0.0 emission columns: dot20 == -0.0, log2f4 must mask the sign bit (score -127, not +129)
    rng = np.random.default_rng(41)
    qp, qtr, qss, qpav, qcols = synth.query_profile(30, 41)
    tg = _synth_targets(rng, (12, 25, 40, 60), qcols)
    for k, (p, tr, ss) in enumerate(tg):
        cols = [1 + k, p.shape[0] // 2, p.shape[0] - 2] if k < 3 else list(range(1, p.shape[0] - 1))
        p[cols] = np.float32(-0.0)
    out.append(Case("F4-negzero-columns", (qp, qtr, qss), tg, expect=dict(negzero_dot=20)))
    # transitions exactly +0.0 / -0.0 with egq = egt = 0: the boundary cells are -0.0
    rng = np.random.default_rng(42)
    Lq = 24
    z = np.float32([0.0, -0.0])
    q = profile(lattice_em(Lq, rng), rng.choice(z, size=(Lq + 1, 7)), rng)
    tg = [profile(lattice_em(L, rng), rng.choice(z, size=(L + 1, 7)), rng) for L in (1, 7, 24, 40)]
    out.append(Case("F4-signed-zero-transitions", q, tg, shift=0.0,
                    expect=dict(mm_tie=500, gd_tie=30, im_tie=30, dg_tie=30, mi_tie=30, best_tie=1)))
    # disjoint support: dot20 == +0.0 on every cell of a column
    rng = np.random.default_rng(43)
    Lq = 20
    qP = rng.dirichlet(np.ones(10), Lq).astype(np.float32)
    q = profile(np.concatenate([qP, np.zeros((Lq, 10), np.float32)], 1), lattice_tr(Lq, rng), rng)
    tg = []
    for L in (5, 19, 33):
        P = rng.dirichlet(np.ones(20), L).astype(np.float32)
        P[rng.random(L) < 0.5, :10] = 0.0
        tg.append(profile(P, lattice_tr(L, rng), rng))
    out.append(Case("F4-zero-dot", q, tg, expect=dict(zero_dot=50)))
    # subnormal dot products (products below FLT_MIN, some underflowing to zero) and overflowing ones (+inf)
    for name, scale in (("F4-subnormal-dot", 1e-20), ("F4-overflow-dot", 1e20)):
        rng = np.random.default_rng(44 if scale < 1 else 45)
        Lq = 20
        q = profile(rng.dirichlet(np.ones(20), Lq) * scale * rng.uniform(0.1, 10, (Lq, 1)), lattice_tr(Lq, rng), rng)
        tg = [profile(rng.dirichlet(np.ones(20), L) * scale * rng.uniform(0.1, 10, (L, 1)), lattice_tr(L, rng), rng)
              for L in (4, 21, 36)]
        out.append(Case(name, q, tg, expect=dict(subnormal_dot=100) if scale < 1 else dict(inf_dot=100)))
    # chains saturated at -FLT_MAX and -inf (local and global)
    rng = np.random.default_rng(46)
    Lq = 22
    sat = (0.0, -1.0, -float(FMAX), -np.inf)
    q = profile(lattice_em(Lq, rng), lattice_tr(Lq, rng, sat, (.4, .3, .2, .1)), rng)
    tg = [profile(lattice_em(L, rng), lattice_tr(L, rng, sat, (.4, .3, .2, .1)), rng) for L in (3, 22, 35)]
    out.append(Case("F4-saturated-chains", q, tg, expect=dict(mm_tie=50, neginf_state=50)))
    out.append(Case("F4-saturated-chains-global", q, tg, local=False, egq=0.5, egt=0.25,
                    expect=dict(mm_tie=50, neginf_state=50)))
    # every cell switched off: score -FLT_MAX, (i2, j2) = (0, 0), one backtrace step
    rng = np.random.default_rng(47)
    qp, qtr, qss, qpav, qcols = synth.query_profile(19, 47)
    tg = _synth_targets(rng, (1, 9, 30), qcols)
    out.append(Case("F4-all-cells-off", (qp, qtr, qss), tg, q_ranges=((1, 19),)))
    # global mode with the last row and the last column switched off: no end cell can be the maximum
    tg = _synth_targets(rng, (26, 26, 26), qcols)
    out.append(Case("F4-global-end-cells-off", (qp, qtr, qss), tg, local=False, egq=0.1, egt=0.2,
                    q_ranges=((19, 19),), t_ranges=((26, 26),)))
    return out


def f5_padding(shift):
    """One long lane (Lmax 90) and short lanes whose last column matches every query row (Si = 4 per cell): along
    the padding, which repeats that column, the diagonal keeps growing far beyond the real best cell."""
    rng = np.random.default_rng(51)
    Lq = 40
    q = profile(onehot(np.zeros(Lq, int), 4.0), const_tr(Lq), rng)
    tg = [profile(lattice_em(90, rng, 3) + onehot(np.full(90, 0), 0.25), lattice_tr(90, rng), rng)]
    for L in (1, 5, 9, 12, 31):
        P = onehot(rng.integers(1, 4, L))            # no match with the query ...
        P[-1] = onehot([0], 4.0)[0]                  # ... except the last column: dot20 = 16, Si = 4
        tg.append(profile(P, lattice_tr(L, rng), rng))
    return Case(f"F5-padding-shift{shift:g}", q, tg, shift=shift, expect=dict(pad_win=100))


def f6_short_query(Lq):
    """Query length Lq (around a strip height) with lattice rows, against lattice and random targets."""
    rng = np.random.default_rng(600 + Lq)
    q = profile(lattice_em(Lq, rng), lattice_tr(Lq, rng), rng)
    tg = [profile(lattice_em(L, rng), lattice_tr(L, rng), rng) for L in (1, 2, Lq, 2 * Lq + 3)]
    tg += _synth_targets(rng, (1, 17, 70))
    return Case(f"F6-Lq{Lq}", q, tg, shift=0.0)


F6_LQ = sorted({v for R in STRIP_ROWS for v in (1, 2, 3, R - 1, R, R + 1, 4 * R - 1, 4 * R + 1)})


def census_cases():
    """F1-F5: the cases small enough for the census and the compiled reference (Lq <= 64, Lt <= 128)."""
    out = [f1_lattice(1, 0.0), f1_lattice(2, -0.03)]
    out += [f2_periodic(R, p) for R in STRIP_ROWS for p in (1, 2, 3)]
    out += [f2_segments(R, s) for R in STRIP_ROWS for s in (0.0, -0.03)]
    out += [f3_hhm(3), f3_hhm(4)]
    out += f4_special()
    out += [f5_padding(0.0), f5_padding(-0.03)]
    return out


def all_cases():
    return census_cases() + [f6_short_query(L) for L in F6_LQ]


def case(name):
    for c in all_cases():
        if c.name == name:
            return c
    raise KeyError(name)


# ------------------------------------------------------------------------------------------------------- census

def log2f4(x):
    """log2f4 (the reference's src/hhutil-inl.h) on a float32 array: the sign bit is masked off."""
    u = np.asarray(x, np.float32).view(np.uint32)
    e = ((u & np.uint32(0x7F800000)) >> np.uint32(23)).astype(np.int32) - 127
    e = e.astype(np.float32)
    m = ((u & np.uint32(0x007FFFFF)) | np.uint32(0x3F800000)).view(np.float32)
    p = np.float32(-0.107254423828329604454)
    p = p * m + np.float32(0.688243882994381274313)
    p = p * m + np.float32(-1.75647175389045657003)
    p = p * m + np.float32(2.61761038894603480148)
    p = p * (m - np.float32(1.0))
    return p + e


def dot20(qrow, T):
    """ScalarProd20Vec: four partial sums over a = k mod 4, combined as (r0 + r1) + (r2 + r3)."""
    r = [T[:, a] * qrow[a] for a in range(4)]
    for m in range(1, 5):
        for a in range(4):
            r[a] = T[:, 4 * m + a] * qrow[4 * m + a] + r[a]
    return (r[0] + r[1]) + (r[2] + r[3])


def _sel(a, b):
    """(a > b) ? a : b"""
    return np.where(a > b, a, b)


def padded(t, Lmax):
    """Target t extended to Lmax columns the way a warp job pads a short lane: every extra column repeats the
    operands of column Lt (emissions, ss, tr[Lt-1][M2M,M2D,D2M,D2D,I2M] and tr[Lt][I2I,M2I])."""
    p, tr, ss = t
    Lt = p.shape[0] - 2
    if Lmax <= Lt:
        return t
    P = np.concatenate([p[:Lt + 1], np.repeat(p[Lt:Lt + 1], Lmax - Lt, 0), p[Lt + 1:]])
    hyb = tr[Lt - 1].copy()
    hyb[[I2I, M2I]] = tr[Lt][[I2I, M2I]]
    TR = np.concatenate([tr[:Lt], np.repeat(hyb[None], Lmax - Lt + 1, 0)])
    S = np.concatenate([ss[:Lt + 1], np.repeat(ss[Lt:Lt + 1], Lmax - Lt, 0), ss[Lt + 1:]])
    return P, TR, S


def census(q, t, local=True, egq=0.0, egt=0.0, shift=-0.03, celloff=None, S33=None, ssw=0.11, Lmax=None):
    """Forward pass of hho_viterbi_align in float32 numpy, on target t padded to Lmax columns.

    Returns dict(score, i2, j2, bt[(Lq+1),(Lt+1)], ties=[(i, j)] tied best cells, counts=dict(...)).  Only the cells
    j <= Lt enter score, (i2, j2), bt and the tie counts; the padded cells are only compared with the real best."""
    f32 = np.float32
    qp, qtr, qss = q
    Lq, Lt = qp.shape[0] - 2, t[0].shape[0] - 2
    Lm = max(Lt, Lmax or Lt)
    tp, ttr, tss = padded(t, Lm)
    smin = f32(0.0) if local else -FMAX
    j = np.arange(1, Lm + 1)
    tt1, tt0 = ttr[j - 1], ttr[j]
    t_m2m, t_m2d, t_d2m, t_d2d, t_i2m = tt1[:, M2M], tt1[:, M2D], tt1[:, D2M], tt1[:, D2D], tt1[:, I2M]
    t_i2i, t_m2i = tt0[:, I2I], tt0[:, M2I]
    T = tp[1:Lm + 1]
    pMM = (np.arange(Lm + 1).astype(f32) * f32(-1)) * f32(egt)
    pDG, pMI, pGD, pIM = (np.full(Lm + 1, -FMAX, f32) for _ in range(4))
    MM = np.zeros((Lq + 1, Lm + 1), f32)
    bt = np.zeros((Lq + 1, Lt + 1), np.uint8)
    cnt = dict(mm_tie=0, gd_tie=0, im_tie=0, dg_tie=0, mi_tie=0, negzero_dot=0, zero_dot=0, subnormal_dot=0,
               inf_dot=0, neginf_state=0, nan=0)
    real = j <= Lt
    with np.errstate(over="ignore", invalid="ignore", under="ignore"):
        for i in range(1, Lq + 1):
            q1, q0 = qtr[i - 1], qtr[i]
            q_m2m, q_m2d, q_d2m, q_d2d, q_i2m = q1[M2M], q1[M2D], q1[D2M], q1[D2D], q1[I2M]
            q_i2i, q_m2i = q0[I2I], q0[M2I]
            dMM, dGD, dIM, dDG, dMI = pMM[:-1], pGD[:-1], pIM[:-1], pDG[:-1], pMI[:-1]
            dMM = dMM.copy()
            dMM[0] = f32(-(i - 1)) * f32(egq)
            c = [(dMM + q_m2m) + t_m2m, (dGD + q_m2m) + t_d2m, (dIM + q_i2m) + t_m2m, (dDG + q_d2m) + t_m2m,
                 (dMI + q_m2m) + t_i2m]
            b = np.where(c[0] > smin, 2, 0).astype(np.uint8)
            mm = np.where(smin > c[0], smin, c[0]).astype(f32)
            for code, ck in zip((3, 4, 5, 6), c[1:]):
                b = np.where(ck > mm, code, b).astype(np.uint8)
                mm = np.where(mm > ck, mm, ck).astype(f32)
            cnt["mm_tie"] += int(((sum((ck == mm).astype(int) for ck in c) + (smin == mm)) >= 2)[real].sum())
            x = dot20(qp[i], T)
            cnt["negzero_dot"] += int(((x == 0) & np.signbit(x))[real].sum())
            cnt["zero_dot"] += int(((x == 0) & ~np.signbit(x))[real].sum())
            cnt["subnormal_dot"] += int(((x != 0) & (np.abs(x) < np.finfo(f32).tiny))[real].sum())
            cnt["inf_dot"] += int(np.isinf(x)[real].sum())
            Si = log2f4(x)
            if S33 is not None:
                Si = f32(ssw) * S33[qss[i].astype(int) * 44 + tss[j].astype(int)] + Si
            Si = Si + f32(shift)
            mm = (mm + Si).astype(f32)
            off = np.zeros(Lm, bool)
            if celloff is not None:
                off[:Lt] = celloff[i, 1:Lt + 1] != 0
            mm = np.where(off, mm + -FMAX, mm).astype(f32)
            uMM, uDG, uMI = pMM[1:], pDG[1:], pMI[1:]
            a1, a2 = uMM + q_m2d, uDG + q_d2d
            b |= np.where(a1 > a2, 32, 0).astype(np.uint8)
            cnt["dg_tie"] += int((a1 == a2)[real].sum())
            dg = np.where(off, _sel(a1, a2) + -FMAX, _sel(a1, a2)).astype(f32)
            a1, a2 = (uMM + q_m2m) + t_m2i, (uMI + q_m2m) + t_i2i
            b |= np.where(a1 > a2, 64, 0).astype(np.uint8)
            cnt["mi_tie"] += int((a1 == a2)[real].sum())
            mi = np.where(off, _sel(a1, a2) + -FMAX, _sel(a1, a2)).astype(f32)
            # gap states from the left: a scan along the row
            gd = np.empty(Lm, f32)
            im = np.empty(Lm, f32)
            lMM, lGD, lIM = f32(-i) * f32(egq), -FMAX, -FMAX
            for k in range(Lm):
                a1, a2 = lMM + t_m2d[k], lGD + t_d2d[k]
                if a1 > a2:
                    b[k] |= 8
                if k < Lt and a1 == a2:
                    cnt["gd_tie"] += 1
                g = a1 if a1 > a2 else a2
                a1, a2 = (lMM + q_m2i) + t_m2m[k], (lIM + q_i2i) + t_m2m[k]
                if a1 > a2:
                    b[k] |= 16
                if k < Lt and a1 == a2:
                    cnt["im_tie"] += 1
                h = a1 if a1 > a2 else a2
                if off[k]:
                    g, h = g + -FMAX, h + -FMAX
                gd[k], im[k] = g, h
                lMM, lGD, lIM = mm[k], g, h
            bt[i, 1:] = b[:Lt]
            MM[i, 1:] = mm
            pMM = np.concatenate([[f32(-i) * f32(egq)], mm]).astype(f32)
            pDG = np.concatenate([[-FMAX], dg]).astype(f32)
            pMI = np.concatenate([[-FMAX], mi]).astype(f32)
            pGD = np.concatenate([[-FMAX], gd]).astype(f32)
            pIM = np.concatenate([[-FMAX], im]).astype(f32)
            for s in (mm, dg, mi, gd, im):
                cnt["neginf_state"] += int(np.isneginf(s)[real].sum())
                cnt["nan"] += int(np.isnan(s).sum())
    # best cell: row-major first occurrence, strict '>' (local: every cell; global: row Lq and column Lt)
    cand = np.zeros((Lq + 1, Lt + 1), bool)
    if local:
        cand[1:, 1:] = True
    else:
        cand[Lq, 1:] = True
        cand[1:, Lt] = True
    best, bi, bj = -FMAX, 0, 0
    for i in range(1, Lq + 1):
        row = np.where(cand[i, 1:], MM[i, 1:Lt + 1], -np.inf)
        k = int(np.argmax(row))
        if row[k] > best:
            best, bi, bj = row[k], i, k + 1
    ties = [] if bi == 0 else [(int(a), int(b_)) for a, b_ in zip(*np.nonzero(cand & (MM[:, :Lt + 1] == best)))]
    cnt["best_tie"] = max(0, len(ties) - 1)
    # padded cells that beat the real best (global mode: only row Lq is a candidate row of a padded column)
    pad = MM[1:, Lt + 1:] if local else MM[Lq:, Lt + 1:]
    cnt["pad_win"] = int((pad > best).sum())
    return dict(score=f32(best), i2=bi, j2=bj, bt=bt, ties=ties, counts=cnt)


def tie_kinds(ties, R):
    """How the tied best cells are spread over strips of R rows: rows of one strip, several strips, and pairs whose
    later row has the earlier column (inside a strip / across strips), which a column-major sweep meets first."""
    k = dict(best_rows_in_strip=0, best_cross_strip=0, best_inverted_in_strip=0, best_inverted_cross_strip=0)
    if len(ties) < 2:
        return k
    strips = {}
    for i, j in ties:
        strips.setdefault((i - 1) // R, set()).add(i)
    k["best_rows_in_strip"] = sum(1 for rows in strips.values() if len(rows) > 1)
    k["best_cross_strip"] = len(strips) - 1
    for a, (i1, j1) in enumerate(ties):
        for i2, j2 in ties[a + 1:]:
            if i1 != i2 and (i1 - i2) * (j1 - j2) < 0:
                same = (i1 - 1) // R == (i2 - 1) // R
                k["best_inverted_in_strip" if same else "best_inverted_cross_strip"] += 1
    return k


def case_census(c, S33=None):
    """census() of every target of case c in one warp job (Lmax = the longest target), counts summed."""
    Lmax = max(t[0].shape[0] - 2 for t in c.targets)
    res = [census(c.q, t, celloff=c.celloff(k), S33=S33, Lmax=Lmax, **c.par()) for k, t in enumerate(c.targets)]
    tot = {}
    for r in res:
        for key, v in r["counts"].items():
            tot[key] = tot.get(key, 0) + v
        for R in STRIP_ROWS:
            for key, v in tie_kinds(r["ties"], R).items():
                tot[f"{key}@R{R}"] = tot.get(f"{key}@R{R}", 0) + v
    return res, tot
