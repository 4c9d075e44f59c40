"""The forward kernel and the backtrace on the adversarial inputs of tests/viterbi_cases.py: exact ties between DP
candidates and between best cells (inside a strip, across strips, in padded lanes), special float values, and lengths
at the strip heights and at the C-ABI's limit.  Everything is compared with the C oracle bit for bit (score, (i2,j2),
every backtrace byte, the path), in every forward-kernel configuration, in local, SS, global and cell-off mode; Hit.score
against the compiled reference; the query-batch search against the single-query calls."""
import numpy as np
import pytest

from tests import viterbi_cases as vc
from tests.test_batch_gpu import _hits_equal
from tests.test_kernel_variants_gpu import CONFIGS, env_ctx
from tests.test_viterbi_gpu import _check_against_oracle
from tests.util import bits, golden

pytestmark = pytest.mark.gpu


def _check_celloff(hhg, ctx, oracle, c):
    """Case c with its excluded regions (hhg_set_excluded_regions) through hhg_viterbi_search, against the oracle with
    the same cell-off mask: score bits, (i2,j2), nsteps, matched columns and the path."""
    ctx.set_query(c.q[0], c.q[1], **c.par())
    ctx.set_excluded_regions(c.q_ranges, c.t_ranges)
    db = hhg.TargetDB.from_profiles(ctx, c.targets)
    try:
        hits, paths = hhg.viterbi_search(ctx, db)
    finally:
        ctx.set_excluded_regions()
        db.close()
    for k, t in enumerate(c.targets):
        sc, i2, j2, bt = oracle.viterbi(c.q[0], c.q[1], t[0], t[1], celloff=c.celloff(k), **c.par())
        h = hits[k]
        assert bits(h["score"]) == bits(sc), (c.name, k, h["score"], sc)
        assert (h["i2"], h["j2"]) == (i2, j2), (c.name, k)
        n, i_s, j_s, st, mc = oracle.backtrace(bt, i2, j2)
        assert h["nsteps"] == n and h["matched_cols"] == mc, (c.name, k)
        assert (h["i1"], h["j1"]) == (i_s[n], j_s[n])
        assert np.array_equal(paths[h["path_off"]:h["path_off"] + n], st[1:]), (c.name, k)


def _regions(c):
    """Excluded regions for a case without its own: two query row ranges and one template column."""
    return c.with_(q_ranges=((2, 4), (c.Lq // 2 + 1, c.Lq // 2 + 2)), t_ranges=((3, 3),))


@pytest.mark.parametrize("cfg", CONFIGS, ids=lambda c: ",".join(f"{k[4:]}={v}" for k, v in c.items()))
def test_adversarial_families_match_oracle(hhg, oracle, cfg):
    G = golden()
    with env_ctx(hhg, **cfg) as ctx:
        for c in vc.all_cases():
            if c.q_ranges or c.t_ranges:
                _check_celloff(hhg, ctx, oracle, c)
                continue
            _check_against_oracle(hhg, ctx, oracle, c.q, c.targets, **c.par())
            _check_against_oracle(hhg, ctx, oracle, c.q, c.targets, S33=G["S33"], use_ss=True, **c.par())
            if c.local:
                for egq, egt in ((c.egq, c.egt), (0.25, 0.5)):
                    _check_against_oracle(hhg, ctx, oracle, c.q, c.targets, **dict(c.par(), local=False, egq=egq, egt=egt))
            _check_celloff(hhg, ctx, oracle, _regions(c))


def test_negative_zero_emission_columns(hhg, gpu_ctx, oracle):
    """dot20 of a column of -0.0 emissions is -0.0; the reference's log2f4 masks the sign bit and scores it -127."""
    c = vc.case("F4-negzero-columns")
    hits = _check_against_oracle(hhg, gpu_ctx, oracle, c.q, c.targets, **c.par())
    assert np.all(hits["score"] < 200)            # +129 per cell of such a column would dominate every score


def test_negative_emissions_are_refused(hhg, gpu_ctx):
    c = vc.case("F1-lattice-s1-shift0")
    p, tr, ss = c.targets[3]
    bad = p.copy()
    bad[4, 7] = -0.5
    with pytest.raises(hhg.HhgError, match="negative"):
        hhg.TargetDB.from_profiles(gpu_ctx, [c.targets[0], (bad, tr, ss)])
    qp = c.q[0].copy()
    qp[2, 0] = -1e-30
    with pytest.raises(hhg.HhgError, match="negative"):
        gpu_ctx.set_query(qp, c.q[1])


@pytest.mark.parametrize("name", [c.name for c in vc.census_cases() if c.name[:2] in ("F1", "F2", "F3", "F4")
                                  and c.local and not c.q_ranges])
def test_hit_score_vs_compiled_reference(hhg, gpu_ctx, refshim, name):
    """Hit.score / score_ss (fast_log2 of zero, subnormal and infinite column sums) against the reference."""
    c = vc.case(name)
    qp, qtr, qss = c.q
    refshim.set_query(qp, qtr, vc.pav(c.q), qss)
    S33 = refshim.S33()
    for use_ss in (False, True):
        gpu_ctx.set_query(qp, qtr, qss, S33, use_ss=use_ss, **c.par())
        db = hhg.TargetDB.from_profiles(gpu_ctx, c.targets)
        hits, _ = hhg.viterbi_search(gpu_ctx, db)
        db.close()
        for b in range(0, len(c.targets), refshim.V):
            res = refshim.viterbi(c.targets[b:b + refshim.V], use_ss=use_ss, egq=c.egq, egt=c.egt, shift=c.shift)
            for k in range(len(res)):
                assert bits(hits[b + k]["score"]) == bits(res[k][0]), (use_ss, b + k)
                hs, hss = refshim.hit_score(k)
                assert bits(hits[b + k]["hit_score"]) == bits(hs), (use_ss, b + k, hits[b + k]["hit_score"], hs)
                assert bits(hits[b + k]["score_ss"]) == bits(hss), (use_ss, b + k)


def test_batch_equals_single_queries_on_ties(hhg):
    """hhg_viterbi_search_batch over the F1 / F2 queries (lengths 37, 11..50) == one single-query search per query."""
    cases = [vc.f1_lattice(1, 0.0), vc.f1_lattice(2, -0.03), vc.f2_periodic(8, 1), vc.f2_periodic(16, 3),
             vc.f2_segments(12, 0.0)]
    tg = [t for c in cases for t in c.targets]
    ctx = hhg.Context()
    db = hhg.TargetDB.from_profiles(ctx, tg)
    rng = np.random.default_rng(3)
    req_q = np.repeat(np.arange(len(cases)), len(tg)).astype(np.int32)
    ids = np.tile(np.arange(len(tg)), len(cases)).astype(np.int32)
    perm = rng.permutation(len(ids))
    req_q, ids = req_q[perm], ids[perm]
    hhg.capi.query_set_batch(ctx, [c.q for c in cases], shift=0.0)
    hb, pb = hhg.capi.viterbi_search_batch(ctx, db, req_q, ids)
    for q, c in enumerate(cases):
        ctx.set_query(c.q[0], c.q[1], shift=0.0)
        m = np.nonzero(req_q == q)[0]
        hs, ps = hhg.viterbi_search(ctx, db, ids=ids[m])
        _hits_equal(hb[m], hs)
        for k, r in enumerate(m):
            n = int(hs[k]["nsteps"])
            assert np.array_equal(pb[hb[r]["path_off"]:hb[r]["path_off"] + n], ps[hs[k]["path_off"]:hs[k]["path_off"] + n])
    db.close(); ctx.close()


def test_query_of_32767_rows_fills_the_strip_tag(hhg, oracle):
    """Lq = 32767 at R = 8: 4096 strips, every value of the 12-bit strip field of the hand-off slot tag."""
    rng = np.random.default_rng(71)
    q = vc.synth_query(32767, 71)
    tg = [vc.profile(vc.lattice_em(L, rng) + np.float32(0.5), vc.lattice_tr(L, rng), rng) for L in (1, 5, 17)]
    with env_ctx(hhg, HHG_STRIP_ROWS=8) as ctx:
        _check_against_oracle(hhg, ctx, oracle, q, tg)
        _check_against_oracle(hhg, ctx, oracle, q, tg, local=False, egq=0.01, egt=0.02)


def test_target_of_32767_columns_and_length_limit(hhg, gpu_ctx, oracle):
    from hhsuite_b200 import synth
    rng = np.random.default_rng(72)
    q = vc.synth_query(20, 72)
    tg = [synth.prepared_profile(32767, rng), synth.prepared_profile(9, rng)]
    _check_against_oracle(hhg, gpu_ctx, oracle, q, tg)
    _check_against_oracle(hhg, gpu_ctx, oracle, q, tg, local=False, egq=0.1, egt=0.1)
    with pytest.raises(hhg.HhgError, match="32767"):
        hhg.TargetDB.from_profiles(gpu_ctx, [synth.prepared_profile(32768, rng)])
    qp, qtr, qss = vc.synth_query(32768, 73)
    with pytest.raises(hhg.HhgError):
        gpu_ctx.set_query(qp, qtr)
