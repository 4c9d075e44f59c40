"""The adversarial Viterbi inputs of tests/viterbi_cases.py on the CPU: the float32 census restatement must reproduce the
C oracle exactly and find the ties each family is built for, and the oracle must equal the compiled reference on them
(local, SS, cell-off and global mode) -- which is what makes the oracle a trustworthy yardstick for the GPU kernel on
ties and special float values."""
import numpy as np
import pytest

from tests import viterbi_cases as vc
from tests.util import bits

NAMES = [c.name for c in vc.census_cases()]


@pytest.mark.parametrize("name", NAMES)
def test_census_reproduces_oracle_and_counts_ties(oracle, name):
    c = vc.case(name)
    res, tot = vc.case_census(c)
    for k, (t, r) in enumerate(zip(c.targets, res)):
        sc, i2, j2, bt = oracle.viterbi(c.q[0], c.q[1], t[0], t[1], celloff=c.celloff(k), **c.par())
        assert bits(r["score"]) == bits(sc) and (r["i2"], r["j2"]) == (i2, j2), (k, r["score"], sc)
        assert np.array_equal(r["bt"][1:, 1:], bt[1:, 1:]), k
        if name == "F4-all-cells-off" or name == "F4-global-end-cells-off":
            assert sc == -np.finfo(np.float32).max and (i2, j2) == (0, 0), k
            assert oracle.backtrace(bt, i2, j2)[0] == 1
    assert tot["nan"] == 0
    short = {key: (tot.get(key, 0), v) for key, v in c.expect.items() if tot.get(key, 0) < v}
    assert not short, f"{name} no longer produces what it is built for: {short}"


def _masks(c, rng):
    """The case's own cell-off masks, or 10 % of the cells switched off at random."""
    if c.q_ranges or c.t_ranges:
        return [c.celloff(k) for k in range(len(c.targets))]
    return [(rng.random((c.Lq + 1, t[0].shape[0] - 1)) < 0.1).astype(np.uint8) for t in c.targets]


def _compare(oracle, refshim, c, res, k, t, **okw):
    sc, i2, j2, bt = oracle.viterbi(c.q[0], c.q[1], t[0], t[1], **okw)
    rs, ri, rj, rbt = res
    assert bits(sc) == bits(rs) and (i2, j2) == (ri, rj), (c.name, k, sc, rs, (i2, j2), (ri, rj))
    assert np.array_equal(bt[1:, 1:], rbt[1:, 1:]), (c.name, k)
    n1 = refshim.backtrace(k)
    n2 = oracle.backtrace(bt, i2, j2)
    assert n1[0] == n2[0] and n1[4] == n2[4]
    for a, b in zip(n1[1:4], n2[1:4]):
        assert np.array_equal(a[1:], b[1:])


@pytest.mark.parametrize("name", NAMES)
def test_oracle_equals_reference_on_adversarial_inputs(oracle, refshim, name):
    c = vc.case(name)
    rng = np.random.default_rng(len(name))
    qp, qtr, qss = c.q
    refshim.set_query(qp, qtr, vc.pav(c.q), qss)
    S33 = refshim.S33()
    masks = _masks(c, rng)
    base = dict(egq=c.egq, egt=c.egt, shift=c.shift)
    if c.local:
        # local mode: batches of up to V lanes of different lengths, as the reference runs them.  With every real
        # cell of a short lane switched off, the reference's maximum comes from that lane's padding (it applies the
        # mask to columns 1..Lt only), so masks over whole regions run one target per call.
        step = 1 if (c.q_ranges or c.t_ranges) else refshim.V
        for use_ss, co in ((False, bool(c.q_ranges or c.t_ranges)), (True, False), (False, True)):
            for b in range(0, len(c.targets), step):
                chunk = c.targets[b:b + step]
                cm = masks[b:b + step] if co else None
                res = refshim.viterbi(chunk, use_ss=use_ss, celloff=cm, local=True, **base)
                for k, t in enumerate(chunk):
                    okw = dict(local=True, **base)
                    if use_ss:
                        okw.update(q_ss=qss, t_ss=t[2], S33=S33)
                    if co:
                        okw.update(celloff=cm[k])
                    _compare(oracle, refshim, c, res[k], k, t, **okw)
    # global mode: the reference defines it for equal-length lanes only, so one target per call
    gkw = dict(egq=c.egq, egt=c.egt) if not c.local else dict(egq=0.25, egt=0.5)
    gkw["shift"] = c.shift
    for k, t in enumerate(c.targets):
        co = masks[k] if (c.q_ranges or c.t_ranges) else None
        res = refshim.viterbi([t], celloff=None if co is None else [co], local=False, **gkw)
        _compare(oracle, refshim, c, res[0], 0, t, local=False, celloff=co, **gkw)
