"""CPU tests (authoring container, where oracle/_ref is built): the C restatement against the
UNMODIFIED compiled reference on fresh seeded inputs -- this is what pins the oracle."""
import numpy as np
import pytest

from tests.util import bits


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_restatement_equals_reference_kernel(oracle, refshim, seed):
    from hhsuite_b200 import synth
    rng = np.random.default_rng(seed)
    qp, qtr, qss, qpav, qcols = synth.query_profile(int(rng.integers(40, 200)), seed)
    refshim.set_query(qp, qtr, qpav, qss)
    S33 = refshim.S33()
    tg = [synth.prepared_profile(int(L), rng, qcols if k % 2 else None, noise=0.3)
          for k, L in enumerate(rng.integers(1, 250, refshim.V))]
    co = [(rng.random((qp.shape[0] - 1, t[0].shape[0] - 1)) < 0.1).astype(np.uint8) for t in tg]
    for kw_ref, kw_or in ((dict(), dict()), (dict(use_ss=True), dict(ss=True)), (dict(celloff=co), dict(co=True)),
                          (dict(celloff=co, use_ss=True), dict(co=True, ss=True))):
        res = refshim.viterbi(tg, **kw_ref)
        for k, (tp, ttr, tss) in enumerate(tg):
            okw = {}
            if kw_or.get("ss"):
                okw.update(q_ss=qss, t_ss=tss, S33=S33)
            if kw_or.get("co"):
                okw.update(celloff=co[k])
            sc, i2, j2, bt = oracle.viterbi(qp, qtr, tp, ttr, **okw)
            rs, ri, rj, rbt = res[k]
            assert bits(sc) == bits(rs) and (i2, j2) == (ri, rj)
            assert np.array_equal(bt[1:, 1:], rbt[1:, 1:])
            n1 = refshim.backtrace(k)
            n2 = oracle.backtrace(bt, i2, j2)
            assert n1[0] == n2[0] and n1[4] == n2[4]
            for a, b in zip(n1[1:4], n2[1:4]):
                assert np.array_equal(a[1:], b[1:])


def test_synthetic_hhm_text_roundtrip_through_reference_reader(refshim, tmp_path):
    """The synthetic HHM text is accepted by HMM::Read and PrepareTemplateHMM gives finite DP inputs."""
    from hhsuite_b200 import synth
    from tests.util import ref_data_path
    refshim.load_query_hhm(ref_data_path("query.hhm"))
    f = tmp_path / "s.hhm"
    f.write_text(synth.hhm_text(77, 5, "s77", with_ss=True))
    t = refshim.prepare_template_hhm(str(f))
    assert t["L"] == 77 and np.isfinite(t["p"]).all() and (t["p"][1:78] > 0).all()
    assert t["ss"][1:78].min() >= 11          # ss_pred/ss_conf were read
