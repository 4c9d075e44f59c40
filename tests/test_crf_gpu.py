"""GPU tests of the context-specific (CRF) query pseudocounts (hhg_query_context_pseudocounts, SURVEY 8a row a12):
context scores on the device + the host tail must equal HMM::AddContextSpecificPseudocounts +
CalculateAminoAcidBackground of the compiled reference, for the query-HMM engine and the prefilter engine."""
import os

import numpy as np
import pytest

from tests import msa_cases
from tests.util import CRF_SAMPLE, bits, ref_data, ref_data_path

pytestmark = pytest.mark.gpu


def test_context_pseudocounts_equal_reference(hhg, gpu_ctx, refshim, tmp_path):
    crf = hhg.capi.Crf(gpu_ctx, ref_data(CRF_SAMPLE))
    assert refshim.set_contxt(ref_data_path(CRF_SAMPLE)) == crf.n_states
    pb = refshim.pb()
    texts = msa_cases.texts()
    for k in (0, 2, 9, len(texts) - 1):                     # incl. the query alignment of the reference's data set
        path = tmp_path / f"m{k}.a3m"
        path.write_bytes(texts[k])
        raw = refshim.msa_to_hmm(str(path))
        for engine, adm in ((0, hhg.capi.Admix.hhm()), (1, hhg.capi.Admix.prefilter())):
            ref_p, ref_pav = refshim.context_pc(raw["f"], raw["neff_m"], raw["neff_hmm"], engine=engine)
            p, pav = crf.pseudocounts(raw["f"], raw["neff_m"], raw["neff_hmm"], pb, adm)
            assert np.array_equal(bits(p), bits(ref_p)), (k, engine)
            assert np.array_equal(bits(pav), bits(ref_pav)), (k, engine)
    crf.close()


def test_default_hhblits_query_path(hhg, gpu_ctx, refshim, tmp_path):
    """Query alignment -> HMM (hhg_msa_to_hmm) -> context pseudocounts -> hhg_query_set, all in the library, then a
    search: the emissions equal the reference's default PrepareQueryHMM branch, the transitions its pseudocount step."""
    qa = msa_cases.texts()[-1]
    path = tmp_path / "q.a3m"
    path.write_bytes(qa)
    raw = hhg.capi.msa_to_hmm(gpu_ctx, qa, refshim.pb())
    crf = hhg.capi.Crf(gpu_ctx, ref_data(CRF_SAMPLE))
    assert refshim.set_contxt(ref_data_path(CRF_SAMPLE)) == crf.n_states
    p, pav = crf.pseudocounts(raw["f"], raw["neff_m"], raw["neff_hmm"], refshim.pb(), hhg.capi.Admix.hhm())
    ref = refshim.msa_to_hmm(str(path))
    ref_p, ref_pav = refshim.context_pc(ref["f"], ref["neff_m"], ref["neff_hmm"], engine=0)
    assert np.array_equal(bits(p), bits(ref_p)) and np.array_equal(bits(pav), bits(ref_pav))
    q = hhg.capi.query_from_a3m(gpu_ctx, qa, refshim.R(), refshim.pb())          # transitions with pseudocounts
    gpu_ctx.set_query(p, q["tr"])
    data = b"".join(t + b"\0" for t in msa_cases.texts()[:3])
    ln = np.array([len(t) + 1 for t in msa_cases.texts()[:3]], np.int64)
    off = np.concatenate([[0], np.cumsum(ln)[:-1]]).astype(np.int64)
    db = hhg.TargetDB.from_a3m(gpu_ctx, data, off, ln, refshim.R(), refshim.pb(), mp=hhg.capi.MsaParams.defaults(wg=1))
    db.apply_null_model(q_pav=pav, pb=refshim.pb(), columnscore=1)
    hits, _ = hhg.viterbi_search(gpu_ctx, db)
    assert len(hits) == 3 and np.all(np.isfinite(hits["score"]))
    db.close(); crf.close()
