"""Parity of the joint logp and its gradient with the reference model (abdpymc's ``abd.model``, PyMC's
unconstrained space) on the bundled test cohort, for the one-, two- and three-chunk models.

The reference's values are stored in tests/golden/model_goldens.npz: tests/golden/make_golden.py evaluated
the reference's own ``abd.py`` at each point (PyTensor / PyMC primitives restated in NumPy by
tests/golden/refshim.py and validated by the reference's unit tests; gradient by complex-step
differentiation), so the comparison needs neither PyMC nor the reference package."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("splits", [None, (14,), (14, 20)])
def test_logp_dlogp_matches_pymc(splits, goldens, cohorts):
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from abdpymc_b200 import build
    from abdpymc_b200.engine import AbdEngine

    build.build()
    z, cases = goldens
    keys = [c["key"] for c in cases
            if c["cohort"] == "test_cohort" and not c["ignore_pcrpos"] and tuple(c["splits"]) == (splits or ())]
    assert len(keys) >= 8
    with AbdEngine(cohorts["test_cohort"], splits=splits) as eng:
        for k in keys:
            lp_ref, g_ref = float(z[f"{k}/logp"]), z[f"{k}/grad"]
            lp, g = eng.logp_dlogp(z[f"{k}/q"], z[f"{k}/i_raw"], z[f"{k}/w"])
            assert abs(lp - lp_ref) <= 1e-10 * abs(lp_ref)
            np.testing.assert_allclose(g, g_ref, rtol=1e-9, atol=1e-9)
