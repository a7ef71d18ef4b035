"""Round-2 additions that run LAST in the GPU suite (the driver runs it with ``-x``): the multi-target surrogate
flow and the hybrid-space flow of tests/test_campaign_binding.py on the CUDA engine, under the reference's real
``Campaign`` (``oracle/_ref``); skipped when the reference package is not on the box."""
from __future__ import annotations

import numpy as np
import pytest

from tests.test_campaign_binding import (REF, bb,  # noqa: F401
                                         test_multi_target_objectives_get_per_target_engine_surrogates)

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(REF is None, reason="the reference package (baybe) is not available on this box")]


def test_hybrid_campaign_recommends_a_batch_on_the_device(bb, cuda_device):  # noqa: F811
    """Hybrid SearchSpace + qNoisyExpectedImprovement through ``Campaign.recommend`` with the real device search
    (baybe_b200.hybrid): the batch has the reference's frame layout, discrete parts are rows of the discrete
    subspace, continuous parts lie inside their bounds, the joint qNEI value is positive."""
    from baybe import Campaign
    from baybe.acquisition import qNoisyExpectedImprovement
    from baybe.objectives import SingleTargetObjective
    from baybe.parameters import CategoricalParameter, NumericalContinuousParameter, NumericalDiscreteParameter
    from baybe.searchspace import SearchSpace
    from baybe.targets import NumericalTarget

    from baybe_b200.surrogates import GaussianProcessSurrogate

    params = [
        NumericalDiscreteParameter("temperature", values=[60, 80, 100]),
        CategoricalParameter("solvent", values=["A", "B"], encoding="OHE"),
        NumericalContinuousParameter("pressure", bounds=(1.0, 5.0)),
        NumericalContinuousParameter("ratio", bounds=(0.0, 1.0)),
    ]
    space = SearchSpace.from_product(params)
    d = len(space.comp_rep_columns)
    hyper = {"lengthscale": np.full(d, 0.9), "noise": 5e-3, "mean_const": 0.0}
    rec = bb.B200BotorchRecommender(surrogate_model=GaussianProcessSurrogate(hyperparameters=hyper),
                                    acquisition_function=qNoisyExpectedImprovement())
    camp = Campaign(space, SingleTargetObjective(NumericalTarget("yield")), rec)
    rng = np.random.default_rng(1)
    meas = space.discrete.exp_rep.sample(10, random_state=3, replace=True).reset_index(drop=True)
    meas["pressure"] = rng.uniform(1, 5, len(meas))
    meas["ratio"] = rng.uniform(0, 1, len(meas))
    meas["yield"] = (0.03 * meas["temperature"] + 0.5 * meas["pressure"] - 5 * (meas["ratio"] - 0.4) ** 2
                     + rng.normal(0, 0.05, len(meas)))
    camp.add_measurements(meas)
    out = camp.recommend(batch_size=3)
    assert list(out.columns) == ["temperature", "solvent", "pressure", "ratio"] and len(out) == 3
    assert out["temperature"].isin([60, 80, 100]).all() and out["solvent"].isin(["A", "B"]).all()
    assert ((out["pressure"] >= 1.0) & (out["pressure"] <= 5.0)).all()
    assert ((out["ratio"] >= 0.0) & (out["ratio"] <= 1.0)).all()
    assert rec._last_acq_values and rec._last_acq_values[0] >= 0.0 and np.isfinite(rec._last_acq_values[0])
