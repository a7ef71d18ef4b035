"""The reference's own ``Campaign`` driving ``B200BotorchRecommender`` (baybe_b200/baybe_plugin.py), unmodified.

``baybe`` is imported from ``oracle/_ref`` (installed there by ``build()``, see ``oracle/install_reference.sh``);
its un-installable dependency ``cattrs`` is replaced by the book-keeping stand-in in ``tests/shims``
(serialisation is not on this path).
Without a GPU the engine is replaced by ``tests.helpers.OracleBackedGP`` (same interface, float64 oracle on the
CPU): what is checked HERE is the binding -- subclass gates, hook signature, metadata masks ->
``FilteredSubspaceDiscrete`` -> position masks, index plumbing, pending experiments, subset-generating
constraints, ``Campaign.posterior_stats`` / ``acquisition_values`` / ``joint_acquisition_value``.  The same flow
runs on the CUDA engine in ``tests/test_gpu_campaign.py``.
"""
from __future__ import annotations

import sys
from pathlib import Path

import numpy as np
import pandas as pd
import pytest

ROOT = Path(__file__).resolve().parents[1]
REF = ROOT / "oracle" / "_ref" if (ROOT / "oracle" / "_ref" / "baybe").is_dir() else None
pytestmark = pytest.mark.skipif(REF is None, reason="the reference package (baybe) is not available on this box")


@pytest.fixture(scope="module")
def bb():
    """Import baybe (with the cattrs stand-in) and the plugin; engine replaced by the oracle-backed stand-in
    when there is no GPU."""
    import torch

    # appended, not prepended: the reference tree has its own top-level ``tests`` package, which must not shadow
    # this repo's for processes spawned later in the session (tests/test_distributed_cpu.py)
    for p in (str(ROOT / "tests" / "shims"), str(REF)):
        if p not in sys.path:
            sys.path.append(p)
    import baybe  # noqa: F401
    from baybe_b200 import baybe_plugin, surrogates
    from tests.helpers import OracleBackedGP

    saved = surrogates.DeviceGP
    if not torch.cuda.is_available():
        surrogates.DeviceGP = OracleBackedGP
    yield baybe_plugin
    surrogates.DeviceGP = saved


def _campaign(plugin, hp=True, campaign_kwargs=None, **rec_kwargs):
    from baybe import Campaign
    from baybe.objectives import SingleTargetObjective
    from baybe.parameters import CategoricalParameter, NumericalDiscreteParameter
    from baybe.searchspace import SearchSpace
    from baybe.targets import NumericalTarget

    from baybe_b200.surrogates import GaussianProcessSurrogate

    params = [
        NumericalDiscreteParameter("temperature", values=[60, 70, 80, 90, 100, 110]),
        NumericalDiscreteParameter("concentration", values=[0.1, 0.2, 0.4, 0.8]),
        CategoricalParameter("solvent", values=["A", "B", "C"], encoding="OHE"),
        NumericalDiscreteParameter("time", values=[1, 2, 4]),
    ]
    space = SearchSpace.from_product(params)  # 6*4*3*3 = 216 candidates: BASELINE config 1
    d = len(space.comp_rep_columns)
    hyper = {"lengthscale": np.full(d, 0.9), "noise": 5e-3, "mean_const": 0.0} if hp else None
    rec = plugin.B200BotorchRecommender(surrogate_model=GaussianProcessSurrogate(hyperparameters=hyper), **rec_kwargs)
    camp = Campaign(space, SingleTargetObjective(NumericalTarget("yield")), rec, **(campaign_kwargs or {}))
    return camp, space


def _fake_measure(df: pd.DataFrame, rng) -> pd.DataFrame:
    out = df.copy()
    s = {"A": 0.0, "B": 1.5, "C": -1.0}
    out["yield"] = (50 + 0.2 * (out["temperature"] - 85) - 0.01 * (out["temperature"] - 85) ** 2 + 8 * out["concentration"]
                    + out["solvent"].map(s).astype(float) + 0.5 * out["time"] + rng.normal(0, 0.1, len(out)))
    return out


def test_plugin_passes_the_reference_gates(bb):
    from baybe.recommenders.base import RecommenderProtocol
    from baybe.recommenders.pure.bayesian.base import BayesianRecommender
    from baybe.recommenders.pure.base import PureRecommender
    import inspect

    rec = bb.B200BotorchRecommender()
    assert isinstance(rec, BayesianRecommender) and isinstance(rec, RecommenderProtocol)
    ref_sig = inspect.signature(PureRecommender._recommend_discrete)
    assert list(inspect.signature(bb.B200BotorchRecommender._recommend_discrete).parameters) == list(ref_sig.parameters)
    assert bb.B200BotorchRecommender.supports_discrete_subset_generating_constraints is True
    assert rec.acquisition_function is None  # default picked like the reference: qLogEI
    from baybe.acquisition import qLogEI, qUCB

    assert bb.mirror_acquisition_function(qLogEI()).abbreviation == "qLogEI"
    assert bb.mirror_acquisition_function(qUCB(beta=0.7)).beta == 0.7


def test_campaign_recommend_add_measurements_recommend(bb):
    rng = np.random.default_rng(0)
    camp, space = _campaign(bb, campaign_kwargs={"allow_recommending_already_measured": False})
    # seed measurements: 15 random rows of the space (BASELINE config 1: 15 training points)
    seed_rows = space.discrete.exp_rep.sample(15, random_state=1)
    camp.add_measurements(_fake_measure(seed_rows, rng))
    rec1 = camp.recommend(batch_size=3)
    assert len(rec1) == 3 and rec1.index.is_unique
    assert set(rec1.columns) == {"temperature", "concentration", "solvent", "time"}
    # rows come back from exp_rep with their ORIGINAL index, and Campaign marks them in its metadata
    pd.testing.assert_frame_equal(rec1, space.discrete.exp_rep.loc[rec1.index])
    assert bool(camp._searchspace_metadata.loc[rec1.index, "recommended"].all())
    # measured rows are excluded through FilteredSubspaceDiscrete (allow_recommending_already_measured=False;
    # the Campaign default lets them through, campaign.py:255-259)
    assert len(set(rec1.index) & set(seed_rows.index)) == 0
    assert int(camp._searchspace_metadata["measured"].sum()) == 15
    camp.add_measurements(_fake_measure(rec1, rng))
    rec2 = camp.recommend(batch_size=2)
    assert len(set(rec2.index) & (set(rec1.index) | set(seed_rows.index))) == 0
    # the winners are the greedy arg-max of the engine's own acquisition values over the remaining candidates
    vals = camp.acquisition_values(space.discrete.exp_rep)
    assert isinstance(vals, pd.Series) and vals.index.equals(space.discrete.exp_rep.index)
    # pending experiments: excluded from the candidates and conditioned on
    pend = space.discrete.exp_rep.loc[[int(vals.idxmax())]]
    rec3 = camp.recommend(batch_size=2, pending_experiments=pend)
    assert pend.index[0] not in rec3.index


def test_first_recommendation_is_the_argmax_of_the_acquisition_values(bb):
    rng = np.random.default_rng(3)
    camp, space = _campaign(bb, campaign_kwargs={"allow_recommending_already_measured": False})
    seed_rows = space.discrete.exp_rep.sample(12, random_state=5)
    camp.add_measurements(_fake_measure(seed_rows, rng))
    import torch

    torch.manual_seed(7)  # the sampler seed is drawn from torch's global RNG, like botorch's
    rec = camp.recommend(batch_size=1)
    torch.manual_seed(7)
    vals = camp.acquisition_values(space.discrete.exp_rep)
    remaining = vals.drop(index=seed_rows.index)
    assert rec.index[0] == remaining.idxmax()
    torch.manual_seed(7)  # same sampler seed -> same base samples
    jv = camp.joint_acquisition_value(rec)
    assert abs(jv - float(vals.loc[rec.index[0]])) < 1e-4 * max(1.0, abs(jv))


def test_campaign_posterior_stats_and_fitted_surrogate(bb):
    rng = np.random.default_rng(1)
    camp, space = _campaign(bb, hp=False)  # hyper-parameters are MAP-fitted (needs the device objective on a GPU box)
    import torch

    if not torch.cuda.is_available():
        camp, space = _campaign(bb, hp=True)
    seed_rows = space.discrete.exp_rep.sample(15, random_state=2)
    meas = _fake_measure(seed_rows, rng)
    camp.add_measurements(meas)
    stats = camp.posterior_stats(space.discrete.exp_rep.iloc[:20], stats=("mean", "std", 0.9))
    assert list(stats.columns) == ["yield_mean", "yield_std", "yield_Q_0.9"] and len(stats) == 20
    at_train = camp.posterior_stats(seed_rows)
    assert float((at_train["yield_mean"] - meas["yield"]).abs().max()) < 0.5 * float(meas["yield"].std())
    assert float(at_train["yield_std"].max()) < float(stats["yield_std"].max()) + 1e-6
    surrogate = camp.get_surrogate()
    assert type(surrogate).__name__ == "GaussianProcessSurrogate" and hasattr(surrogate, "posterior_stats")
    acqf = camp.get_acquisition_function()
    x = torch.from_numpy(space.discrete.comp_rep.iloc[:5].to_numpy(dtype=np.float64)).unsqueeze(1)  # [5, 1, d]
    out = acqf(x)
    assert out.shape == (5,) and torch.isfinite(out).all()


def test_minimisation_and_analytic_acquisition_functions(bb):
    from baybe import Campaign
    from baybe.acquisition import UCB, qLogEI
    from baybe.exceptions import IncompatibleAcquisitionFunctionError
    from baybe.objectives import SingleTargetObjective
    from baybe.targets import NumericalTarget

    rng = np.random.default_rng(4)
    camp0, space = _campaign(bb)
    d = len(space.comp_rep_columns)
    from baybe_b200.surrogates import GaussianProcessSurrogate

    hp = {"lengthscale": np.full(d, 0.9), "noise": 5e-3, "mean_const": 0.0}
    rec = bb.B200BotorchRecommender(surrogate_model=GaussianProcessSurrogate(hyperparameters=hp),
                                    acquisition_function=UCB(beta=0.5))
    camp = Campaign(space, SingleTargetObjective(NumericalTarget("yield", minimize=True)), rec,
                    allow_recommending_already_measured=False)
    seed_rows = space.discrete.exp_rep.sample(10, random_state=3)
    meas = _fake_measure(seed_rows, rng)
    camp.add_measurements(meas)
    r = camp.recommend(batch_size=1)
    vals = camp.acquisition_values(space.discrete.exp_rep).drop(index=seed_rows.index)
    assert r.index[0] == vals.idxmax()
    # minimisation: UCB of the NEGATED target -> the recommended point has a low predicted yield
    stats = camp.posterior_stats(space.discrete.exp_rep)
    assert float(stats.loc[r.index[0], "yield_mean"]) < float(stats["yield_mean"].median())
    with pytest.raises(IncompatibleAcquisitionFunctionError):
        camp.recommend(batch_size=2)  # analytic acquisition function, batch > 1 (discrete.py:110-114)
    _ = qLogEI


def test_subset_generating_constraint_is_honoured(bb):
    """``DiscreteBatchConstraint``: every batch must share one value of the constrained parameter
    (botorch/discrete.py:21-75 splits the candidates into subsets and keeps the best joint batch)."""
    from baybe import Campaign
    from baybe.constraints import DiscreteBatchConstraint
    from baybe.objectives import SingleTargetObjective
    from baybe.parameters import CategoricalParameter, NumericalDiscreteParameter
    from baybe.searchspace import SearchSpace
    from baybe.targets import NumericalTarget

    from baybe_b200.surrogates import GaussianProcessSurrogate

    params = [NumericalDiscreteParameter("x", values=[0.0, 0.25, 0.5, 0.75, 1.0]),
              NumericalDiscreteParameter("y", values=[0.0, 0.5, 1.0]),
              CategoricalParameter("cat", values=["p", "q", "r"], encoding="OHE")]
    space = SearchSpace.from_product(params, constraints=[DiscreteBatchConstraint(parameters=["cat"])])
    assert space.discrete.n_subsets > 0
    d = len(space.comp_rep_columns)
    hp = {"lengthscale": np.full(d, 0.7), "noise": 1e-2, "mean_const": 0.0}
    rec = bb.B200BotorchRecommender(surrogate_model=GaussianProcessSurrogate(hyperparameters=hp))
    camp = Campaign(space, SingleTargetObjective(NumericalTarget("t")), rec)
    rows = space.discrete.exp_rep.sample(8, random_state=0)
    meas = rows.copy()
    meas["t"] = rows["x"] - (rows["y"] - 0.5) ** 2 + rows["cat"].map({"p": 0.0, "q": 0.3, "r": -0.2}).astype(float)
    camp.add_measurements(meas)
    batch = camp.recommend(batch_size=3)
    assert len(batch) == 3 and batch["cat"].nunique() == 1


def test_multi_target_objectives_get_per_target_engine_surrogates(bb):
    """SURVEY.md 8f-4: BayBE's own ``CompositeSurrogate`` (surrogates/composite.py:59-181) replicates the engine
    surrogate per modelled quantity; ``Campaign.posterior_stats`` then reports every target, each column identical
    to a single-target campaign on that target; recommending raises the reference's error type (no multi-output
    acquisition function on the engine)."""
    from baybe import Campaign
    from baybe.exceptions import IncompatibleAcquisitionFunctionError
    from baybe.objectives import ParetoObjective, SingleTargetObjective
    from baybe.surrogates.composite import CompositeSurrogate
    from baybe.targets import NumericalTarget

    from baybe_b200.surrogates import GaussianProcessSurrogate

    rng = np.random.default_rng(4)
    camp1, space = _campaign(bb)
    d = len(space.comp_rep_columns)
    hyper = {"lengthscale": np.full(d, 0.9), "noise": 5e-3, "mean_const": 0.0}
    meas = _fake_measure(space.discrete.exp_rep.sample(14, random_state=2), rng)
    meas["cost"] = 3.0 + 0.02 * meas["temperature"] + 2.0 * meas["concentration"] ** 2 + rng.normal(0, 0.05, len(meas))
    obj = ParetoObjective([NumericalTarget("yield"), NumericalTarget("cost", minimize=True)])
    rec = bb.B200BotorchRecommender(surrogate_model=GaussianProcessSurrogate(hyperparameters=hyper))
    camp = Campaign(space, obj, rec)
    camp.add_measurements(meas)
    cands = space.discrete.exp_rep.head(40)
    stats = camp.posterior_stats(cands)
    assert list(stats.columns) == ["yield_mean", "yield_std", "cost_mean", "cost_std"]
    assert isinstance(camp.get_surrogate(), CompositeSurrogate)
    for tgt in ("yield", "cost"):
        single = Campaign(space, SingleTargetObjective(NumericalTarget(tgt, minimize=(tgt == "cost"))),
                          bb.B200BotorchRecommender(surrogate_model=GaussianProcessSurrogate(hyperparameters=hyper)))
        single.add_measurements(meas.drop(columns=[c for c in ("yield", "cost") if c != tgt]))
        ref = single.posterior_stats(cands)
        assert np.allclose(stats[f"{tgt}_mean"], ref[f"{tgt}_mean"], rtol=1e-6, atol=1e-6)
        assert np.allclose(stats[f"{tgt}_std"], ref[f"{tgt}_std"], rtol=1e-6, atol=1e-6)
    with pytest.raises(IncompatibleAcquisitionFunctionError):
        camp.recommend(batch_size=1)


def test_hybrid_space_reaches_the_device_search_through_the_reference_hook(bb, monkeypatch):
    """SURVEY.md 8f-2 glue: a hybrid SearchSpace + qNoisyExpectedImprovement under the unmodified ``Campaign`` ends in
    ``B200BotorchRecommender._recommend_hybrid(searchspace, candidates_exp, batch_size)`` (pure/base.py:300-302), which
    hands the discrete comp-rep rows, the continuous bounds and the engine config to ``baybe_b200.hybrid`` and
    assembles the reference's frame layout (hybrid.py:137-161).  The device search itself is replaced by a recorder
    here (it needs the GPU: tests/test_gpu_zz_hybrid.py)."""
    from baybe import Campaign
    from baybe.acquisition import qNoisyExpectedImprovement
    from baybe.objectives import SingleTargetObjective
    from baybe.parameters import CategoricalParameter, NumericalContinuousParameter, NumericalDiscreteParameter
    from baybe.searchspace import SearchSpace
    from baybe.targets import NumericalTarget

    import baybe_b200.hybrid as hy
    from baybe_b200.surrogates import GaussianProcessSurrogate

    params = [
        NumericalDiscreteParameter("temperature", values=[60, 80, 100]),
        CategoricalParameter("solvent", values=["A", "B"], encoding="OHE"),
        NumericalContinuousParameter("pressure", bounds=(1.0, 5.0)),
        NumericalContinuousParameter("ratio", bounds=(0.0, 1.0)),
    ]
    space = SearchSpace.from_product(params)
    assert space.type.name == "HYBRID"
    d = len(space.comp_rep_columns)
    hyper = {"lengthscale": np.full(d, 0.9), "noise": 5e-3, "mean_const": 0.0}
    rec = bb.B200BotorchRecommender(surrogate_model=GaussianProcessSurrogate(hyperparameters=hyper),
                                    acquisition_function=qNoisyExpectedImprovement())
    camp = Campaign(space, SingleTargetObjective(NumericalTarget("yield")), rec)
    rng = np.random.default_rng(1)
    meas = space.discrete.exp_rep.sample(8, random_state=3, replace=True).reset_index(drop=True)
    meas["pressure"] = rng.uniform(1, 5, len(meas))
    meas["ratio"] = rng.uniform(0, 1, len(meas))
    meas["yield"] = 0.3 * meas["temperature"] + 2 * meas["pressure"] - 5 * (meas["ratio"] - 0.4) ** 2 + rng.normal(0, 0.1, len(meas))
    camp.add_measurements(meas)
    seen = {}

    def fake(gp, acq, disc_comp, cont_bounds, batch_size, pending, n_samples, seed, search=None):
        seen.update(acq=acq, disc=np.array(disc_comp), cb=np.array(cont_bounds), q=batch_size, pending=pending)
        idx = [1, 1, 4][:batch_size]  # the same configuration twice: duplicate index labels must survive
        pts = np.hstack([np.array(disc_comp)[idx], np.array([[2.5, 0.25], [3.5, 0.75], [1.0, 1.0]])[:batch_size]])
        return pts, idx, 0.123

    monkeypatch.setattr(hy, "recommend_hybrid", fake)
    out = camp.recommend(batch_size=3)
    assert seen["acq"].kind == "qNEI" and seen["q"] == 3 and seen["pending"] is None
    assert seen["disc"].shape == (6, len(space.discrete.comp_rep.columns))
    assert np.allclose(seen["cb"], [[1.0, 0.0], [5.0, 1.0]])
    assert list(out.columns) == ["temperature", "solvent", "pressure", "ratio"] and len(out) == 3
    assert np.allclose(out["pressure"], [2.5, 3.5, 1.0]) and np.allclose(out["ratio"], [0.25, 0.75, 1.0])
    exp = space.discrete.exp_rep
    assert out.iloc[0]["temperature"] == exp.iloc[1]["temperature"] and out.iloc[0]["solvent"] == exp.iloc[1]["solvent"]
    assert out.iloc[2]["temperature"] == exp.iloc[4]["temperature"]
