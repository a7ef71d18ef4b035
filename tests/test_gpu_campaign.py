"""The real ``Campaign`` -> ``B200BotorchRecommender`` flow of tests/test_campaign_binding.py on the CUDA engine
(no stand-in: ``torch.cuda.is_available()`` keeps ``DeviceGP``).  ``baybe`` comes from ``oracle/_ref`` (the
copy of the unmodified reference package that ``build()`` makes) with the cattrs
stand-in of ``tests/shims``; skipped when the reference package is not installed there."""
from __future__ import annotations

import pytest

from tests.test_campaign_binding import (REF, bb, test_campaign_posterior_stats_and_fitted_surrogate,  # noqa: F401
                                         test_campaign_recommend_add_measurements_recommend,
                                         test_first_recommendation_is_the_argmax_of_the_acquisition_values,
                                         test_minimisation_and_analytic_acquisition_functions,
                                         test_plugin_passes_the_reference_gates,
                                         test_subset_generating_constraint_is_honoured)

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(REF is None, reason="the reference package (baybe) is not available on this box")]


def test_engine_is_the_cuda_one(bb, cuda_device):  # noqa: F811
    from baybe_b200 import surrogates
    from baybe_b200.engine import DeviceGP

    assert surrogates.DeviceGP is DeviceGP
