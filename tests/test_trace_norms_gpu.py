"""The two trace quantities that decide a tolerance termination, against the committed golden
vectors: the gradient max-norm (gradient_tolerance; frame part from k_post_eval) and the step
norm (parameter_tolerance; from k_backsub's partials).  test_solve_matches_golden_vectors checks
the costs, flags and final parameters of the same solves."""
import numpy as np
import pytest

from conftest import golden_options, load_golden
from tscm_calib_b200 import capi

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name", ["mono_cfg1", "rig3_small", "rig4_huber", "rig4_cauchy"])
def test_trace_norms_match_golden_vectors(name):
    p, z = load_golden(name)
    a, b, c, s = capi.solve(p, z["init_intrinsics"], z["init_cam_rt"], z["init_board_rt"], golden_options(z))
    assert s.num_iterations == len(z["cost"])
    # the max-norm at the start is one evaluation (1e-10); later ones follow the trajectory (1e-7)
    np.testing.assert_allclose(s.gradient_max_norm[0], z["gradient_max_norm"][0], rtol=1e-10)
    np.testing.assert_allclose(s.gradient_max_norm[1:], z["gradient_max_norm"][1:], rtol=1e-7)
    # the bar of test_oracle_solve_matches_golden
    np.testing.assert_allclose(s.step_norm, z["step_norm"], rtol=1e-6, atol=1e-12)
