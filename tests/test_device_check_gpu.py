"""One device check behind every entry point (tscm::internal::select_device): a device index past
the visible devices is refused with TSCM_ERR_NO_DEVICE and says so, instead of surfacing as a CUDA
error of the first call made on it."""
import numpy as np
import pytest

from tscm_calib_b200 import capi, remap

NO_DEVICE = 3   # TSCM_ERR_NO_DEVICE


def entry_points(device):
    """Each entry point with arguments that pass its own validation, on `device`."""
    intr = np.array([300.0, 300.0, 320.0, 240.0, 0.1, 0.2, 0.5, 0.0, 0.0])
    job = capi.remap_job(intr, remap.IDENTITY, (300.0, 300.0, 32.0, 32.0), (64, 64))
    C_, B, K = 2, 1, 12
    return {
        "tscm_remap_tables": lambda: capi.remap_tables([job], (64, 64), device=device),
        "tscm_pose_graph_init": lambda: capi.pose_graph_init(
            np.zeros((K, 3)), np.tile(intr, (C_, 1)), np.ones((C_, B), np.uint8), np.zeros((C_, B, 3, 3)),
            np.zeros((C_, B, K, 2)), device=device),
        "tscm_mono_init": lambda: capi.mono_init(
            (4, 3), (640, 480), np.zeros((K, 3)), np.ones(1, np.uint8), np.zeros((1, K, 2)), device=device),
        "tscm_device_fp64_peak": lambda: capi.device_fp64_peak(device),
    }


@pytest.mark.gpu
def test_out_of_range_device_is_no_device_everywhere():
    import torch
    visible = torch.cuda.device_count()
    for name, call in entry_points(visible).items():
        with pytest.raises(capi.TscmError) as e:
            call()
        assert e.value.code == NO_DEVICE, (name, str(e.value))
        assert f"device {visible} does not exist" in str(e.value), (name, str(e.value))
