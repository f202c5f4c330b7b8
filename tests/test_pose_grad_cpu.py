"""CPU checks of the pose / ray gradient entries: arguments are validated before any CUDA call, and the autograd wrappers
leave the no-grad path alone."""
import ctypes

import pytest


def _lib():
    from mvip_nerf_b200 import _lib
    return _lib.load()


def test_new_entries_validate_before_cuda():
    from mvip_nerf_b200 import _lib
    lib = _lib.load()
    s = _lib.MvipPoints()
    s.n_points = 4
    assert lib.mvip_mlp_input_grad(None, None, None, None, None, None) == -1
    assert b"null" in lib.mvip_last_error()
    assert lib.mvip_rays_pack_backward(None, None, None, 5, 1, 0, 0, 0, 1., 1., None, None, None, None, None) == -1
    assert lib.mvip_rays_from_pose_backward(None, None, 4, 4, 1., 0, 0, 5, 4, 1, 0, 1., None, None, None, None, None) == -1
    assert b"outside" in lib.mvip_last_error()
    assert lib.mvip_rays_from_pose_backward(None, None, 4, 4, 1., 0, 0, 4, 4, 1, 0, 1., None, None, None, None, None) == -1
    # a static camera without somewhere to put its gradient (and the reverse) is refused, not folded into g_c2w
    buf = ctypes.c_void_p(16)
    assert lib.mvip_rays_from_pose_backward(buf, buf, 4, 4, 1., 0, 0, 4, 4, 1, 0, 1., buf, buf, None, buf, None) == -1
    assert b"together" in lib.mvip_last_error()
    assert lib.mvip_rays_from_pose_backward(buf, None, 4, 4, 1., 0, 0, 4, 4, 1, 0, 1., buf, buf, buf, buf, None) == -1
    assert lib.mvip_composite_backward_rays(None, None, None, 3, None, 4, 64, 0, 0, None, None, None, None, None, None, None,
                                            None, None, None, None, None) == -1
    assert lib.mvip_rays_from_pose_backward_workspace_bytes() >= 148 * 24 * 4


def test_no_grad_inputs_take_the_plain_entries():
    import torch
    from mvip_nerf_b200.run import _needs_grad
    c2w = torch.eye(4)[:3]
    assert not _needs_grad(c2w, None)
    assert _needs_grad(c2w.clone().requires_grad_(True))
    with torch.no_grad():
        assert not _needs_grad(c2w.clone().requires_grad_(True))
    import numpy as np
    assert not _needs_grad(np.eye(4))


@pytest.mark.parametrize("name", ["mvip_mlp_input_grad", "mvip_composite_backward_rays", "mvip_rays_pack_backward",
                                  "mvip_rays_from_pose_backward"])
def test_launch_table_lists_new_entries(name):
    from mvip_nerf_b200 import _lib, ops
    assert name in _lib.EXPORTS and name in ops._LAUNCHES
