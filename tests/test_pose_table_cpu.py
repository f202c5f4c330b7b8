"""CPU checks of the pose-table refinement: the se(3) parametrisation (cameras.CameraPoses) against scipy and float64
autograd, the C entries' argument checks, and the data-parallel reduction of the pose gradient (gloo, two processes)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp


def _init(V, seed, dtype=torch.float64):
    from scipy.spatial.transform import Rotation
    rng = np.random.RandomState(seed)
    R = Rotation.random(V, random_state=seed).as_matrix()
    t = rng.randn(V, 3)
    return torch.tensor(np.concatenate([R, t[:, :, None]], -1), dtype=dtype)


def _omegas():
    rng = np.random.RandomState(3)
    w = [np.zeros(3), np.array([1e-8, 0, 0]), np.array([0, -1e-8, 1e-8]), np.array([3e-3, -2e-3, 1e-3]),
         np.array([0.05, 0.02, -0.07]), np.array([0.0, 0.0, np.pi - 1e-3])]
    w += list(rng.randn(6, 3) * 0.5) + list(rng.randn(4, 3) * 1e-3)
    return np.stack(w)


def test_exp_matches_scipy_rotvec():
    from scipy.spatial.transform import Rotation
    from mvip_nerf_b200.cameras import so3_exp
    w = _omegas()
    got = so3_exp(torch.tensor(w, dtype=torch.float64)).numpy()
    want = Rotation.from_rotvec(w).as_matrix()
    assert np.abs(got - want).max() < 1e-15 * 8, np.abs(got - want).max()
    # float32: within a few ulp of 1 everywhere, including the series / closed-form boundary
    got32 = so3_exp(torch.tensor(w, dtype=torch.float32)).double().numpy()
    assert np.abs(got32 - want).max() < 4e-7, np.abs(got32 - want).max()
    # exactly the identity at 0
    assert torch.equal(so3_exp(torch.zeros(2, 3)), torch.eye(3).expand(2, 3, 3))


def test_camera_poses_identity_at_zero_signed_zeros():
    """-0.0 entries come back as +0.0 (sums with +0.0 terms): equal values, every other bit pattern unchanged"""
    from mvip_nerf_b200.cameras import CameraPoses
    init = torch.tensor([[[1., -0., 0., -0.], [0., 1., -0., 2.], [-0., 0., 1., -0.]]])
    out = CameraPoses(init)()
    assert torch.equal(out, init)
    neg = torch.signbit(init) & (init == 0)
    assert not torch.signbit(out[neg]).any()
    assert torch.equal(out[~neg].view(torch.int32), init[~neg].view(torch.int32))


def test_camera_poses_value_against_scipy():
    from scipy.spatial.transform import Rotation
    from mvip_nerf_b200.cameras import CameraPoses
    w = _omegas()
    V = w.shape[0]
    init = _init(V, 1)
    cam = CameraPoses(init)
    tau = np.random.RandomState(5).randn(V, 3) * 0.1
    with torch.no_grad():
        cam.se3.copy_(torch.tensor(np.concatenate([w, tau], 1)))
    got = cam().detach().numpy()
    R = Rotation.from_rotvec(w).as_matrix() @ init[:, :, :3].numpy()
    t = init[:, :, 3].numpy() + tau
    assert np.abs(got[:, :, :3] - R).max() < 1e-14
    assert np.abs(got[:, :, 3] - t).max() == 0.0


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("shape", [(5, 3, 4), (5, 4, 4)])
def test_camera_poses_identity_at_zero_is_bitwise(dtype, shape):
    from mvip_nerf_b200.cameras import CameraPoses
    init = _init(5, 2, dtype)
    if shape[1] == 4:
        init = torch.cat([init, torch.tensor([0., 0., 0., 1.], dtype=dtype).expand(5, 1, 4)], 1)
    cam = CameraPoses(init)
    assert cam.se3.shape == (5, 6) and cam.se3.dtype == dtype and float(cam.se3.detach().abs().sum()) == 0.0
    assert [n for n, _ in cam.named_parameters()] == ["se3"]
    out = cam()
    assert out.shape == (5, 3, 4) and out.dtype == dtype
    assert torch.equal(out, init[:, :3, :4])
    assert torch.equal(out.view(torch.int64 if dtype == torch.float64 else torch.int32),
                       init[:, :3, :4].contiguous().view(torch.int64 if dtype == torch.float64 else torch.int32))


@pytest.mark.parametrize("scale", [0.0, 1e-8, 1e-3, 0.3])
def test_camera_poses_gradcheck(scale):
    from mvip_nerf_b200.cameras import CameraPoses
    init = _init(3, 4)
    cam = CameraPoses(init)
    x = (torch.tensor(np.random.RandomState(6).randn(3, 6), dtype=torch.float64) * scale).requires_grad_(True)
    assert torch.autograd.gradcheck(lambda x: _with(cam, x), (x,), eps=1e-7, atol=1e-8)


def _with(cam, x):
    """cam's forward at se3 = x, differentiable in x (torch.func.functional_call: the parameter is replaced, not copied)"""
    return torch.func.functional_call(cam, {"se3": x}, ())


def test_camera_poses_gradient_at_zero_is_exact():
    """d c2w / d omega at 0 is hat(e_i) R0 and d c2w / d tau = identity: exact, finite, no 0/0 in the series"""
    from mvip_nerf_b200.cameras import CameraPoses
    init = _init(2, 7)
    cam = CameraPoses(init)
    x = torch.zeros(2, 6, dtype=torch.float64, requires_grad=True)
    J = torch.autograd.functional.jacobian(lambda x: _with(cam, x), x)     # [2,3,4, 2,6]
    assert torch.isfinite(J).all()
    for i in range(3):
        e = torch.zeros(3, dtype=torch.float64)
        e[i] = 1
        hat = torch.tensor([[0, -e[2], e[1]], [e[2], 0, -e[0]], [-e[1], e[0], 0]], dtype=torch.float64)
        for v in range(2):
            assert torch.equal(J[v, :, :3, v, i], hat @ init[v, :, :3])
            assert torch.equal(J[v, :, 3, v, 3 + i], e)


def test_new_entries_validate_before_cuda():
    from mvip_nerf_b200 import _lib
    lib = _lib.load()
    assert lib.mvip_rays_from_poses(None, 1, None, 4, 0, 4, 1., 0., 1., 1, 0, 1., None, None) == -1
    assert lib.mvip_rays_from_poses(None, 1, None, 4, 4, 4, 0., 0., 1., 1, 0, 1., None, None) == -1
    assert b"focal" in lib.mvip_last_error()
    assert lib.mvip_rays_from_poses(None, 1, None, 4, 4, 4, 1., 0., 1., 1, 0, 1., None, None) == -1
    assert b"null" in lib.mvip_last_error()
    assert lib.mvip_rays_from_poses(None, 1, None, 0, 4, 4, 1., 0., 1., 1, 0, 1., None, None) == 0     # empty batch: nothing
    assert lib.mvip_rays_from_poses_backward(None, 2, None, 4, 4, 4, 1., 1, 0, 1., None, None, None, None) == -1
    assert b"null" in lib.mvip_last_error()
    assert lib.mvip_rays_from_poses_backward(None, -1, None, 4, 4, 4, 1., 1, 0, 1., None, None, None, None) == -1
    # workspace: 12 floats per (view, chunk of 1024 entries)
    assert lib.mvip_rays_from_poses_backward_workspace_bytes(4096, 20) == 20 * 4 * 12 * 4
    assert lib.mvip_rays_from_poses_backward_workspace_bytes(0, 3) == 3 * 12 * 4
    assert lib.mvip_rays_from_poses_backward_workspace_bytes(1025, 1) == 2 * 12 * 4


@pytest.mark.parametrize("name", ["mvip_rays_from_poses", "mvip_rays_from_poses_backward"])
def test_launch_table_lists_new_entries(name):
    from mvip_nerf_b200 import _lib, ops
    assert name in _lib.EXPORTS and name in ops._LAUNCHES


def test_ops_refuse_cpu_tensors():
    from mvip_nerf_b200 import ops
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.rays_from_poses(4, 4, 1., torch.zeros(1, 3, 4), torch.zeros(2, 3, dtype=torch.int32), 0., 1.)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.rays_from_poses_backward(torch.zeros(1, 3, 4), torch.zeros(2, 3, dtype=torch.int32), 4, 4, 1., torch.zeros(2, 11))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _pose_sync_worker(rank, world, port):
    """graph.step_syncs, the collectives GraphedTrainStep finishes after its backward: the networks' bucket and the pose table's
    bucket both end as the sums over the ranks, the pose table in a collective of its own after the networks'."""
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    import torch.distributed as dist
    from mvip_nerf_b200 import dist as md
    from mvip_nerf_b200 import graph
    from mvip_nerf_b200.cameras import CameraPoses
    md.init_from_env(backend="gloo")
    torch.manual_seed(0)
    net = torch.nn.Linear(5, 3)
    cam = CameraPoses(torch.eye(4)[:3].expand(4, 3, 4))
    groups = [list(net.parameters())]
    sync, pose_sync = graph.step_syncs(groups, list(cam.parameters()))
    calls = []
    real = dist.all_reduce

    def counting(t, *a, **k):
        calls.append(t.numel())
        return real(t, *a, **k)
    md.dist.all_reduce = counting
    # each rank renders its own pixels: its pose gradient covers only some views
    g_pose = torch.zeros(4, 6)
    g_pose[rank::2] = torch.arange(12, dtype=torch.float32).view(2, 6) + 100 * rank
    cam.se3.grad = g_pose.clone()
    for i, p in enumerate(groups[0]):
        p.grad = torch.full_like(p, float(rank + 1) * (i + 1))
    for s in (sync, pose_sync):
        s.finish()
    md.dist.all_reduce = real
    assert calls == [sum(p.numel() for p in groups[0]), cam.se3.numel()], calls
    want = torch.zeros(4, 6)
    want[0::2] = torch.arange(12, dtype=torch.float32).view(2, 6)
    want[1::2] = torch.arange(12, dtype=torch.float32).view(2, 6) + 100
    assert torch.equal(cam.se3.grad, want)
    for i, p in enumerate(groups[0]):
        assert float((p.grad - 3.0 * (i + 1)).abs().max()) == 0.0
    # frozen networks: only the pose bucket
    assert graph.step_syncs([], list(cam.parameters()))[0] is None
    for s in (sync, pose_sync):
        s.remove()
    dist.barrier()
    dist.destroy_process_group()


def test_world2_gloo_pose_gradient_summed_by_step_syncs():
    mp.spawn(_pose_sync_worker, args=(2, _free_port()), nprocs=2, join=True)
