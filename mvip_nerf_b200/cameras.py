"""A table of camera poses refined during training (BARF / NeRF-- style joint refinement).

    poses = CameraPoses(train_poses)                 # [V,3,4] or [V,4,4]
    rgb, *_ = render(H, W, focal, c2w=poses(), pixels=pix, ...)

The module holds one parameter, `se3` [V,6] = (omega, tau) per view, zero-initialised, and returns
c2w_v = [Exp(omega_v) R0_v | t0_v + tau_v]: a rotation correction applied on the world side of the initial rotation and a
translation offset, so the poses stay on SE(3) whatever the optimiser does.  At se3 = 0 the returned table equals the initial
poses bitwise, except that an entry of -0.0 comes back as +0.0 (it is a sum with +0.0 terms; the two compare equal): Exp(0) is
the identity exactly and the product is written as explicit sums of products (no matmul, so no TF32).

The parameter has the dtype of `init`: give float32 poses for training with optim.FusedAdam, which takes fp32 parameters only
(float64 is for checking against float64 references).
"""
import torch
import torch.nn as nn


def _series_cut(dtype):
    # below this theta^2 the closed forms of A, B cancel badly; the series below is then exact to the dtype's precision
    # (first omitted terms theta^6 / 5040 and theta^6 / 40320)
    return 1e-4 if dtype == torch.float64 else 1e-2


def so3_exp(omega):
    """Rodrigues: omega [..., 3] -> R [..., 3, 3] = I + A K + B K^2, K = hat(omega), A = sin t / t, B = (1 - cos t) / t^2.
    Small t uses the series of A and B in t^2, so the value and the gradient at omega = 0 are exact and finite."""
    th2 = (omega * omega).sum(-1)
    small = th2 < _series_cut(omega.dtype)
    safe = torch.where(small, torch.ones_like(th2), th2)
    th = torch.sqrt(safe)
    A = torch.where(small, 1 - th2 / 6 * (1 - th2 / 20), torch.sin(th) / th)
    B = torch.where(small, 0.5 - th2 / 24 * (1 - th2 / 30), (1 - torch.cos(th)) / safe)
    x, y, z = omega[..., 0], omega[..., 1], omega[..., 2]
    # K^2 = omega omega^T - t^2 I
    d = 1 - B * th2
    Bxy, Bxz, Byz = B * x * y, B * x * z, B * y * z
    rows = [torch.stack([d + B * x * x, Bxy - A * z, Bxz + A * y], -1),
            torch.stack([Bxy + A * z, d + B * y * y, Byz - A * x], -1),
            torch.stack([Bxz - A * y, Byz + A * x, d + B * z * z], -1)]
    return torch.stack(rows, -2)


class CameraPoses(nn.Module):
    """Per-view pose corrections: `se3` [V,6] = (omega, tau); forward() -> c2w [V,3,4] = [Exp(omega) R0 | t0 + tau]."""

    def __init__(self, init):
        super().__init__()
        init = torch.as_tensor(init)
        if not init.is_floating_point():
            init = init.float()
        if init.dim() != 3 or init.shape[1] not in (3, 4) or init.shape[2] != 4:
            raise ValueError("CameraPoses: init must be [V,3,4] or [V,4,4], got %s" % (tuple(init.shape),))
        init = init[:, :3, :4].detach().clone()
        self.register_buffer("R0", init[:, :, :3].contiguous())
        self.register_buffer("t0", init[:, :, 3].contiguous())
        self.se3 = nn.Parameter(torch.zeros(init.shape[0], 6, dtype=init.dtype, device=init.device))

    def __len__(self):
        return self.se3.shape[0]

    def forward(self):
        R = so3_exp(self.se3[:, :3])
        R0 = self.R0
        # (Exp(omega) R0)[a][b] = sum_j R[a][j] R0[j][b], summed j = 0, 1, 2 in that order
        rot = R[:, :, 0:1] * R0[:, None, 0, :] + R[:, :, 1:2] * R0[:, None, 1, :] + R[:, :, 2:3] * R0[:, None, 2, :]
        t = self.t0 + self.se3[:, 3:]
        return torch.cat([rot, t[:, :, None]], -1)
