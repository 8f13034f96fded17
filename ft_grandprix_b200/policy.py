"""Neural-network drivers: the torch twin of policy_kernel (include/ftgp.h, FTGP_DRIVER_POLICY).

A policy is one small MLP of a fixed architecture, packed as FTGP_POLICY_FLOATS fp32 values; a fleet holds a bank of
them (Fleet.set_policies) and every car of kind "policy" runs the one its policy id names, inside the fused tick.
PolicyNet is the same function in torch, differentiable, so a policy can be trained with anything that has gradients
and raced on the device after pack(); policy_inputs computes the network's inputs from fleet state the way the kernel
does.

    x[0:90]   ranges / range_clip; a miss, a range >= range_clip and NaN give 1
    x[90:92]  forward and lateral speed in the yaw frame
    x[92]     yaw rate qvel[5]
    x[93:95]  the car's ctrl (speed, steering) at the head of the tick
    x[95]     0
    h1 = tanh(W1 x + b1), h2 = tanh(W2 h1 + b2), z = W3 h2 + b3
    (speed, steering) = (speed_scale tanh(z0), steer_scale tanh(z1))
"""
import math

import numpy as np
import torch
from torch import nn

# include/ftgp.h FTGP_POLICY_*
POLICY_NIN, POLICY_HIDDEN, POLICY_NOUT = 96, 64, 2
POLICY_SCALARS, POLICY_W1, POLICY_B1, POLICY_W2, POLICY_B2, POLICY_W3, POLICY_B3 = 0, 4, 6148, 6212, 10308, 10372, 10500
POLICY_FLOATS = 10504
NBEAMS = 90


class PolicyNet(nn.Module):
    """Three nn.Linear layers (96 -> 64 -> 64 -> 2, tanh) plus the three scalars of a packed policy: range_clip (metres),
    speed_scale and steer_scale.  forward(x [n, 96]) -> [n, 2] = (speed, steering) in the parameters' dtype."""

    def __init__(self, range_clip=10.0, speed_scale=3.0, steer_scale=math.pi / 2):
        super().__init__()
        self.l1 = nn.Linear(POLICY_NIN, POLICY_HIDDEN)
        self.l2 = nn.Linear(POLICY_HIDDEN, POLICY_HIDDEN)
        self.l3 = nn.Linear(POLICY_HIDDEN, POLICY_NOUT)
        # held as the fp32 values a packed policy carries, so that the twin and the kernel scale by the same numbers
        self.range_clip, self.speed_scale, self.steer_scale = (float(np.float32(v)) for v in (range_clip, speed_scale, steer_scale))

    def forward(self, x):
        x = x.to(self.l1.weight.dtype)
        z = self.l3(torch.tanh(self.l2(torch.tanh(self.l1(x)))))
        t = torch.tanh(z)
        return torch.stack((self.speed_scale * t[:, 0], self.steer_scale * t[:, 1]), dim=1)

    def pack(self):
        """The packed policy: float32 [POLICY_FLOATS] on the CPU (weights input-major, the transpose of nn.Linear's)."""
        row = torch.zeros(POLICY_FLOATS, dtype=torch.float32)
        with torch.no_grad():
            row[POLICY_SCALARS:POLICY_SCALARS + 3] = torch.tensor((self.range_clip, self.speed_scale, self.steer_scale))
            for layer, w, b in ((self.l1, POLICY_W1, POLICY_B1), (self.l2, POLICY_W2, POLICY_B2), (self.l3, POLICY_W3, POLICY_B3)):
                wt = layer.weight.detach().t().to("cpu", torch.float32)
                row[w:w + wt.numel()] = wt.reshape(-1)
                row[b:b + layer.bias.numel()] = layer.bias.detach().to("cpu", torch.float32)
        return row

    @classmethod
    def unpack(cls, row):
        """A float32 PolicyNet from a packed policy (any array-like of POLICY_FLOATS values)."""
        row = torch.as_tensor(row, dtype=torch.float32).detach().cpu().reshape(-1)
        if row.numel() != POLICY_FLOATS:
            raise ValueError(f"a packed policy has {POLICY_FLOATS} floats, not {row.numel()}")
        net = cls(*(float(v) for v in row[POLICY_SCALARS:POLICY_SCALARS + 3]))
        with torch.no_grad():
            for layer, w, b in ((net.l1, POLICY_W1, POLICY_B1), (net.l2, POLICY_W2, POLICY_B2), (net.l3, POLICY_W3, POLICY_B3)):
                nin, nout = layer.in_features, layer.out_features
                layer.weight.copy_(row[w:w + nin * nout].reshape(nin, nout).t())
                layer.bias.copy_(row[b:b + nout])
        return net


def policy_inputs(ranges, qpos, qvel, ctrl, clip):
    """The network inputs x [n, 96] float32 from fleet state on any device: ranges [n, 90], qpos [n, >= 7], qvel
    [n, >= 6], ctrl [n, 2] (the ctrl at the head of the tick), clip: range_clip, a number or [n] (each car's policy's)."""
    r = torch.as_tensor(ranges).to(torch.float32)
    n = r.shape[0]
    clip = torch.as_tensor(clip, dtype=torch.float32, device=r.device).expand(n)[:, None]
    x = torch.zeros(n, POLICY_NIN, dtype=torch.float32, device=r.device)
    x[:, :NBEAMS] = torch.where((r >= 0) & (r < clip), r / clip, torch.ones_like(r))
    q = torch.as_tensor(qpos).to(r.device, torch.float64)
    v = torch.as_tensor(qvel).to(r.device, torch.float64)
    w, qx, qy, qz = q[:, 3], q[:, 4], q[:, 5], q[:, 6]
    yaw = torch.atan2(2 * (w * qz + qx * qy), 1 - 2 * (qy * qy + qz * qz))        # quaternion_to_euler, custom.py:62-76
    c, s = torch.cos(yaw), torch.sin(yaw)
    x[:, 90] = (v[:, 0] * c + v[:, 1] * s).to(torch.float32)
    x[:, 91] = (-v[:, 0] * s + v[:, 1] * c).to(torch.float32)
    x[:, 92] = v[:, 5].to(torch.float32)
    x[:, 93:95] = torch.as_tensor(ctrl).to(r.device, torch.float32)
    return x
