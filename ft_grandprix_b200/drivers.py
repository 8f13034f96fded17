"""Driver plugins.

The plugin surface of the reference is kept as is (SURVEY §8 B1): a driver is any object with
`process_lidar(ranges) -> (speed, steering_angle)` (or `process_lidar(ranges, state)`), see
drivers/template.py:1-18 and ft_grandprix/custom.py:1398-1411.  `Fleet.drive_host` runs such
objects unchanged.  This module adds the batched variants of the two bundled drivers

    BatchedNidcDriver  <- ft_grandprix/nidc.py:3-131
    BatchedFastDriver  <- ft_grandprix/fast.py:3-139

as plain torch tensor programs: `process_lidar(ranges[n, 90]) -> (speed[n], steering[n])` on
whatever device `ranges` lives on.  They reproduce the sequential semantics of the Python loops
(SURVEY Appendix D): disparities are found once on the unmodified scan, then extended one
after the other, each reading what earlier ones wrote; np.argmax first-index ties.  The CUDA
kernel behind `Fleet.drive()` (csrc/fleet.cu) is the fast path; these are the reference-shaped
variant users can subclass.
"""
import math

import torch


class LobotomyDriver:
    """ft_grandprix/lobotomy.py:1-3"""
    def process_lidar(self, ranges):
        return 0.0, 0.0


class BatchedLobotomyDriver:
    def process_lidar(self, ranges):
        z = torch.zeros(ranges.shape[0], dtype=torch.float64, device=ranges.device)
        return z, z.clone()


class BatchedNidcDriver:
    """The class constants are the reference row (include/ftgp.h FTGP_DRV_*, names in _lib.DRV_FIELDS); `params`, a
    float64 tensor [n, 10] of such rows, overrides them per scan.  With rows, each row alone decides its driver (the
    class no longer matters), as in Fleet.set_driver_params()."""
    CAR_WIDTH = 0.12                 # nidc.py:5
    SAFETY_PERCENTAGE = 300.         # nidc.py:10
    DIFFERENCE_THRESHOLD = 0.6       # nidc.py:7
    SPEED = 0.5                      # nidc.py:8
    SPEED_DIVISOR = 1.57 * 2         # nidc.py:130
    MAX_STEER = math.radians(90)     # nidc.py:113
    BOOST_SPEED = 7.0                # fast.py:136
    BOOST_MAX_STEER = 0.0            # fast.py:135 (|st| < 0 never holds: no boost)
    BOOST_MIN_REAR_RANGE = 0.5       # fast.py:135
    SPEED_CAP = math.inf             # fast.py:138 (no cap)

    def __init__(self, params=None):
        self.params = params

    @classmethod
    def default_row(cls):
        from ._lib import DRV_FIELDS
        return [float(getattr(cls, name.upper())) for name in DRV_FIELDS]

    def _rows(self, n, device):
        if self.params is None:
            return torch.tensor(self.default_row(), dtype=torch.float64, device=device).expand(n, -1)
        p = torch.as_tensor(self.params, dtype=torch.float64, device=device)
        if p.shape != (n, 10):
            raise ValueError(f"params must be [{n}, 10]")
        return p

    def _extend(self, ranges, p):
        r = ranges.to(torch.float64)
        n, nb = r.shape
        rpp = (2 * math.pi) / nb                                     # nidc.py:121
        eighth = int(nb / 8)                                         # nidc.py:17
        proc = r[:, eighth:nb - eighth].clone()                      # nidc.py:18
        m = proc.shape[1]
        diff = torch.zeros_like(proc)
        diff[:, 1:] = (proc[:, 1:] - proc[:, :-1]).abs()             # nidc.py:26-29
        disp = diff > p[:, 2:3]                                      # nidc.py:31-40 (computed once)
        width = (p[:, 0] / 2) * (1 + p[:, 1] / 100)                  # nidc.py:93
        idx = torch.arange(m, device=r.device).unsqueeze(0)          # [1, m]
        raised = torch.zeros(n, dtype=torch.bool, device=r.device)
        for i in range(1, m):                                        # nidc.py:94-104, in index order
            act = disp[:, i] & ~raised
            a, b = proc[:, i - 1], proc[:, i]
            # np.argmin / np.argmax on 2 elements: first NaN wins, ties -> first
            amin = torch.where(a.isnan(), 0, torch.where(b.isnan(), 1, (b < a).long()))
            amax = torch.where(a.isnan(), 0, torch.where(b.isnan(), 1, (b > a).long()))
            close = i - 1 + amin
            dist = torch.where(amin.bool(), b, a)
            num = torch.ceil(2 * torch.atan(width / (2 * dist)) / rpp)      # nidc.py:57-58
            bad = num.isnan() & act
            raised |= bad                                            # int(nan) raises -> ctrl kept
            act = act & ~bad
            num = torch.nan_to_num(num, nan=0.0)
            right = (amin < amax).unsqueeze(1)
            c = close.unsqueeze(1); k = num.unsqueeze(1)
            cover = torch.where(right, (idx > c) & (idx <= c + k), (idx < c) & (idx >= c - k))
            cover &= act.unsqueeze(1) & (proc > dist.unsqueeze(1))
            proc = torch.where(cover, dist.unsqueeze(1), proc)
        # np.argmax: first maximum; a NaN anywhere wins at its first position
        nan_any = proc.isnan().any(1)
        first_nan = proc.isnan().float().argmax(1)
        mx = torch.nan_to_num(proc, nan=-math.inf).max(1, keepdim=True).values
        first_max = (torch.nan_to_num(proc, nan=-math.inf) == mx).float().argmax(1)
        best = torch.where(nan_any, first_nan, first_max)
        ang = (best.to(torch.float64) - m / 2.0) * rpp               # nidc.py:112
        lim = p[:, 5]                                                # nidc.py:113
        steer = torch.where(ang < -lim, -lim, torch.where(ang > lim, lim, ang))
        return steer, raised, r

    def process_lidar(self, ranges):
        p = self._rows(ranges.shape[0], ranges.device)
        steer, raised, r = self._extend(ranges, p)
        s = p[:, 3] * 5 * (1 - steer.abs() / p[:, 4])                # nidc.py:130, fast.py:138
        slow = torch.where(s < p[:, 9], s, p[:, 9])
        boost = (steer.abs() < p[:, 7]) & (r[:, 0] > p[:, 8])        # fast.py:135-136
        speed = torch.where(boost, p[:, 6], slow)
        self.raised = raised
        return speed, steer


class BatchedFastDriver(BatchedNidcDriver):
    CAR_WIDTH = 0.06                 # fast.py:4
    SPEED_DIVISOR = math.pi          # fast.py:138
    BOOST_MAX_STEER = 0.1            # fast.py:135
    SPEED_CAP = 2.0                  # fast.py:138
