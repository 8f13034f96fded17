"""GPU: the step kernel runs 64 cars per CTA with M's border in tensor memory.  A fleet of three full waves of CTAs over
148 SMs plus five cars ends in a partial CTA and sends its slow cars through the continuation, which resumes them from
their records (border included) 64 at a time; cut into shards, the same cars are packed into other CTAs.  Cars are
independent, so both must give the same bits."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def test_partial_cta_and_continuation_are_bit_identical_to_shards():
    import ft_grandprix_b200 as ft
    from ft_grandprix_b200.sharding import shard_range
    from conftest import random_poses
    t = ft.Track.bundled("track")
    n, ticks = 64 * 148 * 3 + 5, 30
    poses = random_poses(t.path, n, seed=21, level=True)
    xy = poses[:, :2]; yaw = 2 * np.arctan2(poses[:, 6], poses[:, 3])
    whole = ft.Fleet(t, n)
    whole.reset(xy, yaw); whole.tick(ticks); whole.sync()
    k = 3
    for r in range(k):
        lo, hi = shard_range(n, k, r)
        part = ft.Fleet(t, hi - lo)
        part.reset(xy[lo:hi], yaw[lo:hi]); part.tick(ticks); part.sync()
        for name in ("qpos", "qvel", "warm", "ctrl", "ranges"):
            a, b = getattr(part, name).cpu().numpy(), getattr(whole, name)[lo:hi].cpu().numpy()
            assert np.array_equal(a, b), (name, r)
        part.close()
    whole.close()
