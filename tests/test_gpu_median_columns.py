"""Element mapping of the temporal median's tile kernels: every byte of a frame has its own median, and that median
depends on the byte's position inside its 16-byte column block and on the block, so a result written to the wrong
byte, or frames of one column mixed into another, cannot go unnoticed.  One frame count per dispatch variant of
vu_temporal_median_u8 (tile kernels for n <= 152 / 232 / 304 / 464 / 608, and the subsample pass of the two-pass path
above 608), odd and even.  The frames are 64 x 1010 x 3 bytes: more tiles than the grid has CTAs, so the persistent
kernels refill their buffer, and a leftover of 384 bytes for the direct kernels."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

from oracle import refport as R  # noqa: E402


@pytest.mark.parametrize("n", [100, 151, 200, 231, 300, 303, 400, 463, 600, 607, 1000])
def test_temporal_median_column_dependent(n):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from video_unscreen_b200 import ops
    h, w = 64, 1010
    m = h * w * 3
    e = np.arange(m)
    mu = ((e % 16) * 16 + (e // 16) % 16).astype(np.int16)   # 0..255: column in the block, then the block
    rng = np.random.default_rng(n)
    frames = np.clip(mu[None] + rng.integers(-3, 4, (n, m)), 0, 255).astype(np.uint8).reshape(n, h, w, 3)
    got = ops.temporal_median(torch.from_numpy(frames).cuda()).cpu().numpy()
    want = R.temporal_median(frames)
    bad = np.flatnonzero(got.reshape(-1) != want.reshape(-1))
    assert bad.size == 0, f"{bad.size} bytes differ, first at byte offsets {bad[:8].tolist()}"
