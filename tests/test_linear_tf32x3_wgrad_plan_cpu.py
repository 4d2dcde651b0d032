"""CPU: the split-K plan of the fp32 weight-gradient kernel (msda_layer_linear_tf32x3_wgrad_supported / _scratch_floats)
against a Python restatement of it.  The library loads without a GPU, so this runs on a CPU-only machine.

Plan (csrc/linear_tf32x3.cu): output tiles of 128 features x 128 inputs; K blocks of 32 rows; the rows are cut into
contiguous slices of at least 8 K blocks, aiming at 148 CTAs in all; every (tile, slice) writes a partial block of
128 x 128 dW floats + 128 db floats."""
import pytest

from dfvod_b200 import _lib


def supported(n, k):
    return n >= 32 and n % 32 == 0 and k >= 32 and k % 32 == 0


def scratch_floats(rows, n, k):
    if not supported(n, k) or rows < 1 or rows >= (1 << 31) - 1024:
        return 0
    tiles = -(-n // 128) * -(-k // 128)
    kblocks = -(-rows // 32)
    want = max(1, 148 // tiles)
    per_split = max(8, -(-kblocks // want))
    splits = -(-kblocks // per_split)
    assert (splits - 1) * per_split < kblocks            # every slice has rows
    return tiles * splits * (128 * 128 + 128)


SHAPES = [(256, 256), (384, 256), (1024, 256), (256, 1024), (32, 32), (32, 64), (96, 256), (160, 352), (48, 256),
          (256, 200), (0, 256), (256, 0), (-32, 64), (31, 32), (4096, 4096)]


@pytest.mark.parametrize("n,k", SHAPES)
def test_supported_matches_plan(n, k):
    assert bool(_lib.load().msda_layer_linear_tf32x3_wgrad_supported(n, k)) == supported(n, k)


@pytest.mark.parametrize("n,k", SHAPES)
@pytest.mark.parametrize("rows", [0, 1, 31, 32, 33, 255, 256, 257, 2400, 5000, 88892, 177784, (1 << 31) - 1025,
                                  (1 << 31) - 1024, -1])
def test_scratch_floats_match_plan(rows, n, k):
    got = _lib.load().msda_layer_linear_tf32x3_wgrad_scratch_floats(rows, n, k)
    assert got == scratch_floats(rows, n, k)
    if not supported(n, k):
        assert got == 0
