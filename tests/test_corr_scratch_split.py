"""Dense batches that split across launches.

The correlation sweeps, and the SAD sweep on colour frames, run a batch in chunks of the pairs that the context's pair
scratch holds (capped at 1.5 GB), so a large batch is served by several launches of the same sweep, each with its own
slice of scratch and its own first pair. For each sweep, a batch sized to need two launches (the second partly filled)
must give, byte for byte, what the same pairs give in batches that fit one launch. The pair count comes from the scratch
bytes per pair, which decide the chunk size (usv_dense_corr.cu: corr_scratch; usv_dense.cu:
dense_scratch_bytes_per_pair)."""
import numpy as np
import pytest

from unsynchronized_stereo_vision_proj325_b200 import _abi, api

PAIR_SCRATCH_CAP = 3 << 29  # usv_capi.cu: kPairScratchCap


def scratch_bytes_per_pair(sweep, w, h, c, tw, th):
    nxc, nyc = w - tw + 1, h - th + 1
    planes = c * h * (((w + 15) & ~15) + 16) if c > 1 else 0
    if sweep == "sad":  # the colour planes of both cameras
        return 2 * planes
    win = nxc * nyc
    return 2 * planes + 2 * win * 16 + h * nxc * 8 + win * (2 * 8 + 4) + 1280


@pytest.fixture
def ctx():
    c = api.Context(0)
    yield c
    c.close()


def _frames(n, h, w, c, shift, seed):
    rng = np.random.default_rng(seed)
    shape = (n, h, w) if c == 1 else (n, h, w, c)
    left = rng.integers(0, 256, size=shape, dtype=np.uint8)
    right = np.roll(left, -shift, axis=2)
    right[:, ::7] ^= 0x11
    return left, right


# (sweep: forced through corr_kernel, or "sad" for the SAD sweep; cost, width, height, channels, template w x h, search_max)
CASES = [
    ("alu", "ncc", 200, 64, 1, 16, 48, 48),
    ("mma", "zncc", 200, 64, 1, 16, 48, 48),
    ("tcgen05", "ncc", 200, 64, 1, 16, 48, 48),
    ("mma", "zncc", 1280, 720, 3, 32, 32, 64),  # bench.py C3: colour planes in scratch
    ("sad", "sad", 1280, 720, 3, 8, 8, 64),  # planes only: the largest batch, about 2 GB of frames
]
KERNEL = {"alu": "dense_corr_argmin_kernel", "mma": "dense_corr_mma_kernel", "tcgen05": "dense_corr_umma_kernel",
          "sad": "dense_sad_argmin_kernel"}


@pytest.mark.gpu
@pytest.mark.parametrize("sweep,cost,w,h,c,tw,th,smax", CASES, ids=["alu-gray-ncc", "mma-gray-zncc", "tcgen05-gray-ncc", "mma-c3-zncc",
                                                                     "sad-c3"])
def test_split_batch_equals_unsplit_batches(ctx, sweep, cost, w, h, c, tw, th, smax):
    per_pair = scratch_bytes_per_pair(sweep, w, h, c, tw, th)
    cap_pairs = PAIR_SCRATCH_CAP // per_pair
    # the scratch holds between cap_pairs and 1.25 cap_pairs + 1 pairs (grow-only allocation with headroom): this batch
    # needs two launches, the second partly filled; the unsplit batches hold half of cap_pairs
    n = cap_pairs + cap_pairs // 4 + max(1, cap_pairs // 8) + 1
    small = max(1, cap_pairs // 2)
    assert n < 2 * cap_pairs
    left, right = _frames(n, h, w, c, shift=9, seed=n)
    p = _abi.make_params(tmpl_w=tw, tmpl_h=th, search_max=smax, cost=cost)
    value = _abi.OUT_RAW_COST if _abi.COST_NAMES[cost] <= _abi.COST_SSD else _abi.OUT_SCORE
    # two calls with half the outputs each keep the host arrays below about 1 GB; the SAD sweep's batch has about ten
    # times the windows, so it takes one 2-byte array per call (raw_cost_u16: 255 * 8 * 8 * 3 < 65535)
    masks = [_abi.OUT_MATCHES | _abi.OUT_DISPARITY_U16, _abi.OUT_RIGHT_INDEX | value | _abi.OUT_DISTANCE]
    if sweep == "sad":
        masks = [_abi.OUT_DISPARITY_U16, _abi.OUT_RAW_COST_U16]
    ctx.corr_kernel("auto" if sweep == "sad" else sweep)
    try:
        # the context's first call also builds its distance table (one launch, once): not part of a call's launches
        ctx.match_dense(left[:1], right[:1], p, mask=masks[1])
        for mask in masks:
            before = ctx.launch_count
            ctx.match_dense(left[:1], right[:1], p, mask=mask)
            per_launch = ctx.launch_count - before
            before = ctx.launch_count
            got = ctx.match_dense(left, right, p, mask=mask)
            launches = ctx.launch_count - before
            assert ctx.last_kernel == KERNEL[sweep]
            assert launches == 2 * per_launch, (launches, per_launch)
            for p0 in range(0, n, small):
                exp = ctx.match_dense(left[p0:p0 + small], right[p0:p0 + small], p, mask=mask)
                assert ctx.last_kernel == KERNEL[sweep]
                for name, arr in exp.items():
                    assert got[name][p0:p0 + small].tobytes() == arr.tobytes(), (name, p0)
            del got
    finally:
        ctx.corr_kernel("auto")
