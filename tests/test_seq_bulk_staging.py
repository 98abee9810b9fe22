"""The two ways k_frame_seq stages a frame: bulk copies onto mbarriers (rows of an even number of columns whose mask
rows are a multiple of four words, with 16-byte aligned frames) and per-thread cp.async (every other row up to 2048
columns); rows wider than 2048 columns are replayed frame by frame.  Every frame of each replay is held to the oracle
driven along the same pose chain (labels, nn_idx and nn_dist bit for bit, fit totals against exact sums of the
oracle's correspondences), and each case asserts which path its shape took."""
import ctypes as C

import numpy as np
import pytest

from test_closed_loop_exact import check_stats
from test_sequence_outputs import Rings, pose_chain, seq_frames, unpack_mask

gpu = pytest.mark.gpu
PER_FRAME, CP_ASYNC, BULK = 0, 1, 2   # nav_debug_sequence_path

# shape, frames before the checked replay (an odd number swaps the context's map buffers), frames of the checked
# replay (64: poses as kernel parameters, 65: through the device pose ring; both wrap the parity of the two tile
# slots), motion, frames shifted by one double (not 16-byte aligned), path
CASES = [((2, 256), 0, 12, "large", False, BULK),        # one tile: both row ends in one CTA
         ((4, 768), 0, 12, "scrambled", False, BULK),    # three tiles
         ((3, 2048), 0, 12, "empty_row", False, BULK),   # an empty middle map row every other frame
         ((4, 768), 3, 64, "large", False, BULK),
         ((4, 768), 3, 65, "large", False, BULK),
         ((3, 257), 0, 6, "large", False, CP_ASYNC),     # odd width
         ((3, 1800), 0, 6, "scrambled", False, CP_ASYNC),  # mask rows of 113 words
         ((2, 256), 0, 6, "large", True, CP_ASYNC),      # frames 8 bytes off a 16-byte boundary
         ((2, 4100), 0, 5, "large", False, PER_FRAME)]   # wider than one thread-block cluster


def sequence_path(pkg, ctx):
    L = pkg.load_library()
    L.nav_debug_sequence_path.argtypes = [C.c_void_p]
    L.nav_debug_sequence_path.restype = C.c_int
    return L.nav_debug_sequence_path(ctx.h)


@gpu
@pytest.mark.parametrize("shape,lead,k,motion,shifted,path", CASES)
def test_every_frame_matches_oracle_on_its_path(pkg, oracle, synth, shape, lead, k, motion, shifted, path):
    torch = pytest.importorskip("torch")
    r, c = shape
    n = lead + k
    frames = seq_frames(synth, shape, 1, n + 1, motion)
    pred, last, final = pose_chain(n, 1, motion)
    flat = torch.zeros(frames.size + 1, dtype=torch.float64, device="cuda")
    o = 1 if shifted else 0
    flat[o:o + frames.size] = torch.from_numpy(frames.reshape(-1)).cuda()
    frame_bytes = r * c * 3 * 8

    def fptr(f):
        return flat.data_ptr() + o * 8 + f * frame_bytes

    rings = Rings(torch, k, 1, r, c)
    ctx = pkg.Context(r, c, device=0)
    try:
        ctx.slam_init_dev(fptr(0), np.zeros((1, 6)))
        if lead:
            ctx.frontend_sequence_dev(fptr(1), lead, pred[:lead].reshape(-1, 6), last[:lead].reshape(-1, 6),
                                      final[:lead].reshape(-1, 6))
        ctx.frontend_sequence_out_dev(fptr(1 + lead), k, pred[lead:].reshape(-1, 6), last[lead:].reshape(-1, 6),
                                      final[lead:].reshape(-1, 6), **rings.ptrs(rings.spec.keys()))
        ctx.synchronize()
        assert sequence_path(pkg, ctx) == path
    finally:
        ctx.close()
    for name in rings.spec:
        assert rings.guards_intact(name), name
    mask, idx, dist, stats = (rings.get(nm) for nm in ("label_mask", "nn_idx", "nn_dist", "fit_stats"))
    slam = oracle.slam(r, c, 1)
    try:
        slam.init(np.zeros(6), frames[0, 0])
        for f in range(n):
            cloud = frames[f + 1, 0]
            _, corr, _, _ = slam.localize(cloud, pred[f, 0], last[f, 0])
            ofeat, oidx, odist, _ = slam.frontend_frame(cloud, pred[f, 0], last[f, 0], final[f, 0])
            if f < lead:
                continue
            s = f - lead
            lab = ofeat == 1
            assert np.array_equal(unpack_mask(mask[s, 0], c), ofeat), f
            assert np.array_equal(idx[s, 0][lab], oidx[lab]), f
            assert dist[s, 0][lab].tobytes() == odist[lab].tobytes(), f
            assert (idx[s, 0][~lab] == -1).all() and (dist[s, 0][~lab] == -1.0).all(), f
            if motion == "empty_row" and f % 2 == 0:   # frame f + 1 searched the empty row of frame f's map
                q = lab[r // 2]
                assert q.any() and (idx[s, 0][r // 2][q] == -1).all(), f
            check_stats(stats[s, 0], corr, shape)
    finally:
        slam.close()
