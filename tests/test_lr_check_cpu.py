"""Left-right consistency check, without a GPU: the numpy reference of the check (the spec the CUDA epilogue in
csrc/fill.cu is held to by tests/test_lr_check_gpu.py), its known answers, and what the check does to a synthetic pair
according to the CPU oracle, which the GPU output equals bit for bit.

Right view's map: flip(pipeline(flip R, flip L)).  With L' = flip(R), R' = flip(L), a match L'[y] <-> R'[y - d] is the
match R[c] <-> L[c + d], so the mirrored pair's output, mirrored back, is the disparity map in right-image columns."""
import numpy as np
import pytest

from oracle import oracle as O
from stereo_depth_b200.synthetic import make_pair


def reference_check(dl, dr, tolerance=1.0, invalid=-1.0):
    """dl: left map [..., H, W] (unchecked output), dr: right map [..., H, W] in right-image columns.
    A pixel keeps dl bit for bit if dl is finite, yr = c - rint(dl) is in [0, W) and |dl - dr[r, yr]| <= tolerance in
    fp32; otherwise it becomes `invalid`."""
    dl = np.asarray(dl, np.float32)
    dr = np.asarray(dr, np.float32)
    W = dl.shape[-1]
    c = np.arange(W, dtype=np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        finite = np.isfinite(dl)
        yr = c - np.rint(np.where(finite, dl, 0.0).astype(np.float64))
        inside = finite & (yr >= 0) & (yr < W)
        yi = np.where(inside, yr, 0).astype(np.int64)
        partner = np.take_along_axis(dr, yi, axis=-1)
        ok = inside & (np.abs(dl - partner) <= np.float32(tolerance))   # fp32 subtract; NaN compares false
    return np.where(ok, dl, np.float32(invalid)).astype(np.float32)


def oracle_right_map(cfg, left, right, mode=O.MODE_SAFE):
    """flip(oracle(flip R, flip L)): the right view's disparity map, right-image columns."""
    return O.run(cfg, right[:, :, ::-1], left[:, :, ::-1], mode=mode)["out"][:, ::-1]


def left_ground_truth(g):
    """make_pair's g is indexed by the RIGHT column (right[:, r, c] = left[:, r, c + g]).  Forward-warp it to the left
    view: where two right pixels land on one left pixel the larger disparity wins; left pixels nothing lands on are
    occluded (NaN)."""
    H, W = g.shape
    gl = np.full((H, W), -1, np.int64)
    rows = np.repeat(np.arange(H), W)
    cols = (np.arange(W)[None, :] + g).reshape(-1)
    keep = cols < W
    np.maximum.at(gl, (rows[keep], cols[keep]), g.reshape(-1)[keep])
    return np.where(gl >= 0, gl, np.nan).astype(np.float64)


# ---- known answers of the reference ------------------------------------------------------------------------------

def _row(dl, dr):
    return reference_check(np.array([dl], np.float32), np.array([dr], np.float32))[0]


def test_rint_ties_round_half_to_even():
    W = 8
    dr = np.arange(W, dtype=np.float32) * 100   # every partner distinct
    # c = 5: d = 2.5 -> rint 2 -> yr = 3; d = 3.5 -> rint 4 -> yr = 1
    dl = np.full(W, np.nan, np.float32)
    dl[5] = 2.5
    dr2 = dr.copy()
    dr2[3] = 2.5
    assert _row(dl, dr2)[5] == np.float32(2.5)
    dr2[3], dr2[2] = 0.0, 2.5           # would be the partner with round-half-up
    assert _row(dl, dr2)[5] == -1.0
    dl[5] = 3.5
    dr3 = dr.copy()
    dr3[1] = 3.5
    assert _row(dl, dr3)[5] == np.float32(3.5)
    dl[5] = -0.5                          # rint(-0.5) = -0 -> yr = 5
    dr3[5] = -0.5
    assert _row(dl, dr3)[5] == np.float32(-0.5)


def test_partner_outside_the_image():
    W = 6
    dr = np.zeros(W, np.float32)
    dl = np.full(W, np.nan, np.float32)
    dl[2] = 3.0                           # yr = -1
    dl[3] = 3.0                           # yr = 0: inside
    dl[4] = -1.0                          # yr = 5 = W - 1: inside
    dl[1] = -5.0                          # yr = 6 = W
    dr[0], dr[5] = 3.0, -1.0
    got = _row(dl, dr)
    assert got[2] == -1.0 and got[1] == -1.0
    assert got[3] == 3.0 and got[4] == np.float32(-1.0)


def test_non_finite_inputs():
    W = 5
    dl = np.array([np.nan, np.inf, -np.inf, 0.0, 0.0], np.float32)
    dr = np.array([np.nan, np.inf, -np.inf, np.nan, np.inf], np.float32)
    got = reference_check(dl[None], dr[None], invalid=7.0)[0]
    assert np.all(got == 7.0)
    # (columns 3, 4: a finite left value whose partner is NaN or inf fails too); finite partners that agree pass
    assert reference_check(np.zeros((1, W), np.float32), np.zeros((1, W), np.float32))[0].tolist() == [0.0] * W


def test_tolerance_exactly_the_difference():
    dl = np.array([[0.0, 0.0, 3.75]], np.float32)
    dr = np.array([[0.0, 0.0, 0.0]], np.float32)
    dr[0, 2 - 4] = 3.0                    # c = 2, rint(3.75) = 4 -> yr = -2: outside
    assert reference_check(dl, dr, 1.0)[0, 2] == -1.0
    dl = np.array([[0.0, 1.25, 0.0]], np.float32)   # c = 1, yr = 0
    dr = np.array([[0.5, 9.0, 9.0]], np.float32)
    d = np.float32(np.abs(np.float32(1.25) - np.float32(0.5)))
    assert reference_check(dl, dr, float(d))[0, 1] == np.float32(1.25)
    assert reference_check(dl, dr, float(np.nextafter(d, np.float32(0))))[0, 1] == -1.0


def test_kept_pixels_are_bit_identical():
    rng = np.random.default_rng(3)
    dl = (rng.random((4, 32)) * 6).astype(np.float32)
    dl[0, 0] = -0.0
    dr = dl.copy()
    got = reference_check(dl, dr, 1e9)
    keep = got != -1.0
    assert np.array_equal(got[keep].view(np.uint32), dl[keep].view(np.uint32))


# ---- what the check does, from the oracle ---------------------------------------------------------------------------

def occlusion_stats(left, right, g, H, W, K, D, tolerance=1.0):
    """(occluded fraction, invalid fraction, invalid among occluded, invalid among visible pixels with |e| <= 1)."""
    cfg = O.make_config(height=H, width=W, downscale_factor=K, min_disparity=0, max_disparity=D - 1)
    dl = O.run(cfg, left, right)["out"]
    dr = oracle_right_map(cfg, left, right)
    checked = reference_check(dl, dr, tolerance)
    gt = left_ground_truth(g)
    occluded = np.isnan(gt)
    invalid = checked == -1.0
    good = ~occluded & (np.abs(dl - np.nan_to_num(gt)) <= 1.0)
    return occluded.mean(), invalid.mean(), invalid[occluded].mean(), invalid[good].mean()


@pytest.mark.parametrize("frame", [0, 1])
def test_check_marks_occlusions_not_good_pixels(frame):
    H, W, K, D = 256, 512, 2, 64
    left, right, g = make_pair(H, W, D, seed=70, frame=frame)
    occ, inv, inv_occ, inv_good = occlusion_stats(left, right, g, H, W, K, D)
    assert 0.03 < occ < 0.08, occ
    assert inv_occ >= 0.65, (occ, inv, inv_occ)
    assert inv_good <= 0.02, (occ, inv, inv_good)


def test_mirrored_pipeline_is_the_right_view_map():
    """Where the right pixel is visible in the left view, the right map recovers make_pair's own (right-indexed)
    disparity as well as the left map recovers the forward-warped one."""
    H, W, K, D = 128, 256, 2, 48
    left, right, g = make_pair(H, W, D, seed=71)
    cfg = O.make_config(height=H, width=W, downscale_factor=K, min_disparity=0, max_disparity=D - 1)
    dr = oracle_right_map(cfg, left, right)
    visible = (np.arange(W)[None, :] + g) < W
    assert np.mean(np.abs(dr[visible] - g[visible]) <= 1.0) > 0.9
