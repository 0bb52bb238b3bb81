"""Background fill of the pixels the left-right check rejects, without a GPU: the numpy reference of the rule (the spec
the CUDA row and column passes in csrc/fill.cu are held to by tests/test_lr_fill_gpu.py), its known answers, and what
the fill does to a layered scene according to the CPU oracle, which the GPU output equals bit for bit."""
import numpy as np
import pytest

from oracle import oracle as O
from stereo_depth_b200.synthetic import make_layered_pair
from test_lr_check_cpu import oracle_right_map, reference_check


def keep_mask(dl, dr, tolerance=1.0):
    """The check's predicate: dl finite, yr = c - rint(dl) in [0, W) and |dl - dr[r, yr]| <= tolerance in fp32."""
    dl = np.asarray(dl, np.float32)
    dr = np.asarray(dr, np.float32)
    W = dl.shape[-1]
    c = np.arange(W, dtype=np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        finite = np.isfinite(dl)
        yr = c - np.rint(np.where(finite, dl, 0.0).astype(np.float64))
        inside = finite & (yr >= 0) & (yr < W)
        partner = np.take_along_axis(dr, np.where(inside, yr, 0).astype(np.int64), axis=-1)
        return inside & (np.abs(dl - partner) <= np.float32(tolerance))


def reference_background_fill(dl, dr, tolerance=1.0, invalid=-1.0):
    """dl: unchecked left maps [..., H, W], dr: right maps [..., H, W] in right-image columns.

    Holes are the pixels keep_mask rejects.  In a row with a kept pixel, a hole gets the smaller of the kept values
    that bound its run (dl[b] < dl[a] ? dl[b] : dl[a], the left one on ties), or its one kept neighbour at a border;
    kept pixels keep dl bit for bit.  Rows without a kept pixel copy the first non-empty row when above it, the last
    one when below it, and stay `invalid` in between (all rows of a frame without a kept pixel)."""
    dl = np.asarray(dl, np.float32)
    keep = keep_mask(dl, dr, tolerance)
    shape = dl.shape
    H, W = shape[-2:]
    dl3, keep3 = dl.reshape(-1, H, W), keep.reshape(-1, H, W)
    out = np.full(dl3.shape, np.float32(invalid), np.float32)
    col = np.arange(W)
    for f in range(dl3.shape[0]):
        d, k = dl3[f], keep3[f]
        a = np.maximum.accumulate(np.where(k, col, -1), axis=1)                      # last kept column <= c
        b = np.minimum.accumulate(np.where(k, col, W)[:, ::-1], axis=1)[:, ::-1]    # first kept column >= c
        da = np.take_along_axis(d, np.maximum(a, 0), axis=1)
        db = np.take_along_axis(d, np.minimum(b, W - 1), axis=1)
        both = np.where(db < da, db, da)
        v = np.where((a >= 0) & (b < W), both, np.where(a >= 0, da, db))
        v = np.where(k, d, v)
        rows = np.nonzero(k.any(axis=1))[0]
        if rows.size == 0:
            continue
        out[f, rows] = v[rows]
        out[f, :rows[0]] = v[rows[0]]
        out[f, rows[-1] + 1:] = v[rows[-1]]
    return out.reshape(shape)


def craft(values, keep):
    """(dl, dr) whose check keeps exactly `keep` at tolerance 0: every value lies in (-0.5, 0.5), so the partner of
    column c is column c, and the right map there equals the value for kept pixels and differs by 10 for holes."""
    values = np.asarray(values, np.float32)
    assert np.all(np.abs(values) < 0.5)
    return values, np.where(keep, values, values + np.float32(10)).astype(np.float32)


def fill(values, keep, invalid=-1.0):
    dl, dr = craft(values, keep)
    return reference_background_fill(dl, dr, 0.0, invalid)


def same_bits(a, b):
    return np.array_equal(np.asarray(a, np.float32).view(np.uint32), np.asarray(b, np.float32).view(np.uint32))


# ---- the reference's keep mask is the merged check's -----------------------------------------------------------------

@pytest.mark.parametrize("seed", range(4))
def test_keep_mask_is_the_checks_predicate(seed):
    rng = np.random.default_rng(seed)
    H, W = 6, 40
    dl = (rng.random((3, H, W)) * 8 - 1).astype(np.float32)
    dl[rng.random(dl.shape) < 0.05] = np.nan
    dl[rng.random(dl.shape) < 0.02] = np.inf
    dl[rng.random(dl.shape) < 0.05] = 2.5                      # rint ties
    dr = (rng.random((3, H, W)) * 6).astype(np.float32)
    for tol in (0.5, 1.0, 2.5):
        keep = keep_mask(dl, dr, tol)
        assert 0 < keep.mean() < 1
        inv = np.float32(np.nan)                               # no kept value is NaN: the mask is recoverable
        got = reference_check(dl, dr, tol, inv)
        assert same_bits(got, np.where(keep, dl, inv))


# ---- known answers -----------------------------------------------------------------------------------------------------

def test_interior_run_gets_the_smaller_bound_both_ways():
    k = [True, False, False, True]
    assert fill([[0.3, 0.0, 0.0, 0.1]], k)[0].tolist() == pytest.approx([0.3, 0.1, 0.1, 0.1])
    assert fill([[0.1, 0.4, 0.4, 0.3]], k)[0].tolist() == pytest.approx([0.1, 0.1, 0.1, 0.3])
    # several runs in one row, each with its own bounds
    got = fill([[0.2, 0, 0.4, 0, 0, 0.3, 0.1]], [True, False, True, False, False, True, True])[0]
    assert same_bits(got, np.float32([0.2, 0.2, 0.4, 0.3, 0.3, 0.3, 0.1]))


def test_ties_keep_the_left_value_bit_for_bit():
    got = fill([[-0.0, 0.2, 0.0]], [True, False, True])[0]
    assert same_bits(got, np.float32([-0.0, -0.0, 0.0]))
    got = fill([[0.0, 0.2, -0.0]], [True, False, True])[0]
    assert same_bits(got, np.float32([0.0, 0.0, -0.0]))
    got = fill([[0.25, 0.0, 0.25]], [True, False, True])[0]
    assert same_bits(got, np.float32([0.25, 0.25, 0.25]))


def test_border_runs_get_their_one_neighbour():
    got = fill([[0.4, 0.4, 0.2, 0.1, 0.4, 0.4]], [False, False, True, True, False, False])[0]
    assert same_bits(got, np.float32([0.2, 0.2, 0.2, 0.1, 0.1, 0.1]))


def test_single_kept_pixel_fills_its_row():
    got = fill([[0.4, 0.4, 0.4, -0.3, 0.4]], [False, False, False, True, False])[0]
    assert same_bits(got, np.full(5, -0.3, np.float32))
    got = fill([[0.125]], [True])[0]                           # W = 1
    assert same_bits(got, np.float32([0.125]))


def test_empty_rows_above_below_and_between():
    v = np.full((6, 3), 0.4, np.float32)
    k = np.zeros((6, 3), bool)
    v[1] = [0.1, 0.4, 0.2]
    k[1] = [True, False, True]
    v[4] = [0.3, 0.4, 0.4]
    k[4] = [True, False, False]
    got = fill(v, k)
    assert same_bits(got[0], np.float32([0.1, 0.1, 0.2]))      # above the first non-empty row: a copy of it
    assert same_bits(got[1], np.float32([0.1, 0.1, 0.2]))
    assert np.all(got[2:4] == -1.0)                            # between non-empty rows: invalid
    assert same_bits(got[4], np.float32([0.3, 0.3, 0.3]))
    assert same_bits(got[5], got[4])                           # below the last one: a copy of it


def test_all_rejected_frame_stays_invalid_and_frames_are_independent():
    v = np.full((2, 3, 4), 0.2, np.float32)
    k = np.zeros((2, 3, 4), bool)
    k[1, 1, 2] = True
    got = fill(v, k, invalid=7.0)
    assert np.all(got[0] == 7.0)
    assert np.all(got[1] == np.float32(0.2))


def test_kept_value_equal_to_invalid_is_not_a_hole():
    # invalid_disparity = 0 and a genuine kept 0: a value test would fill it with its neighbours' minimum
    got = fill([[0.3, 0.0, 0.4, 0.2]], [True, True, False, True], invalid=0.0)[0]
    assert same_bits(got, np.float32([0.3, 0.0, 0.0, 0.2]))
    got = fill([[0.3, 0.0, 0.0, 0.4]], [True, False, True, True], invalid=0.0)[0]
    assert same_bits(got, np.float32([0.3, 0.0, 0.0, 0.4]))


def test_nan_invalid():
    v = np.full((4, 3), 0.2, np.float32)
    k = np.zeros((4, 3), bool)
    k[0, 0] = k[3, 2] = True
    got = fill(v, k, invalid=np.nan)
    assert np.all(got[0] == np.float32(0.2)) and np.all(got[3] == np.float32(0.2))
    assert np.all(np.isnan(got[1:3]))
    assert np.all(np.isnan(fill(v, np.zeros_like(k), invalid=np.nan)))


def test_every_value_is_a_kept_value_or_invalid():
    rng = np.random.default_rng(5)
    dl = (rng.random((2, 16, 64)) * 10).astype(np.float32)
    dr = (dl + rng.integers(-3, 4, dl.shape)).astype(np.float32)
    got = reference_background_fill(dl, dr, 1.0, -1.0)
    keep = keep_mask(dl, dr, 1.0)
    assert same_bits(got[keep], dl[keep])
    for f in range(2):
        kept = set(dl[f][keep[f]].view(np.uint32).tolist()) | {np.float32(-1.0).view(np.uint32)}
        assert set(got[f].view(np.uint32).ravel().tolist()) <= kept


# ---- what the fill does to a layered scene, from the oracle ----------------------------------------------------------

def fill_quality(dl, dr, gt, visible, tolerance=1.0):
    """Fractions of pixels with |e| <= 1, unchecked map dl -> filled: on occluded pixels, on all pixels, on visible
    pixels (dr: the right map)."""
    filled = reference_background_fill(dl, dr, tolerance)
    good_plain, good_fill = np.abs(dl - gt) <= 1.0, np.abs(filled - gt) <= 1.0
    occ = ~visible
    return {"occluded": float(occ.mean()), "rejected": float(1.0 - keep_mask(dl, dr, tolerance).mean()),
            "occluded_plain": float(good_plain[occ].mean()), "occluded_filled": float(good_fill[occ].mean()),
            "all_plain": float(good_plain.mean()), "all_filled": float(good_fill.mean()),
            "visible_plain": float(good_plain[visible].mean()), "visible_filled": float(good_fill[visible].mean())}


# Seeds 1 and 3 at 256x512, D = 64 (DESIGN.md §13 lists seeds 1-4): occluded 0.54 -> 0.81 and 0.43 -> 0.93, all pixels
# 0.931 -> 0.941 and 0.916 -> 0.956, visible 0.960 -> 0.951 and 0.965 -> 0.958.
@pytest.mark.parametrize("seed", [1, 3])
def test_fill_beats_the_unchecked_map_on_a_layered_scene(seed):
    H, W, K, D = 256, 512, 2, 64
    left, right, gt, visible = make_layered_pair(H, W, D, seed)
    cfg = O.make_config(height=H, width=W, downscale_factor=K, min_disparity=0, max_disparity=D - 1)
    q = fill_quality(O.run(cfg, left, right)["out"], oracle_right_map(cfg, left, right), gt, visible)
    print(seed, q)
    assert 0.03 < q["occluded"] < 0.15, q
    assert q["occluded_filled"] >= q["occluded_plain"] + 0.15, q
    assert q["all_filled"] >= q["all_plain"] + 0.005, q
    assert q["visible_filled"] >= q["visible_plain"] - 0.012, q


def test_layered_pair_is_consistent():
    H, W, D = 64, 160, 32
    left, right, gt, visible = make_layered_pair(H, W, D, 3)
    assert left.shape == right.shape == (3, H, W) and left.dtype == right.dtype == np.uint8
    assert gt.dtype == np.float32 and visible.dtype == bool
    r, c = np.nonzero(visible)
    t = c - gt[r, c].astype(np.int64)
    diff = right[:, r, t].astype(np.int16) - left[:, r, c].astype(np.int16)
    assert np.abs(diff).max() <= 2                             # visible pixels land where gt says, +-2 of noise
    # a hidden pixel that lands inside the image lands under a nearer one
    hidden = ~visible & ((np.arange(W)[None, :] - gt) >= 0)
    assert hidden.any()
    a, b = make_layered_pair(H, W, D, 3), make_layered_pair(H, W, D, 3)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
