"""Class probability rasters without a GPU: a numpy restatement of `b2u_stitch_finalize_probs` reproduces the
reference's `all_classes` / `specific_class` merge (oracle.stitch.merge_tiles, predict.py:226-254, 307-337) from the
accumulators the device stitch builds, and a pixel-interleaved [Y, X, bands] array written through its [bands, Y, X]
view gives the same GeoTIFF as the contiguous planar array."""
import numpy as np
import pytest

from oracle.stitch import merge_tiles
from unet_b200.geotiff import GeoInfo, write_geotiff


def finalize_probs_ref(acc, cnt, c0, nc, x0, w, large_file):
    """what b2u_stitch_finalize_probs writes, [Y, w, nc]: acc fp32 [C, Y, X], cnt uint8 [Y, X]"""
    a, n = acc[c0:c0 + nc, :, x0:x0 + w], cnt[:, x0:x0 + w]
    if large_file:
        out = a.astype(np.int8)                                   # integer sums wrap modulo 256
        out[:, n == 0] = 0
        n8 = np.broadcast_to(n.astype(np.int8), out.shape)
        out[n8 > 0] //= n8[n8 > 0]                                 # numpy floors; counts >= 128 are negative as int8
    else:
        out = np.zeros(a.shape, dtype=np.float32)
        out[:, n > 0] = a[:, n > 0] / n[n > 0].astype(np.float32)
    return np.ascontiguousarray(np.moveaxis(out, 0, 2))


def stitch_accumulators(preds, windows, Y, X, large_file):
    """the device stitch of per-tile probabilities [C, P, P] at pixel windows (x, y, w, h): acc fp32 [C, Y, X] (mode 1:
    np.around(p * 31) summed), cnt uint8 [Y, X]"""
    acc = np.zeros((preds[0].shape[0], Y, X), dtype=np.float32)
    cnt = np.zeros((Y, X), dtype=np.uint8)
    for p, (x, y, w, h) in zip(preds, windows):
        acc[:, y:y + h, x:x + w] += np.around(p * np.float32(31)) if large_file else p
        cnt[y:y + h, x:x + w] += 1
    return acc, cnt


def _tiles(C, overlap_tiles, seed):
    """probabilities of 16 x 16 tiles at a 4-pixel step (16 tiles over an inner pixel: int8 sums pass 127) over a
    40 x 40 area, plus one tile beyond a 20-column gap where no tile is placed (cnt == 0)"""
    rng = np.random.default_rng(seed)
    P = 16
    wins = [(x, y, P, P) for y in range(0, 40 - P + 1, 4) for x in range(0, 40 - P + 1, 4)] if overlap_tiles else []
    wins += [(60, 8, P, P)] + ([] if overlap_tiles else [(0, 0, P, P), (0, 24, P, P)])
    z = rng.normal(size=(len(wins), C, P, P)) * 3
    e = np.exp(z - z.max(1, keepdims=True))
    return [(q / q.sum(0, keepdims=True)).astype(np.float32) for q in e], wins


@pytest.mark.parametrize("large_file", [False, True])
@pytest.mark.parametrize("C,overlap_tiles", [(2, True), (5, True), (3, False)])
def test_restatement_reproduces_the_reference_merge(C, overlap_tiles, large_file):
    preds, wins = _tiles(C, overlap_tiles, seed=C)
    Y, X = 40, 76
    acc, cnt = stitch_accumulators(preds, wins, Y, X, large_file)
    assert (cnt == 0).any()
    if overlap_tiles and large_file:
        assert cnt.max() == 16 and acc.max() > 127                # the int8 sums wrap
    gts = [[float(x), float(w), 1.0, -float(y), float(h), -1.0] for x, y, w, h in wins]
    ref_all, _ = merge_tiles(preds, gts, large_file=large_file, all_classes=True)
    assert ref_all.shape == (C, Y, X)
    got = finalize_probs_ref(acc, cnt, 0, C, 0, X, large_file)
    assert got.dtype == (np.int8 if large_file else np.float32)
    assert np.array_equal(np.moveaxis(got, 2, 0), ref_all)
    for k in (0, C // 2, C - 1):
        ref_k, _ = merge_tiles(preds, gts, large_file=large_file, specific_class=k)
        assert np.array_equal(finalize_probs_ref(acc, cnt, k, 1, 0, X, large_file)[:, :, 0], ref_k)
    # a column window is the same columns of the whole
    assert np.array_equal(finalize_probs_ref(acc, cnt, 1, C - 1, 7, 33, large_file), got[:, 7:40, 1:])


def test_int8_floor_division_rounds_toward_minus_infinity():
    acc = np.array([[[150.0, 150.0, 124.0, 7905.0, 0.0]]], dtype=np.float32)
    cnt = np.array([[4, 5, 4, 255, 0]], dtype=np.uint8)
    got = finalize_probs_ref(acc, cnt, 0, 1, 0, 5, True)[0, :, 0]
    # 150 -> -106 as int8; -106 // 4 = -27 (C would give -26); count 255 is -1 as int8: the sum stays undivided
    assert got.tolist() == [-27, -22, 31, np.int8(np.int32(7905) % 256 - 256), 0]


@pytest.mark.parametrize("dtype", [np.float32, np.int8])
@pytest.mark.parametrize("class_zero", [False, True])
def test_interleaved_view_writes_the_planar_file(tmp_path, dtype, class_zero):
    rng = np.random.default_rng(3)
    hwc = (rng.integers(-3, 40, size=(37, 53, 4)) / (7 if dtype == np.float32 else 1)).astype(dtype)
    hwc[:5, :5] = 0
    geo = GeoInfo((383000.0, 0.2, 0.0, 5819000.0, 0.0, -0.2), (1, 1, 0, 1, 1024, 0, 1, 1), georeferenced=True)
    view = np.moveaxis(hwc, 2, 0)
    assert np.shares_memory(np.ascontiguousarray(np.moveaxis(view, 0, 2)), hwc)   # no transpose copy in write_geotiff
    write_geotiff(tmp_path / "view.tif", view, geo, class_zero=class_zero)
    write_geotiff(tmp_path / "planar.tif", np.ascontiguousarray(view), geo, class_zero=class_zero)
    assert (tmp_path / "view.tif").read_bytes() == (tmp_path / "planar.tif").read_bytes()
