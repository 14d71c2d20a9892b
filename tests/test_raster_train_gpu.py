"""Tile-free training on the B200: `b2u_crop_train_batch` against torch slicing + flip / rot90, bit for bit, and
`train_geotiff` against `split_raster` + `train_func` on the same data - equal weights, history, metrics and export."""
import math

import numpy as np
import pytest
import torch

from unet_b200 import _lib, ops
from unet_b200.create_tiles import split_raster
from unet_b200.geotiff import GeoInfo, write_geotiff
from unet_b200.reference_api import load_learner, train_func, train_geotiff
from unet_b200.synth import aerial_like_tiles

pytestmark = pytest.mark.gpu

GEO = GeoInfo(geotransform=(383000.0, 0.2, 0.0, 5819000.0, 0.0, -0.2),
              geokeys=(1, 1, 0, 3, 1024, 0, 1, 1, 1025, 0, 1, 1, 3072, 0, 1, 25833), georeferenced=True)


def _bits(a: np.ndarray) -> torch.Tensor:
    """uint16 arrays travel as their int16 bits (torch has few uint16 kernels)"""
    return torch.from_numpy(np.ascontiguousarray(a.view(np.int16) if a.dtype == np.uint16 else a))


@pytest.mark.parametrize("P", [33, 64, 256])
@pytest.mark.parametrize("ldt", [np.uint8, np.float32])
@pytest.mark.parametrize("rdt", [np.uint8, np.uint16, np.int16])
def test_crop_train_batch_matches_torch(rdt, ldt, P):
    lib = _lib.load()
    rng = np.random.default_rng(P)
    C, Y, X = 3, 300, 290
    info = np.iinfo(rdt)
    raster = rng.integers(info.min, info.max, size=(C, Y, X), endpoint=True).astype(rdt)
    labels = (rng.integers(0, 256, size=(Y, X)).astype(np.uint8) if ldt == np.uint8
              else rng.standard_normal((Y, X)).astype(np.float32))
    # every raster edge and corner, and interior windows; each of the eight ops on several windows
    corners = [(0, 0), (0, X - P), (Y - P, 0), (Y - P, X - P), (0, 17), (Y - P, 5), (11, 0), (7, X - P)]
    inner = [(int(rng.integers(0, Y - P + 1)), int(rng.integers(0, X - P + 1))) for _ in range(8)]
    wins = corners + inner
    T = 3 * len(wins)
    y0 = np.array([wins[t % len(wins)][0] for t in range(T)], np.int32)
    x0 = np.array([wins[t % len(wins)][1] for t in range(T)], np.int32)
    op = np.array([t % 8 for t in range(T)], np.int32)
    d = lambda a: a.cuda()
    r_d, l_d = d(_bits(raster)), d(torch.from_numpy(labels))
    t_d = [d(torch.from_numpy(v)) for v in (y0, x0, op)]
    x_d = torch.full((T, C, P, P), 77, dtype=r_d.dtype, device="cuda")
    y_d = torch.full((T, P, P), 77, dtype=l_d.dtype, device="cuda")
    code = {np.uint8: _lib.DT_U8, np.uint16: _lib.DT_U16, np.int16: _lib.DT_I16}[rdt]
    _lib.check(lib.b2u_crop_train_batch(r_d.data_ptr(), code, C, Y, X, l_d.data_ptr(),
                                        _lib.DT_U8 if ldt == np.uint8 else _lib.DT_F32, t_d[0].data_ptr(),
                                        t_d[1].data_ptr(), t_d[2].data_ptr(), T, P, x_d.data_ptr(), y_d.data_ptr(),
                                        ops.stream_ptr()), "b2u_crop_train_batch")
    torch.cuda.synchronize()
    r_t, l_t = _bits(raster), torch.from_numpy(labels)
    for t in range(T):
        xs, ys = r_t[:, y0[t]:y0[t] + P, x0[t]:x0[t] + P], l_t[y0[t]:y0[t] + P, x0[t]:x0[t] + P]
        if op[t] & 4:
            xs, ys = xs.flip(-1), ys.flip(-1)
        xs, ys = torch.rot90(xs, int(op[t]) & 3, (-2, -1)), torch.rot90(ys, int(op[t]) & 3, (-2, -1))
        assert torch.equal(x_d[t].cpu(), xs), (t, int(op[t]))
        assert torch.equal(y_d[t].cpu(), ys), (t, int(op[t]))
    with pytest.raises(_lib.B2UError):          # a window larger than the raster is refused before any launch
        _lib.check(lib.b2u_crop_train_batch(r_d.data_ptr(), code, C, Y, 20, l_d.data_ptr(), _lib.DT_U8,
                                            t_d[0].data_ptr(), t_d[1].data_ptr(), t_d[2].data_ptr(), T, P,
                                            x_d.data_ptr(), y_d.data_ptr(), ops.stream_ptr()))


def _pair(d, name, H, W, seed, kind):
    x, y = aerial_like_tiles(1, 4, H, W, 3, seed=seed)
    img, msk = x[0].numpy(), y[0].numpy()
    if kind == "uint16":
        img = img.astype(np.uint16) * 4 + 3                  # values above 256: the 'int16' dataset kind
    if kind == "regression":
        msk = (img[3].astype(np.float32) - img[0]) / 64.0 + 2.0
    elif kind == "classes2":
        msk = np.minimum(msk, 1)
    write_geotiff(d / f"{name}.tif", img, GEO)
    write_geotiff(d / f"{name}_mask.tif", msk, GEO)
    return str(d / f"{name}.tif"), str(d / f"{name}_mask.tif")


CONFIGS = {
    # scenes, tiling (patch, overlap, split, max_empty, class_zero, seed), training keywords
    "uint8_weighted_aug": ([("scene", 330, 300, 1, "classes2")], (64, 0.25, [0.7, 0.3], 0.9, False, 3),
                           dict(EPOCHS=2, CLASS_WEIGHTS="weighted", transforms=True, n_transform_imgs=0.5, split_idx=4,
                                CODES=("background", "forest"))),
    "uint16": ([("u16", 300, 300, 2, "uint16")], (64, 0.2, [0.6, 0.3, 0.1], 0.9, False, 0),
               dict(EPOCHS=2, CODES=("a", "b", "c"), transforms=True, n_transform_imgs=1.0)),
    "regression": ([("reg", 300, 320, 3, "regression")], (64, 0.25, [0.7, 0.3], 0.9, False, 1),
                   dict(EPOCHS=2, enable_regression=True, CODES=("value",))),
    "two_pairs": ([("b_scene", 260, 300, 4, "classes2"), ("a_scene", 300, 200, 5, "classes2")],
                  (64, 0.25, [0.5, 0.3, 0.2], 0.5, True, 2),
                  dict(EPOCHS=2, transforms=True, n_transform_imgs=0.5, CODES=("nodata", "background", "forest"))),
}


@pytest.mark.parametrize("name", list(CONFIGS))
def test_train_geotiff_matches_split_raster_and_train_func(tmp_path, name):
    scenes, (P, ov, split, max_empty, class_zero, seed), kw = CONFIGS[name]
    src = tmp_path / "src"
    src.mkdir()
    pairs = [_pair(src, n, H, W, s, kind) for n, H, W, s, kind in scenes]
    base = tmp_path / "tiles"
    for r, m in pairs:
        split_raster(r, m, str(base), P, ov, split, max_empty, class_zero, seed)
    B = 8
    kw = dict(kw, ARCHITECTURE="xresnet18", LEARNING_RATE=2e-3)
    a = train_func(base, None, tmp_path / "files", "run", B, False, kw.get("enable_regression", False),
                   kw.get("CLASS_WEIGHTS", "even"), "xresnet18", kw["EPOCHS"], 2e-3, 10, None, None, None, False, "vali",
                   kw["CODES"], kw.get("transforms", False), kw.get("split_idx"), False, None,
                   kw.get("n_transform_imgs", 0), False, class_zero)
    b = train_geotiff(pairs if len(pairs) > 1 else pairs[0], P, ov, split, max_empty, class_zero, seed,
                      model_Path=tmp_path / "raster", description="run", BATCH_SIZE=B, **kw)
    n_valid = sum(1 for _ in (base / "vali" / "img_tiles").glob("*.tif"))
    assert n_valid > 0
    if name == "uint8_weighted_aug":
        assert n_valid % B != 0                                    # a padded last validation batch
        assert a.class_weights != [0.5, 0.5] and a.class_weights == b.class_weights
    if name == "uint16":
        assert a.sixteen_bit and b.sixteen_bit
    sa, sb = a.state_dict(), b.state_dict()
    assert sa.keys() == sb.keys()
    for k in sa:
        assert torch.equal(sa[k], sb[k]), k
    strip = lambda h: [{k: v for k, v in r.items() if k != "time"} for r in h]
    assert strip(a.history) == strip(b.history)
    assert all(math.isfinite(r["valid_loss"]) for r in a.history)
    pa = torch.load(tmp_path / "files" / "run" / "run.pkl", map_location="cpu", weights_only=True)
    pb = torch.load(tmp_path / "raster" / "run" / "run.pkl", map_location="cpu", weights_only=True)
    assert {k: v for k, v in pa.items() if k != "state_dict"} == {k: v for k, v in pb.items() if k != "state_dict"}
    assert all(torch.equal(pa["state_dict"][k], pb["state_dict"][k]) for k in pa["state_dict"])
    if name == "uint8_weighted_aug":
        again = load_learner(tmp_path / "raster" / "run" / "run.pkl")
        tile = torch.from_numpy(np.ascontiguousarray(_read_first_tile(base)))
        _, a1, p1 = again.predict(tile)
        _, a2, p2 = b.predict(tile)
        assert torch.equal(a1, a2) and torch.equal(p1, p2)


def _read_first_tile(base):
    from unet_b200.geotiff import read_geotiff
    return read_geotiff(sorted((base / "vali" / "img_tiles").glob("*.tif"))[0])[0]
