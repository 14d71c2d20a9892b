"""Tile-free training input (`train_geotiff`) against the file path it replaces, on the host: the windows and splits
against the files `split_raster` writes and `train_func` lists, the batch plan (dealing, padding, augmentation draws)
through a numpy restatement of `b2u_crop_train_batch` against `augmented(_tile_batches(files))`, and the rejections."""
import numpy as np
import pytest
import torch

from unet_b200.create_tiles import split_raster
from unet_b200.geotiff import GeoInfo, read_geotiff, write_geotiff
from unet_b200.reference_api import (_BatchDeal, _epoch_table, _raster_windows, _tile_batches, augmented,
                                     train_geotiff)

GEO = GeoInfo(geotransform=(383000.0, 0.2, 0.0, 5819000.0, 0.0, -0.2),
              geokeys=(1, 1, 0, 3, 1024, 0, 1, 1, 1025, 0, 1, 1, 3072, 0, 1, 25833), georeferenced=True)
P = 64


def _scene(d, name, H, W, seed, n_classes=3):
    """a 4-band uint8 raster with no-data 7 in a corner, empty columns (dropped by max_empty) and a mask with no-data 9"""
    rng = np.random.default_rng(seed)
    img = rng.integers(10, 256, size=(4, H, W), dtype=np.uint8)
    img[:, :, :70] = 0
    img[:, :20, -30:] = 7
    msk = rng.integers(0, n_classes, size=(H, W), dtype=np.uint8)
    msk[-25:, 100:140] = 9
    write_geotiff(d / f"{name}.tif", img, GEO, nodata=7)
    write_geotiff(d / f"{name}_mask.tif", msk, GEO, nodata=9)
    return str(d / f"{name}.tif"), str(d / f"{name}_mask.tif")


def _train_func_files(base, valid_scenes=("vali",)):
    """the tile files train_func lists, in its order"""
    train, valid = [], []
    for scene in sorted(p for p in base.iterdir() if p.is_dir()):
        (valid if scene.name in valid_scenes else train).extend(sorted((scene / "img_tiles").glob("*.tif")))
    return train, valid


CASES = [  # (scenes (name, H, W), split, max_empty, class_zero)
    ([("r", 300, 260)], [0.6, 0.4], 0.5, True),
    ([("r", 300, 260)], [0.5, 0.3, 0.2], 0.9, False),
    ([("b", 250, 300), ("a", 300, 200)], [0.5, 0.3, 0.2], 0.5, False),
    ([("b", 250, 300), ("a", 300, 200)], [0.7, 0.3], 0.2, True),
]


def _dataset(tmp_path, scenes, split, max_empty, class_zero):
    src = tmp_path / "src"
    src.mkdir(exist_ok=True)
    pairs = [_scene(src, n, H, W, 11 + i) for i, (n, H, W) in enumerate(scenes)]
    base = tmp_path / "tiles"
    for r, m in pairs:
        split_raster(r, m, str(base), P, 0.25, split, max_empty, class_zero, 5)
    return pairs, base


@pytest.mark.parametrize("scenes,split,max_empty,class_zero", CASES)
def test_windows_name_the_files_split_raster_writes(tmp_path, scenes, split, max_empty, class_zero):
    pairs, base = _dataset(tmp_path, scenes, split, max_empty, class_zero)
    images, labels, train, valid = _raster_windows(pairs if len(pairs) > 1 else pairs[0], P, 0.25, split, max_empty,
                                                   class_zero, 5, ("vali",))
    f_train, f_valid = _train_func_files(base)
    assert [e[0] for e in train] == [f.name for f in f_train]
    assert [e[0] for e in valid] == [f.name for f in f_valid]
    assert len(train) > 10 and valid
    if len(split) == 3:
        assert (base / "test").is_dir()       # `test` trains, as train_func reads it
    for e, f in zip(train + valid, f_train + f_valid):
        name, k, (x, y, w, h) = e
        assert (w, h) == (P, P)
        assert np.array_equal(read_geotiff(f)[0], images[k][:, y:y + h, x:x + w]), name
        m = read_geotiff(str(f).replace("img_tiles", "mask_tiles"))[0][0]
        assert m.dtype == labels[k].dtype and np.array_equal(m, labels[k][y:y + h, x:x + w]), name


def _crop_np(img, lab, table_k, n):
    """numpy restatement of b2u_crop_train_batch for one batch"""
    xs, ys = [], []
    for i in range(n):
        y0, x0, op = (int(v) for v in table_k[:, i])
        a, b = img[:, y0:y0 + P, x0:x0 + P], lab[y0:y0 + P, x0:x0 + P]
        if op & 4:
            a, b = a[..., ::-1], b[..., ::-1]
        xs.append(np.rot90(a, op & 3, axes=(-2, -1)))
        ys.append(np.rot90(b, op & 3, axes=(-2, -1)))
    return np.stack(xs), np.stack(ys)


@pytest.mark.parametrize("world", [1, 2])
@pytest.mark.parametrize("B", [5, 16])
def test_batch_plan_matches_augmented_tile_batches(tmp_path, world, B):
    scenes, split, max_empty, class_zero = CASES[2]
    pairs, base = _dataset(tmp_path, scenes, split, max_empty, class_zero)
    images, labels, train, valid = _raster_windows(pairs, P, 0.25, split, max_empty, class_zero, 5, "vali")
    f_train, f_valid = _train_func_files(base)
    # the device layout: pairs stacked along y, zero-padded to the widest
    yoff = np.cumsum([0] + [a.shape[1] for a in images])
    img = np.zeros((4, yoff[-1], max(a.shape[2] for a in images)), np.uint8)
    lab = np.zeros(img.shape[1:], np.uint8)
    for k, (a, m) in enumerate(zip(images, labels)):
        img[:, yoff[k]:yoff[k + 1], :a.shape[2]] = a
        lab[yoff[k]:yoff[k + 1], :m.shape[1]] = m
    yx = lambda es: np.array([(yoff[e[1]] + e[2][1], e[2][0]) for e in es], np.int32)
    n_padded = 0
    for rank in range(world):
        drop_last = len(train) >= B * world
        sources = [  # (file batches, deal, window origins, share, augmentation seed)
            (augmented(_tile_batches(f_train, B, 3, False, 0, drop_last, False, rank, world), 0.5, seed=3),
             _BatchDeal(len(train), B, 0, drop_last, rank, world), yx(train), 0.5, 3),
            (_tile_batches(f_valid, B, 3, False, None, False), _BatchDeal(len(valid), B, None, False), yx(valid), None, 0),
        ]
        for files, deal, origins, share, seed in sources:
            assert files.n_batches == deal.n_batches
            ops_seen = set()
            for epoch in range(3):
                table, n_real = _epoch_table(deal, epoch, origins, share, seed)
                got = list(files())
                assert len(got) == len(n_real) == deal.n_batches
                for k, (xf, yf, nf) in enumerate(got):
                    assert nf == n_real[k]
                    n_padded += int(nf < B)
                    xc, yc = _crop_np(img, lab, table[k], B)
                    assert np.array_equal(xf.numpy(), xc) and np.array_equal(yf.numpy(), yc), (rank, epoch, k)
                    ops_seen |= set(table[k, 2].tolist())
            if share is not None:
                assert len(ops_seen) > 4
    assert n_padded > 0


def test_rejections(tmp_path):
    (tmp_path / "a").mkdir()
    (tmp_path / "b").mkdir()
    p1 = _scene(tmp_path / "a", "r", 200, 200, 1)
    p2 = _scene(tmp_path / "b", "r", 200, 200, 2)
    kw = dict(model_Path=tmp_path / "m", description="d", BATCH_SIZE=4)
    with pytest.raises(ValueError, match="collide"):
        train_geotiff([p1, p2], P, 0.25, [0.7, 0.3], **kw)
    with pytest.raises(ValueError, match="number of classes"):            # labels 0..2 with two classes
        train_geotiff(p1, P, 0.25, [0.7, 0.3], CODES=("a", "b"), **kw)
    with pytest.raises(ValueError, match="n_transform_imgs"):
        train_geotiff(p1, P, 0.25, [0.7, 0.3], CODES=("a", "b", "c"), transforms=True, n_transform_imgs=1.5, **kw)
    assert not (tmp_path / "m").exists()


def test_augmented_permutes_uint16_tiles_as_int16():
    """`augmented` on uint16 tiles (torch has no CPU flip / rot90 for uint16) gives the bits it gives on int16 tiles"""
    rng = np.random.default_rng(0)
    x = torch.from_numpy(rng.integers(0, 65536, size=(6, 3, 16, 16), dtype=np.uint16))
    y = torch.from_numpy(rng.integers(0, 3, size=(6, 16, 16), dtype=np.uint8))
    src = lambda xx: (lambda: [(xx, y, 6)])
    (xu, yu, _), = augmented(src(x), 1.0, seed=2)()
    (xi, yi, _), = augmented(src(x.view(torch.int16)), 1.0, seed=2)()
    assert xu.dtype == torch.uint16 and torch.equal(xu.view(torch.int16), xi) and torch.equal(yu, yi)
    assert not torch.equal(xi, x.view(torch.int16))
