"""Tile creation for training / prediction: the host-side caller in front of the hot path.

Mirrors `create_tiles_unet.py` of the reference: `compute_windows` (:30-56, slidingwindow 0.0.14 semantics, bit-exact in
`unet_b200/tiling.py`), `split_raster` (:252-431: windows, empty-tile filter :414/:422, georeferenced tile files
:179-249) and `create_train_test_split` (:70-176).  Files are GeoTIFFs written by `unet_b200/geotiff.py`.

Deliberately NOT replicated (SURVEY.md 8(b) portability hazards / out-of-scope rows): the raster-vs-mask re-alignment
of grids that do not coincide (:287-352 - a ValueError here), hard-coded `\\` separators, `Create(path, rows, cols)`
argument order, the y origin computed with the x pixel size (:226) and the unseeded `np.random.shuffle` of the split
(seeded here so that a data set can be re-created).
"""
from __future__ import annotations

import os
import warnings
from pathlib import Path
from typing import Dict, List, NamedTuple, Optional, Sequence, Tuple

import numpy as np

from .geotiff import GeoInfo, read_geotiff, write_geotiff
from .tiling import Window, compute_windows as _windows_hw


def compute_windows(numpy_image: np.ndarray, patch_size: int, patch_overlap: float) -> List[Window]:
    """create_tiles_unet.py:30-56: windows (x, y, w, h) over an image array `[H, W, bands]`, x-outer / y-inner."""
    if patch_overlap > 1:
        raise ValueError(f"Patch overlap {patch_overlap} must be between 0 - 1")     # create_tiles_unet.py:47-48
    return _windows_hw(int(numpy_image.shape[0]), int(numpy_image.shape[1]), patch_size, patch_overlap)


def _keep(crop: np.ndarray, max_empty: float) -> bool:
    """create_tiles_unet.py:412-415: drop empty crops and crops with fewer than (1 - max_empty) non-zero samples."""
    return crop.size != 0 and not (np.sum(crop != 0) < np.prod(crop.shape) * (1 - max_empty))


def split_names(names: Sequence[str], split: Optional[Sequence[float]] = None, seed: int = 0) -> Dict[str, List[str]]:
    """The subset decision of create_tiles_unet.py:70-176: tile names -> {"trai": [...], "vali": [...] (, "test": [...])}
    by a seeded shuffle of the sorted names; a third subset only when the third ratio is non-zero."""
    if split is None:
        split = [0.7, 0.2, 0.1]
    if np.round(np.sum(split), decimals=3) != 1.0:
        split = [0.7, 0.2, 0.1]
        warnings.warn("Train/Vali/Test-Split percentage does not sum to 1, reseting to 70%/20%/10%.")
    files = sorted(names)
    np.random.default_rng(seed).shuffle(files)
    n = len(files)
    three = len(split) == 3 and split[-1] != 0
    a = int(n * split[0])
    b = int(n * np.sum(split[:2])) if three else n
    parts = {"trai": files[:a], "vali": files[a:b]}
    if three:
        parts["test"] = files[b:]
    return parts


def create_train_test_split(path, split: Optional[Sequence[float]] = None, seed: int = 0) -> dict:
    """create_tiles_unet.py:70-176: moves `path/img_tiles/*.tif` + `path/mask_tiles/*.tif` into `trai/`, `vali/` (and
    `test/` when the third ratio is non-zero) as `split_names` decides; returns the file names per subset."""
    src = Path(path)
    parts = split_names([p.name for p in (src / "img_tiles").glob("*.tif")], split, seed)
    for name, fs in parts.items():
        for sub in ("img_tiles", "mask_tiles"):
            (src / name / sub).mkdir(parents=True, exist_ok=True)
            for f in fs:
                if (src / sub / f).exists():
                    os.replace(src / sub / f, src / name / sub / f)
    for sub in ("img_tiles", "mask_tiles"):
        try:
            (src / sub).rmdir()
        except OSError:
            pass
    return parts


class PreparedRaster(NamedTuple):
    """What `split_raster` cuts its tiles from: the raster `[C, H, W]` and its mask `[bands, H, W]` (None without one)
    after the class_zero shift and the no-data zeroing, and the kept tiles as (file name, window (x, y, w, h))."""
    image: np.ndarray
    mask: Optional[np.ndarray]
    geo: GeoInfo
    tiles: List[Tuple[str, Window]]


def prepare_raster(path_to_raster, path_to_mask=None, patch_size: int = 400, patch_overlap: float = 0.20,
                   max_empty: float = 0.9, class_zero: bool = False) -> PreparedRaster:
    """The decisions of create_tiles_unet.py:252-431 before any file is written: class_zero shift of the mask, no-data
    pixels of image and mask zeroed in both, the grid check, the windows, the empty-tile filter (:414/:422) and the
    tile names `<raster stem>_<window index>.tif`."""
    if path_to_raster is None:
        raise ValueError("path_to_raster is required")
    image, geo = read_geotiff(path_to_raster)
    include_mask = path_to_mask is not None
    nodata = geo.nodata
    mask = None
    if include_mask:
        mask, mgeo = read_geotiff(path_to_mask)
        check_same_grid(geo, mgeo, image.shape[1:], mask.shape[1:])
        mask, bad = mask_labels(image, nodata, mask, mgeo.nodata, class_zero)
        image = image.copy()
        image[:, bad] = 0
    elif nodata is not None:
        image = image.copy()
        image[:, (image == nodata).any(axis=0)] = 0
    img_hwc = np.moveaxis(image, 0, 2)
    H, W = img_hwc.shape[:2]
    if H < patch_size or W < patch_size:
        raise ValueError("Patch size of {} is larger than the image dimensions {}".format(patch_size, [H, W]))   # :398-400
    windows = compute_windows(img_hwc, patch_size, patch_overlap)
    stem = os.path.splitext(os.path.basename(str(path_to_raster)))[0]
    tiles = []
    for index, (x, y, w, h) in enumerate(windows):
        if not _keep(image[:, y:y + h, x:x + w], max_empty):
            continue
        if include_mask and not _keep(mask[:1, y:y + h, x:x + w], max_empty):
            continue
        tiles.append((f"{stem}_{index}.tif", (x, y, w, h)))
    return PreparedRaster(image, mask, geo, tiles)


def check_same_grid(geo: GeoInfo, mgeo: GeoInfo, image_hw, mask_hw) -> None:
    """The grid check of create_tiles_unet.py:287-352: the mask must share the raster's origin (to 3 decimals) and its
    height and width; re-aligning them is refused with a ValueError."""
    same_grid = (np.round(geo.geotransform[0], 3) == np.round(mgeo.geotransform[0], 3)
                 and np.round(geo.geotransform[3], 3) == np.round(mgeo.geotransform[3], 3)
                 and tuple(image_hw) == tuple(mask_hw))
    if not same_grid:
        raise ValueError("image and mask grids differ; re-aligning them (create_tiles_unet.py:287-352) is outside "
                         "the built path - resample the mask onto the image grid first")


def mask_labels(image: np.ndarray, nodata, mask: np.ndarray, mask_nodata, class_zero: bool):
    """The label conversion of create_tiles_unet.py:282-283, 366-369 on a raster `[C, H, W]` and its mask `[bands, H, W]`
    (whole or the same window of both): with `class_zero` every label that is not the mask's no-data value is shifted
    by one, then pixels that are no-data in the image or in the mask are zeroed.  Returns (the converted mask, a copy;
    the no-data pixels [H, W], which `prepare_raster` also zeroes in the image)."""
    mask = mask.copy()
    if class_zero:                                                       # :282-283 shift labels, keep no-data
        sel = np.ones(mask.shape, bool) if mask_nodata is None else mask != mask_nodata
        mask[sel] += 1
    bad = np.zeros(image.shape[1:], bool)                                 # :366-369
    if nodata is not None:
        bad |= (image == nodata).any(axis=0)
    if mask_nodata is not None:
        bad |= (mask == mask_nodata).any(axis=0)
    mask[:, bad] = 0
    return mask, bad


def split_raster(path_to_raster=None, path_to_mask=None, base_dir=".", patch_size: int = 400, patch_overlap: float = 0.20,
                 split: Optional[Sequence[float]] = None, max_empty: float = 0.9, class_zero: bool = False,
                 seed: int = 0) -> List[Path]:
    """create_tiles_unet.py:252-431 with the reference's argument order.  Cuts the raster (and its mask) into
    `patch_size` windows with `patch_overlap`, zeroes no-data pixels in both, drops tiles that are more than `max_empty`
    zeros, writes `<base_dir>/img_tiles/<raster>_<index>.tif` (+ `mask_tiles/`) with the window's georeferencing and -
    when a mask is given - distributes them into trai / vali / test.  Returns the image-tile paths written."""
    prep = prepare_raster(path_to_raster, path_to_mask, patch_size, patch_overlap, max_empty, class_zero)
    image, mask, geo = prep.image, prep.mask, prep.geo
    include_mask = mask is not None
    base = Path(base_dir)
    (base / "img_tiles").mkdir(parents=True, exist_ok=True)
    if include_mask:
        (base / "mask_tiles").mkdir(parents=True, exist_ok=True)
    written = []
    for name, (x, y, w, h) in prep.tiles:
        g = geo.window(x, y)
        g = GeoInfo(g.geotransform, g.geokeys, g.geodoubles, g.geoascii, None, g.georeferenced)
        write_geotiff(base / "img_tiles" / name, image[:, y:y + h, x:x + w], g)
        if include_mask:
            write_geotiff(base / "mask_tiles" / name, mask_tile_values(mask[:1, y:y + h, x:x + w]), g)
        written.append(base / "img_tiles" / name)
    if include_mask:
        parts = create_train_test_split(base, split=split, seed=seed)
        where = {f: k for k, fs in parts.items() for f in fs}
        written = [base / where[p.name] / "img_tiles" / p.name for p in written]
    return written


def mask_tile_values(mask: np.ndarray) -> np.ndarray:
    """The values a mask tile is stored with (:236-241): a floating-point mask keeps its type, any other becomes Byte."""
    return mask if mask.dtype.kind == "f" else mask.astype(np.uint8)
