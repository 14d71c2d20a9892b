"""Tile index arithmetic of the reference (integer, bit-exact) and the scheduling helpers of tiled prediction.

`compute_windows` reproduces what the reference obtains from `slidingwindow.generate(img, HeightWidthChannel,
patch_size, patch_overlap)` (create_tiles_unet.py:30-56, slidingwindow 0.0.14 generateForSize): window side
min(patch, dim), overlap floor(side*overlap) pixels, step side-overlap, offsets range(0, last+1, step) plus the last
offset, enumerated x-outer / y-inner — the tile number in the reference's file names (create_tiles_unet.py:408-431).
"""
from __future__ import annotations

import math
from typing import List, Sequence, Tuple

Window = Tuple[int, int, int, int]  # (x, y, w, h) == slidingwindow's getRect()


def axis_offsets(dim: int, patch_size: int, patch_overlap: float) -> Tuple[List[int], int]:
    win = min(patch_size, dim)
    step = win - int(math.floor(win * patch_overlap))
    last = dim - win
    if step <= 0:
        raise ValueError("patch_overlap leaves no positive step")
    offs = list(range(0, last + 1, step))
    if not offs or offs[-1] != last:
        offs.append(last)
    return offs, win


def compute_windows(height: int, width: int, patch_size: int, patch_overlap: float) -> List[Window]:
    if patch_overlap > 1:
        raise ValueError(f"Patch overlap {patch_overlap} must be between 0 - 1")  # create_tiles_unet.py:48-49
    xs, ww = axis_offsets(width, patch_size, patch_overlap)
    ys, wh = axis_offsets(height, patch_size, patch_overlap)
    return [(x, y, ww, wh) for x in xs for y in ys]


def tile_origin_geo(gt: Sequence[float], x: int, y: int) -> Tuple[float, float]:
    """geo origin the reference writes into a tile (create_tiles_unet.py:224-226; it uses the x pixel size for y too)"""
    return x * gt[1] + gt[0], gt[3] - y * gt[1]


def placement_from_geotransform(ulx: float, xsize: int, xres: float, uly: float, ysize: int, yres: float,
                                upleft_x_full: float, upleft_y_full: float) -> Tuple[int, int, int, int]:
    """pixel placement of a tile in the merged raster exactly as predict.py:294-297 computes it (python round())."""
    x0 = round((ulx - upleft_x_full) / xres)
    y0 = round((uly - upleft_y_full) / yres)
    x1 = round((ulx + xsize * xres - upleft_x_full) / xres)
    y1 = round((uly + ysize * yres - upleft_y_full) / yres)
    return x0, y0, x1, y1


def _axis_colours(offsets: Sequence[int], win: int) -> Tuple[List[int], int]:
    """greedy interval colouring: tiles of one colour never overlap along this axis"""
    order = sorted(range(len(offsets)), key=lambda i: offsets[i])
    end_of_colour: List[int] = []
    colour = [0] * len(offsets)
    for i in order:
        o = offsets[i]
        for c, e in enumerate(end_of_colour):
            if e <= o:
                colour[i] = c
                end_of_colour[c] = o + win
                break
        else:
            colour[i] = len(end_of_colour)
            end_of_colour.append(o + win)
    return colour, len(end_of_colour)


def colour_classes(windows: Sequence[Window]) -> List[List[int]]:
    """Partition tile indices into classes of mutually non-overlapping tiles (product of per-axis interval colourings).
    Stitch launches handle one class at a time, so overlap sums never race and never depend on scheduling."""
    if not windows:
        return []
    xs = sorted({w[0] for w in windows})
    ys = sorted({w[1] for w in windows})
    ww, wh = windows[0][2], windows[0][3]
    cx, nx = _axis_colours(xs, ww)
    cy, ny = _axis_colours(ys, wh)
    mx = {x: c for x, c in zip(xs, cx)}
    my = {y: c for y, c in zip(ys, cy)}
    classes: List[List[int]] = [[] for _ in range(nx * ny)]
    for i, (x, y, _, _) in enumerate(windows):
        classes[my[y] * nx + mx[x]].append(i)
    return [c for c in classes if c]


def split_range(n: int, parts: int, k: int) -> Tuple[int, int]:
    """[begin, end) of part k of the balanced partition of range(n) into `parts` contiguous parts: the first n % parts
    parts take one more.  Every sharding of the output and every gather of the shards uses this one partition."""
    base, rem = divmod(n, parts)
    b = k * base + min(k, rem)
    return b, b + base + (1 if k < rem else 0)


def shard_windows_by_columns(windows: Sequence[Window], width: int, rank: int, world: int):
    """Owner-computes sharding for multi-GPU prediction (SURVEY 8(e)): rank r owns output columns [X_r, X_{r+1}) and
    runs every tile that intersects them, so sum / count / argmax of its strip are local and bit-identical to a
    single-GPU run.  Returns (tile indices, x_begin, x_end)."""
    xb, xe = split_range(width, world, rank)
    idx = [i for i, (x, y, w, h) in enumerate(windows) if x < xe and x + w > xb]
    return idx, xb, xe


def column_owned(windows: Sequence[Window], idx: Sequence[int], xb: int, xe: int) -> List[bool]:
    """Per tile of `idx`: whether its left edge column lies in [xb, xe).  Over the strips of `shard_windows_by_columns`
    every tile has exactly one owner, so work done once per tile (counting it in an assessment) is done by one rank."""
    return [xb <= windows[i][0] < xe for i in idx]


def shard_grid(windows: Sequence[Window], width: int, height: int, world: int) -> Tuple[int, int]:
    """(gx, gy) with gx * gy == world that minimises the largest number of tiles any rank has to run when every rank
    owns one cell of a gx x gy grid of the output (tiles straddling a cell border run on both sides).  Column strips
    (gy == 1) duplicate one tile column per border: 7 of 97 on the 20000^2 raster at 8 ranks, 13 x 90 = 1170 tiles on
    the fullest rank against 1012.5 ideal; a 4 x 2 grid needs 24 x 46 = 1104."""
    best = None
    for gx in range(1, world + 1):
        if world % gx:
            continue
        gy = world // gx
        worst = 0
        for r in range(world):
            xb, xe = split_range(width, gx, r % gx)
            yb, ye = split_range(height, gy, r // gx)
            worst = max(worst, sum(1 for (x, y, w, h) in windows if x < xe and x + w > xb and y < ye and y + h > yb))
        key = (worst, gy)              # ties: fewer row cuts (strips keep whole raster rows contiguous)
        if best is None or key < best[0]:
            best = (key, (gx, gy))
    return best[1]


def shard_windows_2d(windows: Sequence[Window], width: int, height: int, rank: int, world: int,
                     grid: Tuple[int, int] = None):
    """Owner-computes sharding over a gx x gy grid of output cells: rank r owns cell (r % gx, r // gx) and runs every
    tile that intersects it - sums, counts and argmax of the cell are local, exactly as with column strips.
    Returns (tile indices, (x_begin, x_end, y_begin, y_end))."""
    gx, gy = grid or shard_grid(windows, width, height, world)
    xb, xe = split_range(width, gx, rank % gx)
    yb, ye = split_range(height, gy, rank // gx)
    idx = [i for i, (x, y, w, h) in enumerate(windows) if x < xe and x + w > xb and y < ye and y + h > yb]
    return idx, (xb, xe, yb, ye)
