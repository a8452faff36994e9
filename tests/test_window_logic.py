"""Host logic of windowed reads (no GPU): which frames a pixel window needs, their byte ranges, and the bbox -> pixel
window rounding."""
import io
import math

import numpy as np
import pytest

from flac_raster_b200 import _native as nat, flacfmt
from flac_raster_b200.engine import bbox_to_window, tile_grid, window_frames


def brute_force_runs(tiles, window, blocksize):
    """Every sample of every tile, kept when its pixel lies inside the window: (tile, first frame, frame count)."""
    c0, r0, ww, wh = window
    out = []
    for i, t in enumerate(tiles):
        r, c, h, w = int(t["row_off"]), int(t["col_off"]), int(t["h"]), int(t["w"])
        s = np.arange(h * w, dtype=np.int64)
        y, x = r + s // w, c + s % w
        inside = (y >= r0) & (y < r0 + wh) & (x >= c0) & (x < c0 + ww)
        if inside.any():
            f = s[inside] // blocksize
            out.append((i, int(f.min()), int(f.max() - f.min() + 1)))
    return out


def geometries(seed=0):
    rng = np.random.default_rng(seed)
    for H, W, ts in ((37, 53, 16), (100, 9, 32), (64, 64, 64), (130, 97, 40), (5, 300, 7), (300, 5, 64)):
        tiles = tile_grid(H, W, ts)                  # ragged edge tiles where ts does not divide the raster
        wins = [(0, 0, W, H), (0, 0, 1, 1), (W - 1, H - 1, 1, 1), (0, H - 1, W, 1), (W - 1, 0, 1, H),
                (0, 0, 1, H), (0, 0, W, 1), (W // 2, H // 2, 1, 1)]
        for _ in range(12):
            c0, r0 = int(rng.integers(0, W)), int(rng.integers(0, H))
            wins.append((c0, r0, int(rng.integers(1, W - c0 + 1)), int(rng.integers(1, H - r0 + 1))))
        for win in wins:
            yield tiles, win


@pytest.mark.parametrize("blocksize", [4096, 1152, 16, 100])
def test_window_frames_equal_brute_force(blocksize):
    n = 0
    for tiles, win in geometries():
        runs = window_frames(tiles, win, blocksize)
        got = [(int(r["tile"]), int(r["first_frame"]), int(r["n_frames"])) for r in runs]
        assert got == brute_force_runs(tiles, win, blocksize), (win, blocksize)
        assert (runs["byte_offset"] == -1).all() and (runs["byte_length"] == -1).all()
        n += 1
    assert n > 100


def test_window_frames_whole_raster_and_a_single_tile():
    tiles = tile_grid(10980, 10980, 1024)
    runs = window_frames(tiles, (0, 0, 10980, 10980), 4096)
    assert len(runs) == len(tiles) and (runs["first_frame"] == 0).all()
    assert (runs["n_frames"] == (tiles["h"].astype(np.int64) * tiles["w"] + 4095) // 4096).all()
    # a 256-row window inside one tile-1024 tile needs at most 65 of its 256 frames (the figure in DESIGN.md)
    runs = window_frames(tiles, (2048 + 100, 1024 + 300, 512, 256), 4096)
    assert len(runs) == 1 and int(runs[0]["n_frames"]) <= 65
    # one C3-sized file: a 512-row window needs at most 1 374 of the 29 434 frames, whatever its width
    one = tile_grid(10980, 10980, 10980)
    for c0, w in ((0, 10980), (5000, 1), (123, 4000)):
        r = window_frames(one, (c0, 7777, w, 512), 4096)
        assert int(r[0]["n_frames"]) <= 1374


def test_window_frames_byte_ranges_from_a_synthetic_index():
    rng = np.random.default_rng(3)
    tiles = tile_grid(70, 45, 20)
    bs = 64
    fpt = (tiles["h"].astype(np.int64) * tiles["w"] + bs - 1) // bs
    sizes = [rng.integers(20, 900, size=int(n)).astype(np.uint32) for n in fpt]
    for _, win in geometries(5):
        win = (min(win[0], 44), min(win[1], 69), 1 + win[2] % 20, 1 + win[3] % 30)
        win = (win[0], win[1], min(win[2], 45 - win[0]), min(win[3], 70 - win[1]))
        runs = window_frames(tiles, win, bs, sizes)
        for r in runs:
            fb = sizes[int(r["tile"])].astype(np.int64)
            f0, n = int(r["first_frame"]), int(r["n_frames"])
            assert int(r["byte_offset"]) == int(fb[:f0].sum())
            assert int(r["byte_length"]) == int(fb[f0:f0 + n].sum())
            # the run's bytes end where the next frame starts (prefix sum)
            assert int(r["byte_offset"] + r["byte_length"]) == int(np.cumsum(fb)[f0 + n - 1])


def test_window_frames_skip_tiles_outside_the_window():
    tiles = tile_grid(100, 100, 25)
    runs = window_frames(tiles, (30, 30, 10, 10), 4096)
    assert [int(r["tile"]) for r in runs] == [5]
    runs = window_frames(tiles, (20, 20, 10, 10), 4096)       # crosses the corner of four tiles
    assert [int(r["tile"]) for r in runs] == [0, 1, 4, 5]


def test_bbox_to_window_rounding():
    tr = (10.0, 0.0, 500000.0, 0.0, -10.0, 4000000.0)           # 10 m pixels, north-up
    W, H = 1000, 800
    # exact pixel edges give the exact window
    assert bbox_to_window(tr, W, H, (500000 + 100, 4000000 - 300, 500000 + 250, 4000000 - 100)) == (10, 10, 15, 20)
    # partial pixels: near edges floored, far edges ceiled
    assert bbox_to_window(tr, W, H, (500000 + 101, 4000000 - 299, 500000 + 249, 4000000 - 101)) == (10, 10, 15, 20)
    assert bbox_to_window(tr, W, H, (500000 + 109.9, 4000000 - 290.1, 500000 + 240.1, 4000000 - 109.9)) == (10, 10, 15, 20)
    # a bbox inside one pixel is that pixel
    assert bbox_to_window(tr, W, H, (500000 + 3, 4000000 - 7, 500000 + 4, 4000000 - 6)) == (0, 0, 1, 1)
    # clipped to the raster
    assert bbox_to_window(tr, W, H, (499000, 3000000, 600000, 4100000)) == (0, 0, W, H)
    assert bbox_to_window(tr, W, H, (500000 + 9995, 4000000 - 7995, 600000, 3000000)) == (999, 799, 1, 1)
    # pixel-space transform of files without georeferencing (y grows downwards as -row)
    assert bbox_to_window((1.0, 0.0, 0.0, 0.0, -1.0, 0.0), 50, 40, (2.5, -7.5, 4.5, -3.5)) == (2, 3, 3, 5)
    # an empty intersection raises
    for bb in ((0, 0, 1, 1), (500000 + 10000, 4000000 - 10, 500000 + 10010, 4000000), (500000 - 20, 4000000 - 10, 500000, 4000000)):
        with pytest.raises(ValueError):
            bbox_to_window(tr, W, H, bb)
    with pytest.raises(ValueError):
        bbox_to_window((10.0, 0.5, 0.0, 0.0, -10.0, 0.0), W, H, (0, -10, 10, 0))


def test_read_header_reads_only_the_metadata_chain():
    si = flacfmt.StreamInfo(4096, 4096, 0, 0, 44100, 3, 16, 123456)
    fb = np.arange(1, 31, dtype=np.uint32) * 100
    sidx = flacfmt.pack_seek_index(3, 4096, fb, np.arange(90, dtype=np.uint32))
    frames = b"\xff\xf8" + bytes(200000)
    for padding in (0, 1024):
        blob = flacfmt.build_header(si, {"GEOSPATIAL_CRS": "EPSG:4326", "X": "y" * 70000}, padding=padding, seek_index=sidx) + frames
        want = flacfmt.parse_header(blob)
        reads = []

        def read(start, n):
            reads.append((start, n))
            return blob[start:start + n]

        got = flacfmt.read_header(read, first=4096)
        assert got.first_frame_offset == want.first_frame_offset
        assert got.tags == want.tags and got.applications == want.applications and got.streaminfo == want.streaminfo
        hi = max(s + n for s, n in reads)
        # nothing behind the chain is read, and a trailing PADDING body is skipped
        assert hi <= want.first_frame_offset - (padding if padding else 0)
