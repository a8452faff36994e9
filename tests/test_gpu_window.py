"""Windowed reads on the GPU: RasterFLACConverter.read_window and SpatialFLACStreamer.read_bbox against whole decodes."""
import numpy as np
import pytest

from conftest import GOLDEN
from flac_raster_b200 import flacfmt

pytestmark = pytest.mark.gpu

DTYPES = ["uint8", "int8", "uint16", "int16", "uint32", "int32", "float32", "float64"]


def _raster(dtype, bands, H, W, seed):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:H, 0:W]
    base = np.sin(xx / 13.0) * np.cos(yy / 7.0)
    planes = []
    for b in range(bands):
        v = base + 0.05 * b + 0.02 * rng.standard_normal((H, W))     # correlated bands: two-band frames go mid/side
        planes.append(v)
    v = np.stack(planes)
    dt = np.dtype(dtype)
    if np.issubdtype(dt, np.integer):
        info = np.iinfo(dt)
        lo, hi = max(info.min, -30000), min(info.max, 60000)
        return np.clip(np.round((v + 1.2) / 2.4 * (hi - lo) + lo), info.min, info.max).astype(dt)
    return (v * 1000.0).astype(dt)


def _windows(H, W, blocksize, seed):
    """1x1, full raster, edges, widths that are not multiples of 8, odd column offsets, starts and ends inside frames."""
    rng = np.random.default_rng(seed)
    wins = [(0, 0, W, H), (0, 0, 1, 1), (W - 1, H - 1, 1, 1), (3, 5, 13, 7), (1, 0, W - 1, 2), (W - 7, 1, 7, H - 1)]
    s0 = blocksize + 5                                            # starts inside frame 1, ends inside frame 2
    wins.append((s0 % W, s0 // W, min(W - s0 % W, 29), 3))
    for _ in range(4):
        c0 = int(rng.integers(0, (W - 1) // 2)) * 2 + 1           # odd
        r0 = int(rng.integers(0, H - 1))
        w = int(rng.integers(1, W - c0 + 1))
        if w % 8 == 0:
            w -= 1
        wins.append((c0, r0, max(w, 1), int(rng.integers(1, H - r0 + 1))))
    return wins


def _strip_index(blob: bytes) -> bytes:
    h = flacfmt.parse_header(blob)
    tags = {k: v[0] for k, v in h.tags.items()}
    return flacfmt.build_header(h.streaminfo, tags, vendor=h.vendor, padding=64) + blob[h.first_frame_offset:]


def _eq(a, b):
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a, b, equal_nan=a.dtype.kind == "f")


@pytest.mark.parametrize("bands", [1, 2, 3, 8])
@pytest.mark.parametrize("dtype", DTYPES)
def test_read_window_equals_whole_decode_cropped(tmp_path, dtype, bands):
    from flac_raster_b200.converter import RasterFLACConverter
    from flac_raster_b200.engine import tile_grid, window_frames

    H, W = 97, 211                                               # 20 467 samples: 5 frames of 4096, the last one short
    conv = RasterFLACConverter()
    data = _raster(dtype, bands, H, W, seed=bands * 17 + DTYPES.index(dtype))
    path = tmp_path / "r.flac"
    conv.array_to_flac(data, path, transform=(10.0, 0.0, 1000.0, 0.0, -10.0, 5000.0), crs="EPSG:32633")
    full, md = conv.flac_to_array(path)
    plain = tmp_path / "plain.flac"
    plain.write_bytes(_strip_index(path.read_bytes()))
    tiles = tile_grid(H, W, max(H, W))
    for k, (c, r, w, h) in enumerate(_windows(H, W, 4096, seed=k_seed(dtype, bands))):
        want = full[:, r:r + h, c:c + w]
        got, meta = conv.read_window(path, c, r, w, h)
        assert _eq(got, want), (dtype, bands, (c, r, w, h))
        # a subset decode: exactly the frames of the run (indexed path)
        assert meta["frames_decoded"] == int(window_frames(tiles, (c, r, w, h), 4096)[0]["n_frames"])
        assert (meta["width"], meta["height"]) == (w, h)
        assert meta["transform"][:6] == [10.0, 0.0, 1000.0 + 10.0 * c, 0.0, -10.0, 5000.0 - 10.0 * r]
        if k % 3 == 0:
            got2, _ = conv.read_window(plain, c, r, w, h)         # no seek index: scan path
            assert _eq(got2, want), (dtype, bands, (c, r, w, h), "scan")


def k_seed(dtype, bands):
    return 1000 + DTYPES.index(dtype) * 10 + bands


def test_read_window_rejects_windows_outside_the_raster(tmp_path):
    from flac_raster_b200.converter import RasterFLACConverter
    conv = RasterFLACConverter()
    path = tmp_path / "r.flac"
    conv.array_to_flac(_raster("uint16", 1, 40, 50, 1), path)
    for win in ((0, 0, 51, 1), (0, 0, 1, 41), (-1, 0, 2, 2), (0, 0, 0, 1), (49, 39, 2, 1)):
        with pytest.raises(ValueError):
            conv.read_window(path, *win)


def test_read_window_on_the_reference_golden_equals_the_oracle(rgb_pcm):
    """sample_rgb.flac was written by the reference: no seek index (scan path), metadata in the sidecar."""
    from flac_raster_b200.converter import RasterFLACConverter
    from oracle import normalization_oracle as no
    conv = RasterFLACConverter()
    px = no.denormalize_from_audio(rgb_pcm.astype(np.int16), 1.0, 255.0, "uint8", 32767).reshape(256, 256, 3).transpose(2, 0, 1)
    for c, r, w, h in ((0, 0, 256, 256), (17, 30, 61, 5), (255, 255, 1, 1), (0, 16, 256, 16), (101, 0, 3, 256)):
        got, meta = conv.read_window(GOLDEN / "sample_rgb.flac", c, r, w, h)
        assert _eq(got, px[:, r:r + h, c:c + w])
        assert meta["transform"][:6] == pytest.approx([0.0001, 0.0, -120.0 + 0.0001 * c, 0.0, -0.0001, 37.0 - 0.0001 * r])


def test_read_window_over_http_reads_only_metadata_and_the_window_frames(range_http_server):
    from flac_raster_b200.converter import RasterFLACConverter
    from flac_raster_b200.engine import tile_grid, window_frames
    base, d, log = range_http_server
    conv = RasterFLACConverter()
    H, W = 1200, 1200                                            # 352 frames
    rng = np.random.default_rng(9)
    data = (30000 + 2000 * np.sin(np.arange(W) / 50.0)[None, None] + rng.integers(-3000, 3000, (1, H, W))).astype(np.uint16)
    conv.array_to_flac(data, d / "big.flac")
    size = (d / "big.flac").stat().st_size
    blob = (d / "big.flac").read_bytes()
    hdr = flacfmt.parse_header(blob)
    for win in ((600, 700, 16, 16), (0, 0, 1, 1), (1100, 1199, 100, 1)):
        log.clear()
        got, meta = conv.read_window(f"{base}/big.flac", *win)
        local, _ = conv.read_window(d / "big.flac", *win)
        assert _eq(got, local) and _eq(got, data[:, win[1]:win[1] + win[3], win[0]:win[0] + win[2]])
        spans = [tuple(int(v) for v in r.split("=")[1].split("-")) for r in log]
        read = sum(b - a + 1 for a, b in spans)
        assert read < 0.10 * size, (read, size)
        # one range for the frames, and it is the run's byte range
        run = window_frames(tile_grid(H, W, W), win, 4096, [flacfmt.unpack_seek_index(hdr.applications[b"frbI"], 1, 4096, 352)[0]])[0]
        a = hdr.first_frame_offset + int(run["byte_offset"])
        assert spans[-1] == (a, a + int(run["byte_length"]) - 1)
        assert len(spans) <= 3


def test_read_window_reports_a_damaged_frame(tmp_path):
    from flac_raster_b200.converter import RasterFLACConverter
    from flac_raster_b200.engine import tile_grid, window_frames
    conv = RasterFLACConverter()
    H, W = 200, 300
    for bands in (1, 3):
        path = tmp_path / f"d{bands}.flac"
        conv.array_to_flac(_raster("uint16", bands, H, W, 4), path)
        blob = bytearray(path.read_bytes())
        hdr = flacfmt.parse_header(bytes(blob))
        fb = flacfmt.unpack_seek_index(hdr.applications[b"frbI"], bands, 4096, (H * W + 4095) // 4096)[0]
        win = (10, 50, 100, 40)
        run = window_frames(tile_grid(H, W, W), win, 4096, [fb])[0]
        blob[hdr.first_frame_offset + int(run["byte_offset"]) + int(run["byte_length"]) // 2] ^= 0x24
        bad = tmp_path / f"bad{bands}.flac"
        bad.write_bytes(bytes(blob))
        with pytest.raises(ValueError):
            conv.read_window(bad, *win)


@pytest.fixture(scope="module")
def container(tmp_path_factory):
    import torch
    from flac_raster_b200.spatial_encoder import build_streaming_container, write_streaming_container
    d = tmp_path_factory.mktemp("win_container")
    data = _raster("uint16", 3, 300, 260, 11)
    dev = torch.from_numpy(data.view(np.int16)).cuda().view(torch.uint16)
    tr = (10.0, 0.0, 500000.0, 0.0, -10.0, 4000000.0)
    index, headers, enc = build_streaming_container(dev, tr, "EPSG:32633", None, "uint16", 128)
    path = d / "c.flac"
    write_streaming_container(path, index, headers, enc.payload.cpu().numpy(), enc.offsets, enc.sizes)
    return path, data, tr


def test_read_bbox_equals_tiles_stitched_and_cropped(container):
    from flac_raster_b200.spatial_encoder import SpatialFLACStreamer
    path, data, tr = container
    s = SpatialFLACStreamer(path)

    def bbox(c0, r0, c1, r1):        # pixel coordinates (fractions allowed) -> map coordinates
        return (tr[2] + tr[0] * c0, tr[5] + tr[4] * r1, tr[2] + tr[0] * c1, tr[5] + tr[4] * r0)

    cases = {
        "inside one tile": (130.3, 10.5, 200.2, 100.7),
        "across four tiles": (100.5, 100.5, 150.5, 140.5),
        "ragged edge tiles": (250.1, 250.2, 260.0, 300.0),
        "whole scene": (0, 0, 260, 300),
    }
    for name, px in cases.items():
        bb = bbox(*px)
        got, meta = s.read_bbox(*bb)
        win = meta["window"]
        c0, r0, w, h = win["col_off"], win["row_off"], win["width"], win["height"]
        assert (c0, r0) == (int(np.floor(px[0])), int(np.floor(px[1]))), name
        assert (c0 + w, r0 + h) == (int(np.ceil(px[2])), int(np.ceil(px[3]))), name
        canvas = np.zeros_like(data)
        covered = np.zeros(data.shape[1:], dtype=bool)
        for arr, m in s.get_tiles_by_bbox(*bb, shard=False):
            wn = m["window"]
            canvas[:, wn["row_off"]:wn["row_off"] + wn["height"], wn["col_off"]:wn["col_off"] + wn["width"]] = arr
            covered[wn["row_off"]:wn["row_off"] + wn["height"], wn["col_off"]:wn["col_off"] + wn["width"]] = True
        assert covered[r0:r0 + h, c0:c0 + w].all(), name
        assert _eq(got, canvas[:, r0:r0 + h, c0:c0 + w]), name
        assert meta["transform"][:6] == [10.0, 0.0, tr[2] + 10.0 * c0, 0.0, -10.0, tr[5] - 10.0 * r0]
    with pytest.raises(ValueError):
        s.read_bbox(*bbox(270, 10, 280, 20))                      # east of the raster
