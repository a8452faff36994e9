"""Drop-in for flac_raster.converter.RasterFLACConverter (reference src/flac_raster/converter.py).

Same public methods and file formats; the codec work (normalisation, FLAC
encode/decode, denormalisation) runs on the GPU through the C ABI.  Raster I/O
(rasterio when present, else tiffio) and VORBIS tags stay in Python.
"""
from __future__ import annotations

import json
import logging
from pathlib import Path
from typing import Dict, Optional

import numpy as np

from . import flacfmt
from .normalization import NormalizationParams, audio_params_for
from .tiffio import Raster, read_geotiff, write_geotiff

# tag names written by the reference (converter.py:275-297)
_GEO_FIELDS = [
    "GEOSPATIAL_CRS", "GEOSPATIAL_WIDTH", "GEOSPATIAL_HEIGHT", "GEOSPATIAL_COUNT", "GEOSPATIAL_DTYPE",
    "GEOSPATIAL_NODATA", "GEOSPATIAL_DATA_MIN", "GEOSPATIAL_DATA_MAX", "GEOSPATIAL_TRANSFORM",
    "GEOSPATIAL_BOUNDS", "GEOSPATIAL_SPATIAL_TILING",
]


def affine9(transform) -> list:
    """list(rasterio Affine) has nine entries (a,b,c,d,e,f,0,0,1); the reference stores that list."""
    if transform is None:
        return []
    t = [float(v) for v in transform[:6]]
    return t + [0.0, 0.0, 1.0]


def metadata_tags(metadata: Dict) -> Dict[str, str]:
    """VORBIS_COMMENT tags exactly as _embed_metadata_in_flac writes them (converter.py:275-297)."""
    return {
        "TITLE": "Geospatial Raster Data",
        "DESCRIPTION": "TIFF raster converted to FLAC with geospatial metadata",
        "ENCODER": "FLAC-Raster v0.1.0",
        "GEOSPATIAL_CRS": str(metadata.get("crs", "")),
        "GEOSPATIAL_WIDTH": str(metadata.get("width", 0)),
        "GEOSPATIAL_HEIGHT": str(metadata.get("height", 0)),
        "GEOSPATIAL_COUNT": str(metadata.get("count", 1)),
        "GEOSPATIAL_DTYPE": str(metadata.get("dtype", "")),
        "GEOSPATIAL_NODATA": str(metadata.get("nodata", "")),
        "GEOSPATIAL_DATA_MIN": str(metadata.get("data_min", "")),
        "GEOSPATIAL_DATA_MAX": str(metadata.get("data_max", "")),
        "GEOSPATIAL_TRANSFORM": json.dumps(metadata.get("transform", [])),
        "GEOSPATIAL_BOUNDS": json.dumps(metadata.get("bounds", [])),
        "GEOSPATIAL_SPATIAL_TILING": str(metadata.get("spatial_tiling", False)),
    }


def parse_metadata_tags(tags: Dict[str, list]) -> Optional[Dict]:
    """Inverse of metadata_tags with the reference's type rules (converter.py:356-377)."""
    if "GEOSPATIAL_CRS" not in tags:
        return None
    md: Dict = {}
    for field in _GEO_FIELDS:
        if field not in tags:
            continue
        value = tags[field][0]
        key = field.replace("GEOSPATIAL_", "").lower()
        if key in ("width", "height", "count"):
            md[key] = int(value) if value else 0
        elif key in ("data_min", "data_max"):
            md[key] = float(value) if value else 0.0
        elif key in ("transform", "bounds"):
            md[key] = json.loads(value) if value else []
        elif key == "spatial_tiling":
            md[key] = value.lower() == "true"
        elif key == "nodata":
            md[key] = None if value == "None" else float(value) if value else None
        else:
            md[key] = value
    return md


def tile_metadata(width, height, count, dtype, crs, transform, data_min, data_max, nodata, scale_factor) -> Dict:
    """The raster_metadata dict of tiff_to_flac (converter.py:117-135)."""
    t = transform or (1.0, 0.0, 0.0, 0.0, -1.0, 0.0)
    left, top = t[2], t[5]
    return {
        "width": width, "height": height, "count": count, "dtype": str(dtype),
        "crs": crs, "transform": affine9(transform) if transform else None,
        "bounds": {"left": left, "bottom": top + height * t[4], "right": left + width * t[0], "top": top},
        "data_min": data_min, "data_max": data_max, "nodata": nodata, "driver": "GTiff",
        "scale_factor": scale_factor,
    }


def build_flac_file(frames: bytes, n_samples: int, channels: int, bps: int, sample_rate: int, blocksize: int,
                    metadata: Optional[Dict], padding: int = 0, seek_index: Optional[bytes] = None) -> bytes:
    """STREAMINFO + VORBIS tags (+ seek index) (+ padding) + frames: one standalone FLAC file."""
    si = flacfmt.StreamInfo(blocksize, blocksize, 0, 0, sample_rate, channels, bps, n_samples)
    tags = metadata_tags(metadata) if metadata else {}
    return flacfmt.build_header(si, tags, padding=padding, seek_index=seek_index) + bytes(frames)


class RasterFLACConverter:
    """Handles conversion between TIFF and FLAC formats for raster data (GPU codec)."""

    def __init__(self):
        self.metadata_key = "RASTER_METADATA"
        self.logger = logging.getLogger("flac_raster.converter")

    # ------------------------------------------------------------------ encode
    def tiff_to_flac(self, tiff_path: Path, flac_path: Path, compression_level: int = 5,
                     spatial_tiling: bool = False, tile_size: int = 512):
        """Convert TIFF raster to FLAC format (reference converter.py:41-172)."""
        tiff_path, flac_path = Path(tiff_path), Path(flac_path)
        self.logger.info(f"Starting TIFF to FLAC conversion: {tiff_path} -> {flac_path}")
        if spatial_tiling:
            from .spatial_encoder import SpatialFLACEncoder

            encoder = SpatialFLACEncoder(tile_size=tile_size)
            return encoder.encode_spatial_flac(tiff_path, flac_path, compression_level)
        raster = read_geotiff(tiff_path)
        data = self.array_to_flac(raster.data, flac_path, compression_level, transform=raster.transform,
                                  crs=raster.crs, nodata=raster.nodata)
        out_size, in_size = flac_path.stat().st_size, tiff_path.stat().st_size
        self.logger.info(f"Conversion complete: {out_size / 1024 / 1024:.2f} MB "
                         f"(compression: {(1 - out_size / in_size) * 100:.1f}%)")
        return data

    def array_to_flac(self, data: np.ndarray, flac_path: Path, compression_level: int = 5, transform=None,
                      crs: Optional[str] = None, nodata=None):
        """Encode a (bands,H,W) or (H,W) array as one FLAC file (the body of tiff_to_flac)."""
        import torch
        from .engine import default_engine, tile_grid

        arr = data if data.ndim == 3 else data[None]
        bands, H, W = arr.shape
        if bands > 8:
            raise ValueError("FLAC supports at most 8 channels (bands)")
        eng = default_engine()
        dev = torch.from_numpy(np.ascontiguousarray(arr).view(np.uint8).reshape(-1)).to(eng.device)
        from .engine import TORCH_DTYPES
        dev = dev.view(TORCH_DTYPES[str(arr.dtype)]).reshape(bands, H, W)
        tiles = tile_grid(H, W, max(H, W))
        enc = eng.encode_tiles(dev, tiles, compression_level)
        frames = enc.payload.cpu().numpy().tobytes()
        scale = 32767 if enc.bits_per_sample == 16 else 8388607
        md = tile_metadata(W, H, bands, arr.dtype, crs, transform, float(enc.minmax[0, 0]), float(enc.minmax[0, 1]),
                           nodata, scale)
        sidx = None
        if enc.frame_bytes is not None:
            sidx = flacfmt.pack_seek_index(bands, enc.blocksize, enc.frame_bytes.cpu().numpy().view(np.uint32),
                                           enc.sub_bitoff.cpu().numpy().view(np.uint32))
        blob = build_flac_file(frames, int(enc.n_samples[0]), bands, enc.bps, int(enc.sample_rates[0]), enc.blocksize,
                               md, padding=1024, seek_index=sidx)
        Path(flac_path).write_bytes(blob)
        return None

    # ------------------------------------------------------------------ decode
    def flac_to_tiff(self, flac_path: Path, tiff_path: Path):
        """Convert FLAC back to TIFF format (reference converter.py:174-261)."""
        flac_path, tiff_path = Path(flac_path), Path(tiff_path)
        data, metadata = self.flac_to_array(flac_path)
        transform = tuple(metadata["transform"][:6]) if metadata.get("transform") else None
        write_geotiff(tiff_path, data, transform, metadata.get("crs") or None, metadata.get("nodata"))
        self.logger.info(f"TIFF written successfully: {tiff_path.stat().st_size / 1024 / 1024:.2f} MB")

    def flac_to_array(self, flac_path: Path):
        """Decode one FLAC file to ((bands,H,W) array in the original dtype, metadata dict)."""
        flac_path = Path(flac_path)
        blob = flac_path.read_bytes()
        hdr = flacfmt.parse_header(blob)
        metadata = parse_metadata_tags(hdr.tags)
        if not metadata:
            sidecar = flac_path.with_suffix(".json")
            if sidecar.exists():
                metadata = json.loads(sidecar.read_text())
        if not metadata:
            self.logger.error("No metadata found in FLAC file or sidecar file")
            raise ValueError("No metadata found in FLAC file or sidecar file")
        return decode_tile_blobs([blob], [hdr], [metadata])[0], metadata

    def read_window(self, flac_path_or_url, col_off: int, row_off: int, width: int, height: int):
        """The pixels of one window of a FLAC raster file (local path or URL) -> ((bands, height, width) array in the
        original dtype, metadata).  Only the frames that cover the window are decoded: the metadata chain is read first,
        then, when the file carries the "frbI" seek index, only the byte range of those frames (one read, or one HTTP
        range request).  A file without the index (e.g. one the reference wrote) is read whole and its frames are found by
        the sync scan.  The metadata is the file's, with width, height, transform and bounds of the window, and
        `frames_decoded`.  Only the decoded frames are validated: damage in a frame outside the window goes unnoticed."""
        import torch
        from . import _native as nat
        from .engine import TORCH_DTYPES, default_engine, window_frames
        from .remote import RemoteFile, is_remote_url
        from .tiffio import window_transform

        src = str(flac_path_or_url)
        if is_remote_url(src):
            rf = RemoteFile(src)

            def read(start: int, n: int) -> bytes:
                return rf.read_range(start, start + n - 1) if n > 0 else b""
        else:
            path = Path(src)

            def read(start: int, n: int) -> bytes:
                with open(path, "rb") as f:
                    f.seek(start)
                    return f.read(n)          # n = -1: to the end
        hdr = flacfmt.read_header(read)
        metadata = parse_metadata_tags(hdr.tags)
        if not metadata and not is_remote_url(src) and Path(src).with_suffix(".json").exists():
            metadata = json.loads(Path(src).with_suffix(".json").read_text())
        if not metadata:
            raise ValueError("No metadata found in FLAC file or sidecar file")
        si = hdr.streaminfo
        bands, bps, blocksize = si.channels, si.bits_per_sample, si.max_blocksize
        W, H = int(metadata["width"]), int(metadata["height"])
        if metadata["count"] != bands:
            raise ValueError("band count in tags does not match the FLAC channel count")
        col_off, row_off, width, height = int(col_off), int(row_off), int(width), int(height)
        if width < 1 or height < 1 or col_off < 0 or row_off < 0 or col_off + width > W or row_off + height > H:
            raise ValueError(f"window (col_off={col_off}, row_off={row_off}, width={width}, height={height}) "
                             f"is not inside the {W} x {H} raster")
        window = (col_off, row_off, width, height)
        tiles = np.zeros(1, dtype=nat.TILE_DTYPE)
        tiles[0] = (0, 0, H, W)
        n_frames = (W * H + blocksize - 1) // blocksize
        blk = hdr.applications.get(flacfmt.SEEK_INDEX_ID)
        index = flacfmt.unpack_seek_index(blk, bands, blocksize, n_frames) if blk else None
        dtype = np.dtype(metadata["dtype"])
        scale = float(metadata.get("scale_factor") or (32767 if bps == 16 else 8388607))     # as flac_to_array
        if bps == 16:
            scale = 32767.0
        minmax = np.array([[metadata["data_min"], metadata["data_max"]]], dtype=np.float64)
        rates = np.array([si.sample_rate], dtype=np.uint32)
        eng = default_engine()
        out = torch.empty((bands, height, width), dtype=TORCH_DTYPES[str(dtype)], device=eng.device)

        def to_device(blob: bytes) -> "torch.Tensor":
            host = np.zeros(len(blob) + 64, dtype=np.uint8)
            host[:len(blob)] = np.frombuffer(blob, dtype=np.uint8)
            return torch.from_numpy(host).to(eng.device)

        status = None
        if index is not None:
            run = window_frames(tiles, window, blocksize, [index[0]])[0]
            blob = read(hdr.first_frame_offset + int(run["byte_offset"]), int(run["byte_length"]))
            if len(blob) == int(run["byte_length"]):
                status = eng.decode_window(to_device(blob), np.zeros(1, np.int64), np.array([len(blob)]), tiles, rates, minmax,
                                           scale, window, out, bps, blocksize, index=index, runs_only=True)
        if status is None or nat.status_damaged(status):
            # no index, or one that does not describe the frames: every frame is needed to find the window's by scanning
            blob = read(hdr.first_frame_offset, -1) if not is_remote_url(src) else rf.read_all()[hdr.first_frame_offset:]
            status = eng.decode_window(to_device(blob), np.zeros(1, np.int64), np.array([len(blob)]), tiles, rates, minmax,
                                       scale, window, out, bps, blocksize)
        _raise_for_status(status)
        res = out.cpu().numpy()
        meta = dict(metadata)
        tr = metadata.get("transform")
        t6 = window_transform(tuple(tr[:6]), col_off, row_off) if tr else None
        left, top = (t6[2], t6[5]) if t6 else (float(col_off), -float(row_off))
        meta.update({"width": width, "height": height, "transform": affine9(t6) if t6 else tr,
                     "bounds": {"left": left, "bottom": top + height * (t6[4] if t6 else -1.0),
                                "right": left + width * (t6[0] if t6 else 1.0), "top": top},
                     "window": {"col_off": col_off, "row_off": row_off, "width": width, "height": height},
                     "frames_decoded": int(status[nat.ST_FRAMES_DECODED])})
        return res, meta

    # kept for signature compatibility with the reference (converter.py:263, :329)
    def _embed_metadata_in_flac(self, flac_path: Path, metadata: Dict):
        blob = Path(flac_path).read_bytes()
        hdr = flacfmt.parse_header(blob)
        out = flacfmt.build_header(hdr.streaminfo, metadata_tags(metadata), padding=1024) + blob[hdr.first_frame_offset:]
        Path(flac_path).write_bytes(out)

    def _read_embedded_metadata(self, flac_path: Path) -> Optional[Dict]:
        try:
            hdr = flacfmt.parse_header(Path(flac_path).read_bytes())
            md = parse_metadata_tags(hdr.tags)
            if md:
                return md
        except ValueError as e:
            self.logger.warning(f"Failed to read embedded metadata: {e}")
        sidecar = Path(flac_path).with_suffix(".json")
        if sidecar.exists():
            return json.loads(sidecar.read_text())
        return None


def decode_tile_blobs(blobs, headers, metadatas, mosaic=None, staged=None):
    """Batch-decode complete per-tile FLAC files on the GPU.

    blobs: list of bytes (each a standalone FLAC file as the streaming container holds them,
    cli.py:594-598); headers/metadatas: parsed per tile.  Returns a list of (bands,h,w) arrays
    in the original dtype (denormalize_from_audio integer path, normalization.py:222-249).
    staged=(pinned uint8 tensor, nbytes, tile_starts): the tiles already sit in one pinned buffer (read straight
    from the file, see SpatialFLACStreamer._decode); blobs are then views into it and nothing is copied on the host.
    """
    import torch
    from . import _native as nat
    from .engine import TORCH_DTYPES, default_engine

    eng = default_engine()
    n = len(blobs)
    si0 = headers[0].streaminfo
    channels, bps, blocksize = si0.channels, si0.bits_per_sample, si0.max_blocksize
    offs = np.zeros(n, dtype=np.int64)
    lens = np.zeros(n, dtype=np.int64)
    nsamp = np.zeros(n, dtype=np.int64)
    rates = np.zeros(n, dtype=np.uint32)
    tiles = np.zeros(n, dtype=nat.TILE_DTYPE)
    minmax = np.zeros((n, 2), dtype=np.float64)
    pos = 0
    row = 0
    maxw = 0
    bodies = []
    idx_fb, idx_sb = [], []          # seek index of every tile ("frbI" block); None as soon as one tile has none
    for i, (b, h, md) in enumerate(zip(blobs, headers, metadatas)):
        si = h.streaminfo
        if (si.channels, si.bits_per_sample, si.max_blocksize) != (channels, bps, blocksize):
            raise ValueError("tiles of one batch must share channels, bits per sample and blocksize")
        if md["count"] != si.channels:
            raise ValueError("band count in tags does not match the FLAC channel count")
        if staged is None:
            body = memoryview(b)[h.first_frame_offset:]
            offs[i], lens[i] = pos, len(body)
            bodies.append(body)
            pos += (len(body) + 3) & ~3
        else:
            offs[i], lens[i] = int(staged[2][i]) + h.first_frame_offset, len(b) - h.first_frame_offset
        nsamp[i] = md["width"] * md["height"]
        if idx_fb is not None:
            blk = h.applications.get(flacfmt.SEEK_INDEX_ID) if getattr(h, "applications", None) else None
            got = flacfmt.unpack_seek_index(blk, channels, blocksize, (int(nsamp[i]) + blocksize - 1) // blocksize) if blk else None
            if got is None:
                idx_fb = idx_sb = None
            else:
                idx_fb.append(got[0])
                idx_sb.append(got[1])
        rates[i] = si.sample_rate
        tiles[i] = (row, 0, md["height"], md["width"])
        row += md["height"]
        maxw = max(maxw, md["width"])
        minmax[i] = (md["data_min"], md["data_max"])
    if staged is None:
        # frames of all tiles -> one pinned staging buffer (no intermediate bytes objects) -> one H2D copy
        stage = eng._pinned("dec_stage", pos + 64)
        stage_np = stage.numpy()
        for i, body in enumerate(bodies):
            o = int(offs[i])
            stage_np[o:o + len(body)] = np.frombuffer(body, dtype=np.uint8)
            pad = (-len(body)) % 4
            if pad:
                stage_np[o + len(body):o + len(body) + pad] = 0
    else:
        stage, pos = staged[0], int(staged[1])
        stage_np = stage.numpy()
    stage_np[pos:pos + 64] = 0
    data = eng._buf("dec_data", pos + 64)[:pos + 64]
    data.copy_(stage[:pos + 64], non_blocking=True)
    dtype = np.dtype(metadatas[0]["dtype"])
    # decode default scale by audio width (converter.py:220-229)
    scale = float(metadatas[0].get("scale_factor") or (32767 if bps == 16 else 8388607))
    if bps == 16:
        scale = 32767.0
    out = torch.zeros(channels * row * maxw * dtype.itemsize, dtype=torch.uint8, device=eng.device)
    out = out.view(TORCH_DTYPES[str(dtype)]).reshape(channels, row, maxw)
    # one fused launch: Rice decode + predictor restore + denormalise straight into the tile windows
    index = None
    if idx_fb:
        index = (np.concatenate(idx_fb), np.concatenate(idx_sb) if channels > 1 else None)
    status = eng.decode_tiles(data, offs, lens, tiles, rates, minmax, scale, out, bps, blocksize, index=index)
    _raise_for_status(status)
    # D2H through a pinned buffer, then every tile becomes its own array (the buffer is reused by the next call);
    # the per-tile copies run on a few threads (numpy releases the GIL while copying)
    nbytes = out.numel() * dtype.itemsize
    pinned = eng._pinned("dec_out", nbytes)
    pinned[:nbytes].copy_(out.reshape(-1).view(torch.uint8), non_blocking=True)
    torch.cuda.current_stream().synchronize()
    host_out = pinned[:nbytes].numpy().view(dtype).reshape(channels, row, maxw)

    def take(i):
        r0, h_, w_ = int(tiles[i]["row_off"]), int(tiles[i]["h"]), int(tiles[i]["w"])
        # a real copy, always: host_out is a view of the engine's reusable pinned buffer, and ascontiguousarray would hand
        # an already contiguous slice (single tile, full-width single-band tiles) straight back to the caller, to be
        # overwritten by the next decode (the reference returns independent arrays)
        return np.array(host_out[:, r0:r0 + h_, :w_], copy=True, order="C")

    if n >= 64:
        from concurrent.futures import ThreadPoolExecutor
        jobs = [range(a, min(n, a + (n + 31) // 32)) for a in range(0, n, (n + 31) // 32)]
        with ThreadPoolExecutor(8) as ex:
            res = [a for part in ex.map(lambda rg: [take(i) for i in rg], jobs) for a in part]
    else:
        res = [take(i) for i in range(n)]
    return res


_DTYPE_NAMES = ["uint8", "int8", "uint16", "int16", "uint32", "int32", "float32", "float64"]


def decode_staged_tiles(stage, nbytes: int, starts: np.ndarray, sizes: np.ndarray, data=None, while_copying=None):
    """Fast form of decode_tile_blobs for tiles that already sit in ONE pinned staging buffer (SpatialFLACStreamer reads the
    byte ranges of a bbox query straight into it): the per-tile metadata walk runs in C (frb_parse_tile_headers) instead of
    4096 Python header parses, the seek indices are gathered in C, and single-band tiles of equal width come back as views
    of a pinned result buffer that belongs to the returned arrays (no second host copy; torch's pinned allocator recycles the
    block once the arrays are dropped).  Returns (arrays, header records) or None when a tile does not qualify (no
    GEOSPATIAL tags, mixed geometry): the caller then takes the general path.
    data: the staging buffer's bytes already on the device (the reader sent them piece by piece), else they are copied here.
    while_copying(header records): called while the device-to-host copy of the pixels is in flight."""
    import ctypes as C

    import torch
    from . import _native as nat
    from .engine import TORCH_DTYPES, default_engine

    eng = default_engine()
    L = nat.lib()
    n = len(starts)
    stage_np = stage.numpy()
    offs64 = np.ascontiguousarray(starts, dtype=np.uint64)
    size64 = np.ascontiguousarray(sizes, dtype=np.uint64)
    hdr = np.zeros(n, dtype=nat.TILE_HEADER_DTYPE)
    rc = L.frb_parse_tile_headers(stage_np.ctypes.data, offs64.ctypes.data, size64.ctypes.data, n, hdr.ctypes.data)
    if rc != nat.FRB_OK:
        raise ValueError("not a FLAC stream (missing fLaC marker)")
    h0 = hdr[0]
    channels, bps, blocksize = int(h0["channels"]), int(h0["bps"]), int(h0["max_blocksize"])
    same = (hdr["channels"] == channels) & (hdr["bps"] == bps) & (hdr["max_blocksize"] == blocksize) & (hdr["dtype"] == h0["dtype"])
    if not same.all():
        raise ValueError("tiles of one batch must share channels, bits per sample and blocksize")
    if not ((hdr["flags"] & 1) != 0).all() or h0["dtype"] < 0 or (hdr["width"] == 0).any() or (hdr["height"] == 0).any():
        return None
    if not (hdr["count"] == channels).all():
        raise ValueError("band count in tags does not match the FLAC channel count")
    dtype = np.dtype(_DTYPE_NAMES[int(h0["dtype"])])
    hdr_in = hdr                                   # records in the caller's tile order (what is returned)
    widths = hdr["width"].astype(np.int64)
    heights = hdr["height"].astype(np.int64)
    # Multi-band tiles: the decode writes band-major planes (band, tile rows stacked, width), so a tile is strided across its
    # bands.  Tiles of the full size (all of them, or the interior of a scene whose edge tiles are ragged) are decoded FIRST:
    # their part of the planes is re-laid out to (tile, band, h, w) on the device and handed out as views of the result block;
    # only the ragged rest takes a strided host copy per tile (1.9 GB of host copies for a bbox query over an 8-band C3 scene).
    order, n_full = full_tiles_first(widths, heights, channels)
    if order is not None:
        hdr, offs64, size64 = hdr[order], np.ascontiguousarray(offs64[order]), np.ascontiguousarray(size64[order])
        widths, heights = widths[order], heights[order]
    nsamp = widths * heights
    tiles = np.zeros(n, dtype=nat.TILE_DTYPE)
    rows0 = np.zeros(n, dtype=np.int64)
    np.cumsum(heights[:-1], out=rows0[1:])
    tiles["row_off"] = rows0
    tiles["h"] = heights
    tiles["w"] = widths
    row, maxw = int(heights.sum()), int(widths.max())
    offs = offs64.astype(np.int64) + hdr["first_frame_offset"].astype(np.int64)
    lens = size64.astype(np.int64) - hdr["first_frame_offset"].astype(np.int64)
    minmax = np.stack([hdr["data_min"], hdr["data_max"]], axis=1)
    scale = 32767.0 if bps == 16 else 8388607.0                  # decode default by audio width (converter.py:220-229)
    # seek indices of all tiles, concatenated in C
    index = None
    fpt = ((nsamp + blocksize - 1) // blocksize).astype(np.uint32)
    if ((hdr["flags"] & 4) != 0).all():
        nf = int(fpt.sum())
        fb = np.empty(nf, dtype=np.uint32)
        sb = np.empty(nf * channels, dtype=np.uint32) if channels > 1 else None
        rc = L.frb_gather_seek_index(stage_np.ctypes.data, offs64.ctypes.data, hdr.ctypes.data, n, channels, blocksize, fpt.ctypes.data,
                                     fb.ctypes.data, sb.ctypes.data if sb is not None else None)
        if rc == nat.FRB_OK:
            index = (fb, sb)
    if data is None:
        stage_np[nbytes:nbytes + 64] = 0
        data = eng._buf("dec_data", nbytes + 64)[:nbytes + 64]
        data.copy_(stage[:nbytes + 64], non_blocking=True)
    out = torch.zeros(channels * row * maxw * dtype.itemsize, dtype=torch.uint8, device=eng.device)
    out = out.view(TORCH_DTYPES[str(dtype)]).reshape(channels, row, maxw)
    status = eng.decode_tiles(data, offs, lens, tiles, hdr["sample_rate"].astype(np.uint32), minmax, scale, out, bps, blocksize, index=index)
    _raise_for_status(status)
    nb = out.numel() * dtype.itemsize
    # result buffer: a fresh pinned block per call (cached by torch's host allocator), owned by the arrays handed out
    host = torch.empty(nb, dtype=torch.uint8, pin_memory=True)
    if n_full:
        hf = int(heights[0])
        nb_full = channels * n_full * hf * maxw * dtype.itemsize
        tm_dev = out[:, :n_full * hf].reshape(channels, n_full, hf, maxw).permute(1, 0, 2, 3).contiguous()
        host[:nb_full].copy_(tm_dev.reshape(-1).view(torch.uint8), non_blocking=True)
        if n_full < n:
            rest_dev = out[:, n_full * hf:].contiguous()
            host[nb_full:].copy_(rest_dev.reshape(-1).view(torch.uint8), non_blocking=True)
        if while_copying is not None:
            while_copying(hdr_in)
        torch.cuda.current_stream().synchronize()
        tm = host[:nb_full].numpy().view(dtype).reshape(n_full, channels, hf, maxw)
        arrays = [tm[i] for i in range(n_full)]
        if n_full < n:
            rest = host[nb_full:].numpy().view(dtype).reshape(channels, row - n_full * hf, maxw)
            arrays += _copy_tiles_out(rest, rows0[n_full:] - n_full * hf, heights[n_full:], widths[n_full:])
        if order is not None:
            back = [None] * n
            for i, o in enumerate(order):
                back[int(o)] = arrays[i]
            arrays = back
        return arrays, hdr_in
    host.copy_(out.reshape(-1).view(torch.uint8), non_blocking=True)
    if while_copying is not None:
        while_copying(hdr_in)
    torch.cuda.current_stream().synchronize()
    host_out = host.numpy().view(dtype).reshape(channels, row, maxw)
    if n == 1:
        arrays = [host_out]                      # one tile (get_tile_by_id): the result block IS the tile, whatever its band count
    elif channels == 1 and (widths == maxw).all():
        arrays = [host_out[:, int(r0):int(r0 + h_)] for r0, h_ in zip(rows0, heights)]     # C-contiguous views, one owner
    else:
        arrays = _copy_tiles_out(host_out, rows0, heights, widths)
    return arrays, hdr_in


def full_tiles_first(widths, heights, channels: int):
    """Decode order of a batch of multi-band tiles: (order, n_full).  The n_full tiles of the full size (largest width AND
    largest height of the batch) come first, in their original relative order, then the ragged ones; order is None when nothing
    moves (every tile is full size, or they already lead).  n_full is 0 for single-band batches, single tiles and batches with
    fewer than two full-size tiles: those keep the band-major result layout."""
    widths, heights = np.asarray(widths), np.asarray(heights)
    n = len(widths)
    if n < 2 or channels < 2:
        return None, 0
    full = (widths == widths.max()) & (heights == heights.max())
    n_full = int(full.sum())
    if n_full < 2:
        return None, 0
    if n_full == n or bool(full[:n_full].all()):
        return None, n_full
    return np.argsort(~full, kind="stable"), n_full


def _raise_for_status(status):
    from . import _native as nat
    if status[nat.ST_OFFSET_WAIT_TIMEOUTS]:
        raise RuntimeError("decode kernel timed out waiting for a subframe offset")
    if status[nat.ST_FRAMES_MISSING] or status[nat.ST_PARSE_ERRORS]:
        raise ValueError(f"malformed FLAC stream (missing frames={status[nat.ST_FRAMES_MISSING]}, parse errors={status[nat.ST_PARSE_ERRORS]})")
    if status[nat.ST_CRC16_ERRORS]:
        raise ValueError(f"FLAC frame CRC-16 mismatch in {status[nat.ST_CRC16_ERRORS]} frame(s)")


def _copy_tiles_out(host_out, rows0, heights, widths):
    """Every tile becomes its own C-contiguous array (multi-band or ragged tiles are strided inside the stacked buffer); the
    copies run on a few threads (numpy releases the GIL while copying)."""
    n = len(rows0)

    def take(i):
        return np.array(host_out[:, int(rows0[i]):int(rows0[i] + heights[i]), :int(widths[i])], copy=True, order="C")

    if n >= 64:
        from concurrent.futures import ThreadPoolExecutor
        step = (n + 31) // 32
        jobs = [range(a, min(n, a + step)) for a in range(0, n, step)]
        with ThreadPoolExecutor(8) as ex:
            return [a for part in ex.map(lambda rg: [take(i) for i in rg], jobs) for a in part]
    return [take(i) for i in range(n)]
