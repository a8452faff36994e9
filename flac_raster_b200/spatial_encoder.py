"""Drop-in for flac_raster.spatial_encoder (reference src/flac_raster/spatial_encoder.py) plus the
streaming container of cli.py:521-639 behind the README API (README.md:195-202):

    SpatialFLACEncoder(tile_size=1024).encode("in.tif", "out.flac", streaming=True)
    streamer = SpatialFLACStreamer("out.flac")
    tile, meta = streamer.get_tile_by_id(42)
    tiles = streamer.get_tiles_by_bbox(xmin, ymin, xmax, ymax)

Streaming container (cli.py:625-630): [u32 BE index length][JSON index][tile FLAC files...];
every tile is a complete standalone FLAC file with its own per-tile min/max tags, exactly what
_create_streaming_flac produces by running tiff_to_flac on each window.  All tiles are encoded
by ONE batched GPU call instead of the reference's serial per-tile loop, and all tiles of a
bbox query are decoded by one batched call.
"""
from __future__ import annotations

import base64
import gzip
import json
import logging
import os
import struct
from pathlib import Path
from typing import Dict, List, Optional, Tuple

import numpy as np

from . import flacfmt
from .converter import (RasterFLACConverter, build_flac_file, decode_staged_tiles, decode_tile_blobs, parse_metadata_tags,
                        tile_metadata)
from .tiffio import read_geotiff, window_transform


class _Window:
    """Stand-in for rasterio.windows.Window (only the four attributes the index needs)."""

    def __init__(self, col_off, row_off, width, height):
        self.col_off, self.row_off, self.width, self.height = col_off, row_off, width, height


class SpatialFrame:
    """Represents a spatial FLAC frame with bbox metadata (spatial_encoder.py:34-64)."""

    def __init__(self, frame_id: int, bbox: Tuple[float, float, float, float], window, byte_offset: int = 0,
                 byte_size: int = 0):
        self.frame_id = frame_id
        self.bbox = bbox
        self.window = window
        self.byte_offset = byte_offset
        self.byte_size = byte_size

    def to_dict(self) -> Dict:
        return {
            "frame_id": self.frame_id,
            "bbox": self.bbox,
            "window": {
                "row_off": self.window.row_off,
                "col_off": self.window.col_off,
                "height": self.window.height,
                "width": self.window.width,
            },
            "byte_offset": self.byte_offset,
            "byte_size": self.byte_size,
        }


class SpatialIndex:
    """Spatial index for FLAC frames with bbox lookup (spatial_encoder.py:67-96)."""

    def __init__(self, frames: List[SpatialFrame], crs, transform):
        self.frames = frames
        self.crs = crs
        self.transform = transform
        self.total_bytes = sum(frame.byte_size for frame in frames)

    def query_bbox(self, bbox: Tuple[float, float, float, float]) -> List[SpatialFrame]:
        xmin, ymin, xmax, ymax = bbox
        out = []
        for frame in self.frames:
            fxmin, fymin, fxmax, fymax = frame.bbox
            if xmin < fxmax and xmax > fxmin and ymin < fymax and ymax > fymin:   # strict, spatial_encoder.py:85
                out.append(frame)
        return out

    def to_dict(self) -> Dict:
        return {
            "crs": str(self.crs),
            "transform": list(self.transform) if self.transform else [],
            "frames": [frame.to_dict() for frame in self.frames],
        }


def _tile_bbox(transform, col, row, w, h):
    """cli.py:561-565: xmin=c, ymax=f of the window transform; north-up assumed."""
    t = window_transform(transform or (1.0, 0.0, 0.0, 0.0, -1.0, 0.0), col, row)
    xmin, ymax = t[2], t[5]
    return [xmin, ymax + h * t[4], xmin + w * t[0], ymax], t


def build_streaming_container(raster_dev, transform, crs, nodata, dtype_name: str, tile_size: int,
                              compression_level: int = 5, tiles: Optional[np.ndarray] = None, engine=None,
                              row_origin: int = 0, full_shape: Optional[Tuple[int, int, int]] = None, seek_index: bool = True):
    """Encode every tile of a device-resident (bands,H,W) raster and lay out the container.

    Returns (index dict, list of per-tile header bytes, EncodedTiles).  Tile t's complete FLAC
    file is headers[t] + payload[offsets[t]:offsets[t]+sizes[t]]; index byte_offset/byte_size are
    the exclusive scan of the file sizes (cli.py:615-621).
    `tiles` are in the coordinates of the FULL raster (`full_shape`, default: raster_dev's own); `row_origin` is the
    global row raster_dev[:, 0] holds (a rank of the sharded path passes only the rows its tiles touch), so every
    tile's transform/bounds tags are computed exactly as the one-GPU path computes them.
    """
    from .engine import default_engine, tile_grid

    eng = engine or default_engine()
    bands, H, W = full_shape if full_shape is not None else raster_dev.shape
    if tiles is None:
        tiles = tile_grid(H, W, tile_size)
    local = tiles
    if row_origin:
        local = tiles.copy()
        local["row_off"] -= row_origin
    if raster_dev.is_cuda:
        enc = eng.encode_tiles(raster_dev, local, compression_level)
    else:       # host raster: tile rows pipelined over copy / compute / copy streams (Engine.encode_tiles_host)
        enc = eng.encode_tiles_host(raster_dev, local, compression_level)
    scale = 32767 if enc.bits_per_sample == 16 else 8388607
    headers, frames = [], []
    total = 0
    a9 = (list(transform[:6]) + [0.0, 0.0, 1.0]) if transform else []
    # seek index per tile ("frbI" APPLICATION block): frame sizes + subframe bit offsets, so that a tile fetched later is
    # decoded without the sync scan and the walk for subframe starts
    fb_all = sb_all = None
    if seek_index and enc.frame_bytes is not None:
        fb_all = enc.frame_bytes.cpu().numpy().view(np.uint32)
        sb_all = enc.sub_bitoff.cpu().numpy().view(np.uint32)
        fstart = np.concatenate([[0], np.cumsum(enc.frames_per_tile())])
    for i, t in enumerate(tiles):
        r, c, h, w = int(t["row_off"]), int(t["col_off"]), int(t["h"]), int(t["w"])
        bbox, ttrans = _tile_bbox(transform, c, r, w, h)
        md = tile_metadata(w, h, bands, dtype_name, crs, ttrans if transform else None,
                           float(enc.minmax[i, 0]), float(enc.minmax[i, 1]), nodata, scale)
        si = flacfmt.StreamInfo(enc.blocksize, enc.blocksize, 0, 0, int(enc.sample_rates[i]), bands, enc.bps, int(enc.n_samples[i]))
        from .converter import metadata_tags
        sidx = None
        if fb_all is not None:
            f0, f1 = int(fstart[i]), int(fstart[i + 1])
            sidx = flacfmt.pack_seek_index(bands, enc.blocksize, fb_all[f0:f1], sb_all[f0 * bands:f1 * bands])
        hdr = flacfmt.build_header(si, metadata_tags(md), seek_index=sidx)
        headers.append(hdr)
        size = len(hdr) + int(enc.sizes[i])
        frames.append({
            "frame_id": i,
            "bbox": bbox,
            "window": {"col_off": c, "row_off": r, "width": w, "height": h},
            "byte_offset": total,
            "byte_size": size,
        })
        total += size
    index = {
        "crs": str(crs), "transform": a9, "width": W, "height": H, "bands": bands, "dtype": dtype_name,
        "tile_size": tile_size, "frames": frames,
    }
    return index, headers, enc


def write_streaming_container(path, index: Dict, headers: List[bytes], payload: np.ndarray, offsets, sizes):
    """cli.py:625-630."""
    index_json = json.dumps(index, separators=(",", ":")).encode("utf-8")
    mv = memoryview(payload)
    with open(path, "wb") as f:
        f.write(len(index_json).to_bytes(4, "big"))
        f.write(index_json)
        for h, o, s in zip(headers, offsets, sizes):
            f.write(h)
            f.write(mv[int(o):int(o) + int(s)])
    return 4 + len(index_json)


class SpatialFLACEncoder:
    """Enhanced FLAC encoder with spatial tiling and bbox metadata (GPU-batched)."""

    def __init__(self, tile_size: int = 512):
        self.tile_size = tile_size
        self.logger = logging.getLogger("flac_raster.spatial_encoder")
        self.frames: List[SpatialFrame] = []
        self.current_frame_id = 0
        self.bytes_written = 0
        self.output_file = None

    def _calculate_tiles(self, height: int, width: int) -> List[Tuple[int, int, int, int]]:
        tiles = []
        for row_start in range(0, height, self.tile_size):
            for col_start in range(0, width, self.tile_size):
                row_end = min(row_start + self.tile_size, height)
                col_end = min(col_start + self.tile_size, width)
                tiles.append((row_start, col_start, row_end - row_start, col_end - col_start))
        return tiles

    def _tile_to_bbox(self, row_off, col_off, height, width, transform):
        bbox, _ = _tile_bbox(transform, col_off, row_off, width, height)
        return tuple(bbox)

    # ---- README API -------------------------------------------------------------------
    def encode(self, input_path, output_path, streaming: bool = True, compression_level: int = 5,
               tile_size: Optional[int] = None):
        """README.md:196-197.  streaming=True writes the Netflix-style container of cli.py:521-639."""
        if tile_size is not None:
            self.tile_size = tile_size
        if not streaming:
            return self.encode_spatial_flac(Path(input_path), Path(output_path), compression_level)
        import torch
        from .engine import TORCH_DTYPES, default_engine

        raster = read_geotiff(input_path)
        arr = raster.data
        if arr.shape[0] > 8:
            raise ValueError("FLAC supports at most 8 channels (bands)")
        eng = default_engine()
        from .distributed import current_rank_world, encode_streaming_sharded, shard_plan
        rank, world = current_rank_world()
        if world > 1:
            # one process per GPU (torch.distributed initialised by the caller): the tiles of this raster are split
            # over the ranks, every rank writes its own part of ONE container (distributed.encode_streaming_sharded)
            bands, H, W = arr.shape
            _, _, (r0, r1) = shard_plan(H, W, self.tile_size, rank, world)
            sl = np.ascontiguousarray(arr[:, r0:r1])
            host = torch.from_numpy(sl.view(np.uint8).reshape(-1)).view(TORCH_DTYPES[str(arr.dtype)]).reshape(sl.shape)
            index, _, _ = encode_streaming_sharded(host, r0, (bands, H, W), raster.transform, raster.crs, raster.nodata,
                                                   str(arr.dtype), self.tile_size, compression_level, str(output_path),
                                                   rank, world, engine=eng)
            self.frames = [SpatialFrame(f["frame_id"], tuple(f["bbox"]),
                                        _Window(f["window"]["col_off"], f["window"]["row_off"], f["window"]["width"], f["window"]["height"]),
                                        f["byte_offset"], f["byte_size"]) for f in index["frames"]]
            return SpatialIndex(self.frames, raster.crs, raster.transform)
        host = torch.from_numpy(np.ascontiguousarray(arr).view(np.uint8).reshape(-1)).view(TORCH_DTYPES[str(arr.dtype)]).reshape(arr.shape)
        index, headers, enc = build_streaming_container(host, raster.transform, raster.crs, raster.nodata, str(arr.dtype),
                                                        self.tile_size, compression_level, engine=eng)
        payload = enc.payload.cpu().numpy()
        write_streaming_container(output_path, index, headers, payload, enc.offsets, enc.sizes)
        self.frames = [SpatialFrame(f["frame_id"], tuple(f["bbox"]),
                                    _Window(f["window"]["col_off"], f["window"]["row_off"], f["window"]["width"], f["window"]["height"]),
                                    f["byte_offset"], f["byte_size"]) for f in index["frames"]]
        return SpatialIndex(self.frames, raster.crs, raster.transform)

    # ---- legacy --spatial format ----------------------------------------------------------
    def encode_spatial_flac(self, tiff_path: Path, flac_path: Path, compression_level: int = 5,
                            enable_streaming: bool = True) -> SpatialIndex:
        """Concatenated per-tile streams + gz/b64 index in stream 0's tags (spatial_encoder.py:155-258).

        Unlike the reference, byte offsets are recorded AFTER stream 0's tags are in place, so they
        are valid (SURVEY Q6), and each tile stream carries its own min/max tags.
        """
        import torch
        from .converter import metadata_tags
        from .engine import TORCH_DTYPES, default_engine

        raster = read_geotiff(tiff_path)
        arr = raster.data
        eng = default_engine()
        dev = torch.from_numpy(np.ascontiguousarray(arr).view(np.uint8).reshape(-1)).to(eng.device)
        dev = dev.view(TORCH_DTYPES[str(arr.dtype)]).reshape(arr.shape)
        index, headers, enc = build_streaming_container(dev, raster.transform, raster.crs, raster.nodata, str(arr.dtype),
                                                        self.tile_size, compression_level, engine=eng)
        payload = enc.payload.cpu().numpy()
        frames_meta = index["frames"]

        def make_index_tag(first_header_len):
            shift = first_header_len - len(headers[0])
            fl = []
            for f in frames_meta:
                w = f["window"]
                fl.append({"frame_id": f["frame_id"], "bbox": f["bbox"],
                           "window": {"row_off": w["row_off"], "col_off": w["col_off"], "height": w["height"], "width": w["width"]},
                           "byte_offset": f["byte_offset"] + (shift if f["frame_id"] > 0 else 0),
                           "byte_size": f["byte_size"] + (shift if f["frame_id"] == 0 else 0)})
            d = {"crs": str(raster.crs), "transform": index["transform"], "frames": fl}
            raw = json.dumps(d).encode("utf-8")
            return base64.b64encode(gzip.compress(raw, mtime=0)).decode("ascii"), fl, len(raw)

        hdr0 = flacfmt.parse_header(headers[0])
        base_tags = {k: v[0] for k, v in hdr0.tags.items()}
        first_len = len(headers[0])
        for _ in range(8):       # header length depends on the index text: iterate to a fixed point
            tag, fl, rawlen = make_index_tag(first_len)
            tags = dict(base_tags)
            tags.update({"GEOSPATIAL_SPATIAL_TILING": "True", "GEOSPATIAL_SPATIAL_INDEX": tag,
                         "GEOSPATIAL_SPATIAL_INDEX_COMPRESSED": "gzip+base64",
                         "GEOSPATIAL_SPATIAL_INDEX_ORIGINAL_SIZE": str(rawlen)})
            new0 = flacfmt.build_header(hdr0.streaminfo, tags)
            if len(new0) == first_len:
                break
            first_len = len(new0)
        headers = [new0] + headers[1:]
        mv = memoryview(payload)
        with open(flac_path, "wb") as f:
            for h, o, s in zip(headers, enc.offsets, enc.sizes):
                f.write(h)
                f.write(mv[int(o):int(o) + int(s)])
        self.frames = [SpatialFrame(d["frame_id"], tuple(d["bbox"]),
                                    _Window(d["window"]["col_off"], d["window"]["row_off"], d["window"]["width"], d["window"]["height"]),
                                    d["byte_offset"], d["byte_size"]) for d in fl]
        return SpatialIndex(self.frames, raster.crs, raster.transform)


def _intersects(bbox, fb) -> bool:
    """Strict intersection test of cli.py:273-278."""
    return bbox[0] < fb[2] and bbox[2] > fb[0] and bbox[1] < fb[3] and bbox[3] > fb[1]


class SpatialFLACStreamer:
    """Reads tiles from a streaming container or a legacy --spatial file (local path or URL)."""

    def __init__(self, flac_path_or_url):
        self.source = str(flac_path_or_url)
        self.logger = logging.getLogger("flac_raster.spatial_encoder")
        self.is_url = self.source.startswith(("http://", "https://", "s3://", "gs://", "az://"))
        self.flac_path = None if self.is_url else Path(self.source)
        self.metadata: Optional[Dict] = None      # streaming container index
        self.header_size = 0
        self.spatial_index: Optional[SpatialIndex] = None
        self.legacy_tags: Dict[str, List[str]] = {}
        self._load_spatial_index()

    # ---- byte access ---------------------------------------------------------------------
    def _read_range(self, start: int, end_inclusive: int) -> bytes:
        if self.is_url:
            from .remote import RemoteFile

            return RemoteFile(self.source).read_range(start, end_inclusive)
        with open(self.flac_path, "rb") as f:
            f.seek(start)
            return f.read(end_inclusive - start + 1)

    def _load_spatial_index(self):
        if not self.is_url and not self.flac_path.exists():
            raise FileNotFoundError(f"FLAC file not found: {self.flac_path}")
        head = self._read_range(0, 3)
        if head == b"fLaC":
            self._load_legacy_index()
            return
        # streaming container: [u32 BE][JSON] (cli.py:224-235)
        index_size = struct.unpack(">I", head)[0]
        self.metadata = json.loads(self._read_range(4, 3 + index_size).decode("utf-8"))
        self.header_size = 4 + index_size
        frames = [SpatialFrame(f["frame_id"], tuple(f["bbox"]),
                               _Window(f["window"]["col_off"], f["window"]["row_off"], f["window"]["width"], f["window"]["height"]),
                               f["byte_offset"], f["byte_size"]) for f in self.metadata["frames"]]
        self.spatial_index = SpatialIndex(frames, self.metadata.get("crs"), self.metadata.get("transform"))

    def _load_legacy_index(self):
        """Index from the first stream's VORBIS tags (spatial_encoder.py:434-515).

        The reference ALWAYS stores GEOSPATIAL_SPATIAL_INDEX as base64(gzip(json)) and writes no marker tag
        (spatial_encoder.py:366-375, read back at :464-474), so that is tried first; plain JSON is accepted too.
        Reference-written files carry STALE byte offsets: they are recorded while the tile streams are appended
        (:238-241) and mutagen then grows stream 0 by its tags and padding (:251), moving every later stream
        (SURVEY Q6).  An entry that does not point at a "fLaC" marker triggers a rescan for the real stream starts."""
        blob = self._read_range(0, (1 << 20) - 1)           # same first-MiB probe as the reference
        hdr = flacfmt.parse_header(blob)
        tag = hdr.tags.get("GEOSPATIAL_SPATIAL_INDEX")
        if not tag:
            raise ValueError("No spatial index found in FLAC metadata")
        raw = tag[0]
        try:
            raw = gzip.decompress(base64.b64decode(raw.encode("ascii"), validate=True)).decode("utf-8")
        except (ValueError, OSError, EOFError, UnicodeError):
            pass                                            # not base64+gzip: plain JSON text
        d = json.loads(raw)
        frames = [SpatialFrame(f["frame_id"], tuple(f["bbox"]),
                               _Window(f["window"]["col_off"], f["window"]["row_off"], f["window"]["width"], f["window"]["height"]),
                               f["byte_offset"], f["byte_size"]) for f in d["frames"]]
        self.spatial_index = SpatialIndex(frames, d.get("crs"), d.get("transform"))
        self.header_size = 0
        self.legacy_tags = hdr.tags                         # global metadata: the tile streams carry none
        self._fix_stale_legacy_offsets(blob)

    @staticmethod
    def _stream_starts(data) -> List[int]:
        """Positions of 'fLaC' markers that are followed by a STREAMINFO block header (type 0, length 34): eight
        fixed bytes, so a chance hit inside compressed audio is a 2^-64 event per position."""
        out, pos, mv = [], 0, bytes(data) if not isinstance(data, (bytes, bytearray)) else data
        while True:
            pos = mv.find(b"fLaC", pos)
            if pos < 0:
                return out
            if mv[pos + 4:pos + 8] in (b"\x00\x00\x00\x22", b"\x80\x00\x00\x22"):
                out.append(pos)
            pos += 4

    def _fix_stale_legacy_offsets(self, first_mib: bytes):
        frames = self.spatial_index.frames
        if not frames:
            return

        def marker_at(off: int) -> bool:
            if off + 4 <= len(first_mib):
                return first_mib[off:off + 4] == b"fLaC"
            try:
                return self._read_range(off, off + 3) == b"fLaC"
            except Exception:  # noqa: BLE001  (offset beyond the end of the file)
                return False

        if all(marker_at(f.byte_offset) for f in frames):
            return
        # stale: locate the real stream starts (whole file: legacy files are small, one stream per tile)
        if self.is_url:
            from .remote import RemoteFile
            data = RemoteFile(self.source).read_all()
        else:
            data = self.flac_path.read_bytes()
        starts = self._stream_starts(data)
        order = sorted(range(len(frames)), key=lambda i: frames[i].byte_offset)
        if len(starts) == len(frames):
            ends = starts[1:] + [len(data)]
            for rank_, i in enumerate(order):
                frames[i].byte_offset, frames[i].byte_size = starts[rank_], ends[rank_] - starts[rank_]
        elif len(starts) >= 2:
            # the only thing that moved is stream 0's length: shift every later stream by that growth
            delta = starts[1] - frames[order[0]].byte_size - frames[order[0]].byte_offset
            for rank_, i in enumerate(order):
                if rank_ == 0:
                    frames[i].byte_size += delta
                else:
                    frames[i].byte_offset += delta
            if not all(data[f.byte_offset:f.byte_offset + 4] == b"fLaC" for f in frames):
                raise ValueError("legacy spatial FLAC: byte offsets do not point at FLAC streams and cannot be repaired")
        else:
            raise ValueError("legacy spatial FLAC: byte offsets do not point at FLAC streams and cannot be repaired")
        self.logger.info("legacy spatial FLAC: stale byte offsets corrected from the stream markers")
        self.spatial_index.total_bytes = sum(f.byte_size for f in frames)

    def _legacy_tile_metadata(self, frame: SpatialFrame, streaminfo) -> Dict:
        """Per-tile metadata of a legacy file: the tile streams have no tags of their own, only stream 0 carries the
        GLOBAL ones (spatial_encoder.py:338-356; the per-tile normalisation parameters were discarded at :222,
        SURVEY Q6), so a tile is denormalised with the global min/max -- all the information the file holds."""
        g = parse_metadata_tags(self.legacy_tags) or {}
        w, h = int(frame.window.width), int(frame.window.height)
        tr = g.get("transform") or None
        md = {
            "crs": g.get("crs", ""), "width": w, "height": h, "count": int(g.get("count", streaminfo.channels)),
            "dtype": g.get("dtype", "int16" if streaminfo.bits_per_sample == 16 else "int32"),
            "nodata": g.get("nodata"), "data_min": float(g.get("data_min", 0.0)), "data_max": float(g.get("data_max", 0.0)),
            "transform": (list(window_transform(tuple(tr[:6]), int(frame.window.col_off), int(frame.window.row_off))) + [0.0, 0.0, 1.0]) if tr else [],
            "bounds": list(frame.bbox), "spatial_tiling": True,
        }
        return md

    # ---- reference methods (byte ranges only, spatial_encoder.py:517-567) ----------------------
    def get_byte_ranges_for_bbox(self, bbox) -> List[Tuple[int, int]]:
        frames = self.spatial_index.query_bbox(bbox)
        ranges = sorted((self.header_size + f.byte_offset, self.header_size + f.byte_offset + f.byte_size - 1) for f in frames)
        merged: List[Tuple[int, int]] = []
        for s, e in ranges:
            if merged and s <= merged[-1][1] + 1:
                merged[-1] = (merged[-1][0], max(merged[-1][1], e))
            else:
                merged.append((s, e))
        return merged

    def stream_bbox_data(self, bbox) -> bytes:
        return b"".join(self._read_range(s, e) for s, e in self.get_byte_ranges_for_bbox(bbox))

    # ---- README API: decode on the GPU ----------------------------------------------------------
    def _read_tiles_pinned(self, frames: List[SpatialFrame], to_device: bool = False, slot: Optional[int] = None):
        """Local file: read the (merged) byte ranges of the tiles straight into ONE pinned staging buffer -- no bytes object
        per range and no second host copy before the H2D transfer.  Big queries are read by several threads (pread releases
        the GIL; one thread moves ~8 GB/s out of the page cache).  Returns (pinned uint8 tensor, bytes used, start of
        every tile in it).  to_device: every piece is also sent to the engine's "dec_data" device buffer as soon as it has
        been read (H2D overlaps the reads of the following pieces); the 4th result is then that device tensor.
        slot: use the staging / device buffers of that number (the grouped pipeline of _decode alternates between two)."""
        import torch
        from .engine import default_engine

        eng = default_engine()
        order = sorted(range(len(frames)), key=lambda i: frames[i].byte_offset)
        total = sum(f.byte_size for f in frames)
        sfx = "" if slot is None else str(int(slot))
        stage = eng._pinned("dec_stage" + sfx, total + 64)
        view = memoryview(stage.numpy())
        starts = np.zeros(len(frames), dtype=np.int64)
        jobs = []                                   # (file offset, position in stage, length)
        pos = 0
        i = 0
        while i < len(order):
            j = i
            start = frames[order[i]].byte_offset
            end = start + frames[order[i]].byte_size
            while j + 1 < len(order) and frames[order[j + 1]].byte_offset == end:
                j += 1
                end += frames[order[j]].byte_size
            for k in range(i, j + 1):
                f = frames[order[k]]
                starts[order[k]] = pos + (f.byte_offset - start)
            want = end - start
            piece = (8 << 20) if self.is_url else (int(os.environ.get("FRB_READ_PIECE_MB", "32")) << 20)
            for o in range(0, want, piece):
                jobs.append((self.header_size + start + o, pos + o, min(piece, want - o)))
            pos += want
            i = j + 1
        fd = None if self.is_url else os.open(self.flac_path, os.O_RDONLY)
        try:
            if self.is_url:
                # remote container: the same pieces as HTTP / object-store range requests (remote.py:137-177), several in
                # flight; each lands in its slice of the pinned buffer and goes on to the GPU while the others are fetched
                from .remote import RemoteFile
                rf = RemoteFile(self.source)

                def read(job):
                    off, p, n = job
                    if rf.read_range_into(off, off + n - 1, view[p:p + n]) != n:
                        raise ValueError("streaming container is shorter than its index says")
            else:
                def read(job):
                    off, p, n = job
                    got = 0
                    while got < n:
                        r = os.preadv(fd, [view[p + got:p + n]], off + got)
                        if r <= 0:
                            raise ValueError("streaming container is shorter than its index says")
                        got += r

            data = None
            if to_device:
                data = eng._buf("dec_data" + sfx, pos + 64)[:pos + 64]

            def send(job):
                if data is not None:
                    _, p, n = job
                    data[p:p + n].copy_(stage[p:p + n], non_blocking=True)

            if len(jobs) > 2:
                from concurrent.futures import ThreadPoolExecutor
                with ThreadPoolExecutor(min(int(os.environ.get("FRB_READ_THREADS", "8")), len(jobs))) as ex:
                    for job, _ in zip(jobs, ex.map(read, jobs)):       # results come back in submission order
                        send(job)
            else:
                for job in jobs:
                    read(job)
                    send(job)
            if data is not None:
                stage[pos:pos + 64].zero_()
                data[pos:pos + 64].copy_(stage[pos:pos + 64], non_blocking=True)
        finally:
            if fd is not None:
                os.close(fd)
        return (stage, pos, starts, data) if to_device else (stage, pos, starts)

    def _tile_meta_from_index(self, f: SpatialFrame, rec) -> Dict:
        """A tile's metadata dict without parsing its tags in Python: the numbers come from frb_parse_tile_headers, the
        georeferencing from the container index with the arithmetic the writer used (build_streaming_container), so the
        result equals parse_metadata_tags on the tile's own tags."""
        from .converter import _DTYPE_NAMES, affine9
        w, h = int(rec["width"]), int(rec["height"])
        tr = self.metadata.get("transform") or None
        if tr:
            tt = window_transform(tuple(tr[:6]), int(f.window.col_off), int(f.window.row_off))
            transform = affine9(tt)
        else:
            tt, transform = (1.0, 0.0, 0.0, 0.0, -1.0, 0.0), None
        left, top = tt[2], tt[5]
        return {
            "crs": self.metadata.get("crs", ""), "width": w, "height": h, "count": int(rec["count"]),
            "dtype": _DTYPE_NAMES[int(rec["dtype"])],
            "nodata": float(rec["nodata"]) if int(rec["flags"]) & 2 else None,
            "data_min": float(rec["data_min"]), "data_max": float(rec["data_max"]),
            "transform": transform, "bounds": {"left": left, "bottom": top + h * tt[4], "right": left + w * tt[0], "top": top},
            "spatial_tiling": False,
        }

    # a big query is cut into groups of about this many compressed bytes (see _decode_grouped)
    GROUP_BYTES = 160 << 20

    def _decode_grouped(self, frames: List[SpatialFrame]):
        """Big queries (BASELINE config 5: 4096 tiles, 1.5 GB of frames in, 2.1 GB of pixels out): the tiles are cut into
        groups and the groups are pipelined -- a background thread reads group g+1 and sends it to the device on its own
        stream while this thread decodes group g and brings its pixels back, so the two PCIe directions run at the same
        time instead of one after the other (one batch: 27 ms up, THEN 40 ms down).  Returns None when a group does not
        qualify for the fast path (the caller then takes the general one)."""
        import torch
        from concurrent.futures import ThreadPoolExecutor
        from .engine import default_engine

        eng = default_engine()
        total = sum(f.byte_size for f in frames)
        n_groups = max(2, min(16, (total + self.GROUP_BYTES - 1) // self.GROUP_BYTES))
        per = (len(frames) + n_groups - 1) // n_groups
        groups = [frames[i:i + per] for i in range(0, len(frames), per)]
        with torch.cuda.device(eng.device):
            if not hasattr(self, "_h2d_stream"):
                self._h2d_stream = torch.cuda.Stream()
            s_h2d = self._h2d_stream
            main = torch.cuda.current_stream()

            def fetch(g):
                with torch.cuda.device(eng.device), torch.cuda.stream(s_h2d):
                    got = self._read_tiles_pinned(groups[g], to_device=True, slot=g & 1)
                    ev = torch.cuda.Event()
                    ev.record(s_h2d)
                return got, ev

            out: List = []
            s_h2d.wait_stream(main)
            with ThreadPoolExecutor(1) as bg:
                fut = bg.submit(fetch, 0)
                for g, part in enumerate(groups):
                    (stage, nbytes, starts, data), ev = fut.result()
                    if g + 1 < len(groups):
                        fut = bg.submit(fetch, g + 1)       # slot (g+1)&1: its previous user (group g-1) is done and synchronised
                    main.wait_event(ev)
                    sizes = np.fromiter((f.byte_size for f in part), dtype=np.int64, count=len(part))
                    metas: List[Dict] = []

                    def build_metas(recs, part=part, metas=metas):
                        for f, rec in zip(part, recs):
                            meta = self._tile_meta_from_index(f, rec)
                            meta.update({"frame_id": f.frame_id, "bbox": list(f.bbox),
                                         "window": {"col_off": f.window.col_off, "row_off": f.window.row_off,
                                                    "width": f.window.width, "height": f.window.height},
                                         "byte_offset": f.byte_offset, "byte_size": f.byte_size})
                            metas.append(meta)

                    res = decode_staged_tiles(stage, nbytes, starts, sizes, data=data, while_copying=build_metas)
                    if res is None:
                        if g + 1 < len(groups):
                            fut.result()                    # let the read in flight finish before its buffers are reused
                        return None
                    out.extend(zip(res[0], metas))
        return out

    def _decode(self, frames: List[SpatialFrame]):
        fast = self.metadata is not None and os.environ.get("FRB_SLOW_TILE_PARSE") != "1"
        if fast and not self.is_url and len(frames) >= 64 and os.environ.get("FRB_NO_GROUPED_DECODE") != "1" \
                and sum(f.byte_size for f in frames) >= 2 * self.GROUP_BYTES:
            res = self._decode_grouped(frames)
            if res is not None:
                return res
        if fast:
            # streaming container written with per-tile tags: the pieces go to the GPU as they arrive, metadata walk and index
            # gather in C, one batched decode; the metadata dicts are put together while the pixels travel back to the host
            stage, nbytes, starts, data = self._read_tiles_pinned(frames, to_device=True)
            sizes = np.fromiter((f.byte_size for f in frames), dtype=np.int64, count=len(frames))
            metas: List[Dict] = []

            def build_metas(recs):
                for f, rec in zip(frames, recs):
                    meta = self._tile_meta_from_index(f, rec)
                    meta.update({"frame_id": f.frame_id, "bbox": list(f.bbox),
                                 "window": {"col_off": f.window.col_off, "row_off": f.window.row_off,
                                            "width": f.window.width, "height": f.window.height},
                                 "byte_offset": f.byte_offset, "byte_size": f.byte_size})
                    metas.append(meta)

            res = decode_staged_tiles(stage, nbytes, starts, sizes, data=data, while_copying=build_metas)
            if res is not None:
                return list(zip(res[0], metas))
        else:
            stage, nbytes, starts = self._read_tiles_pinned(frames)
        view = memoryview(stage.numpy())
        blobs = [view[int(starts[i]):int(starts[i]) + frames[i].byte_size] for i in range(len(frames))]
        staged = (stage, nbytes, starts)
        headers = [flacfmt.parse_header(b) for b in blobs]
        metas = []
        legacy = self.metadata is None
        for f, h in zip(frames, headers):
            md = parse_metadata_tags(h.tags)
            if legacy and not (md and int(md.get("width", 0)) * int(md.get("height", 0)) == int(f.window.width) * int(f.window.height)):
                # reference-written legacy file: no per-tile tags (stream 0 holds the GLOBAL ones)
                md = self._legacy_tile_metadata(f, h.streaminfo)
            if not md:
                raise ValueError("No metadata found in FLAC file or sidecar file")
            metas.append(md)
        arrays = decode_tile_blobs(blobs, headers, metas, staged=staged)
        out = []
        for f, a, md in zip(frames, arrays, metas):
            meta = dict(md)
            meta.update({"frame_id": f.frame_id, "bbox": list(f.bbox),
                         "window": {"col_off": f.window.col_off, "row_off": f.window.row_off,
                                    "width": f.window.width, "height": f.window.height},
                         "byte_offset": f.byte_offset, "byte_size": f.byte_size})
            out.append((a, meta))
        return out

    def get_tile_by_id(self, tile_id: int):
        """README.md:200-201 -> (tile_data (bands,h,w), metadata).  cli.py:243-247 semantics."""
        frame = next((f for f in self.spatial_index.frames if f.frame_id == tile_id), None)
        if frame is None:
            raise KeyError(f"Tile ID {tile_id} not found")
        return self._decode([frame])[0]

    def get_tiles_by_bbox(self, xmin, ymin, xmax, ymax, shard=None):
        """README.md:202 -> list of (tile_data, metadata) for ALL intersecting tiles (one batched decode).

        Multi-GPU (one process per GPU): the intersecting tiles are split over the ranks in contiguous blocks (balanced by pixel count) and each
        rank fetches and decodes only its own block -- no collective (SURVEY 8e); the call returns this rank's tiles.
        `shard`: (rank, world) to split explicitly, None = the initialised torch.distributed group (or no split),
        False = never split."""
        frames = [f for f in self.spatial_index.frames if _intersects((xmin, ymin, xmax, ymax), f.bbox)]
        if shard is None:
            from .distributed import current_rank_world
            shard = current_rank_world()
        if shard and shard[1] > 1:
            from .distributed import shard_ranges_weighted
            a, b = shard_ranges_weighted([f.window.width * f.window.height for f in frames], int(shard[1]))[int(shard[0])]
            frames = frames[a:b]
        if not frames:
            return []
        return self._decode(frames)

    def read_bbox(self, xmin, ymin, xmax, ymax):
        """One mosaic of the pixels inside a bbox -> ((bands, h, w) array in the original dtype, metadata with its window,
        transform and bounds).  The pixel window floors the bbox's near edges and ceils its far edges, clipped to the raster
        (ValueError when the bbox misses it).  The tiles that intersect the window are fetched like get_tiles_by_bbox, and one
        decode launch writes each tile's visible part straight into the mosaic, decoding only the frames that cover it."""
        import torch
        from . import _native as nat
        from .converter import _raise_for_status, affine9
        from .engine import TORCH_DTYPES, bbox_to_window, default_engine

        frames = self.spatial_index.frames
        H = max(int(f.window.row_off) + int(f.window.height) for f in frames)
        W = max(int(f.window.col_off) + int(f.window.width) for f in frames)
        tr = (self.metadata or {}).get("transform") or self.spatial_index.transform or None
        t6 = tuple(float(v) for v in tr[:6]) if tr else (1.0, 0.0, 0.0, 0.0, -1.0, 0.0)     # _tile_bbox's default
        col0, row0, width, height = bbox_to_window(t6, W, H, (xmin, ymin, xmax, ymax))
        sel = [f for f in frames if int(f.window.col_off) < col0 + width and int(f.window.col_off) + int(f.window.width) > col0
               and int(f.window.row_off) < row0 + height and int(f.window.row_off) + int(f.window.height) > row0]
        stage, nbytes, starts = self._read_tiles_pinned(sel)
        view = memoryview(stage.numpy())
        n = len(sel)
        tiles = np.zeros(n, dtype=nat.TILE_DTYPE)
        offs, lens = np.zeros(n, dtype=np.int64), np.zeros(n, dtype=np.int64)
        rates = np.zeros(n, dtype=np.uint32)
        minmax = np.zeros((n, 2), dtype=np.float64)
        fb, sb = [], []
        md0 = None
        for i, f in enumerate(sel):
            blob = view[int(starts[i]):int(starts[i]) + f.byte_size]
            h = flacfmt.parse_header(blob)
            md = parse_metadata_tags(h.tags)
            if self.metadata is None and not (md and int(md.get("width", 0)) * int(md.get("height", 0)) == int(f.window.width) * int(f.window.height)):
                md = self._legacy_tile_metadata(f, h.streaminfo)        # reference-written legacy file (see _decode)
            if not md:
                raise ValueError("No metadata found in FLAC file or sidecar file")
            si = h.streaminfo
            if md0 is None:
                md0, si0 = md, si
            elif (si.channels, si.bits_per_sample, si.max_blocksize, md["dtype"]) != (si0.channels, si0.bits_per_sample, si0.max_blocksize, md0["dtype"]):
                raise ValueError("tiles of one mosaic must share channels, bits per sample, blocksize and dtype")
            if int(md["width"]) != int(f.window.width) or int(md["height"]) != int(f.window.height):
                raise ValueError(f"tile {f.frame_id}: its tags do not match its window in the index")
            tiles[i] = (int(f.window.row_off), int(f.window.col_off), int(f.window.height), int(f.window.width))
            offs[i], lens[i] = int(starts[i]) + h.first_frame_offset, f.byte_size - h.first_frame_offset
            rates[i] = si.sample_rate
            minmax[i] = (md["data_min"], md["data_max"])
            if fb is not None:
                blk = h.applications.get(flacfmt.SEEK_INDEX_ID)
                nf = (int(f.window.width) * int(f.window.height) + si.max_blocksize - 1) // si.max_blocksize
                got = flacfmt.unpack_seek_index(blk, si.channels, si.max_blocksize, nf) if blk else None
                if got is None:
                    fb = sb = None
                else:
                    fb.append(got[0])
                    sb.append(got[1])
        bands, bps, blocksize = si0.channels, si0.bits_per_sample, si0.max_blocksize
        index = (np.concatenate(fb), np.concatenate(sb) if bands > 1 else None) if fb else None
        scale = 32767.0 if bps == 16 else 8388607.0                  # decode default by audio width (converter.py:220-229)
        dtype = np.dtype(md0["dtype"])
        eng = default_engine()
        stage[nbytes:nbytes + 64].zero_()
        data = eng._buf("dec_data", nbytes + 64)[:nbytes + 64]
        data.copy_(stage[:nbytes + 64], non_blocking=True)
        out = torch.empty((bands, height, width), dtype=TORCH_DTYPES[str(dtype)], device=eng.device)
        status = eng.decode_window(data, offs, lens, tiles, rates, minmax, scale, (col0, row0, width, height), out, bps, blocksize,
                                   index=index)
        _raise_for_status(status)
        wt = window_transform(t6, col0, row0)
        left, top = wt[2], wt[5]
        meta = {
            "crs": (self.metadata or {}).get("crs", md0.get("crs", "")), "width": width, "height": height, "count": bands,
            "dtype": str(dtype), "nodata": md0.get("nodata"), "transform": affine9(wt) if tr else None,
            "bounds": {"left": left, "bottom": top + height * wt[4], "right": left + width * wt[0], "top": top},
            "window": {"col_off": col0, "row_off": row0, "width": width, "height": height},
            "tiles": [f.frame_id for f in sel], "frames_decoded": int(status[nat.ST_FRAMES_DECODED]),
        }
        return out.cpu().numpy(), meta

    def get_center_tile(self):
        """cli.py:250-262: tile whose centroid is nearest the centroid of the union of bboxes."""
        fr = self.spatial_index.frames
        cx = (min(f.bbox[0] for f in fr) + max(f.bbox[2] for f in fr)) / 2
        cy = (min(f.bbox[1] for f in fr) + max(f.bbox[3] for f in fr)) / 2
        best = min(fr, key=lambda f: ((f.bbox[0] + f.bbox[2]) / 2 - cx) ** 2 + ((f.bbox[1] + f.bbox[3]) / 2 - cy) ** 2)
        return self._decode([best])[0]
