"""Batch device API: tiles of a device-resident raster <-> FLAC frames on the GPU.

This is the fast path behind SpatialFLACEncoder.encode(streaming=True) and
SpatialFLACStreamer.get_tiles_by_bbox: the reference's serial per-tile loop
(cli.py:553-622: window read -> temp TIFF -> tiff_to_flac -> bytes) becomes
four batched launches over all tiles at once:
  minmax_tiles -> normalize_tiles -> encode_analyse -> encode_emit
and the reverse (extract, cli.py:297-315, looped) becomes
  sync_scan -> decode_frames -> crc16 -> denormalize_tiles.
PyTorch is used only for device buffers and streams.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _native as nat
from .normalization import audio_params_for, sample_rates_for_pixel_counts

TORCH_DTYPES = {
    "uint8": torch.uint8, "int8": torch.int8, "uint16": torch.uint16, "int16": torch.int16,
    "uint32": torch.uint32, "int32": torch.int32, "float32": torch.float32, "float64": torch.float64,
}


def tile_grid(height: int, width: int, tile_size: int) -> np.ndarray:
    """Row-major tile windows exactly as cli.py:553-556 enumerates them (edge tiles are smaller)."""
    rows = range(0, height, tile_size)
    cols = range(0, width, tile_size)
    t = np.zeros(len(rows) * len(cols), dtype=nat.TILE_DTYPE)
    i = 0
    for r in rows:
        for c in cols:
            t[i] = (r, c, min(tile_size, height - r), min(tile_size, width - c))
            i += 1
    return t


def _check_tile_sizes(npx: np.ndarray) -> None:
    """The mapping kernels index a tile's pixels with 32 bits (h * w, k * blocksize): reject what would wrap instead of
    coding garbage.  The reference has no such limit (numpy), but pyflac's 32-bit frame counters end well below it."""
    if len(npx) and int(npx.max()) >= 1 << 32:
        raise ValueError(f"a tile of {int(npx.max())} pixels exceeds the 2^32 - 1 pixels one tile may hold; use a smaller tile_size")


RUN_DTYPE = np.dtype([("tile", "<i8"), ("first_frame", "<i8"), ("n_frames", "<i8"), ("byte_offset", "<i8"), ("byte_length", "<i8")])


def window_frames(tiles: np.ndarray, window, blocksize: int, frame_bytes=None) -> np.ndarray:
    """The frames a pixel window needs: one run per tile that intersects it (RUN_DTYPE records, in tile order).

    tiles: TILE_DTYPE records in image coordinates; window: (col_off, row_off, width, height) in image coordinates.  A tile's
    samples are its pixels in row-major order, so the visible ones lie between sample y0*w + x0 (first visible row, first
    visible column) and (y1-1)*w + x1-1; the run is every frame from the one holding the first to the one holding the last.
    frame_bytes (optional): per tile, the byte size of each of its frames (the "frbI" seek index); byte_offset / byte_length
    of the run then give where its frames sit behind the stream's first frame.  Without it they are -1."""
    col0, row0, width, height = (int(v) for v in window)
    out = []
    for i, t in enumerate(tiles):
        r, c, h, w = int(t["row_off"]), int(t["col_off"]), int(t["h"]), int(t["w"])
        y0, y1 = max(row0 - r, 0), min(row0 + height - r, h)
        x0, x1 = max(col0 - c, 0), min(col0 + width - c, w)
        if y0 >= y1 or x0 >= x1:
            continue
        f0 = (y0 * w + x0) // blocksize
        f1 = ((y1 - 1) * w + x1 - 1) // blocksize + 1
        off = length = -1
        if frame_bytes is not None:
            fb = np.asarray(frame_bytes[i], dtype=np.int64)
            off, length = int(fb[:f0].sum()), int(fb[f0:f1].sum())
        out.append((i, f0, f1 - f0, off, length))
    return np.array(out, dtype=RUN_DTYPE)


def bbox_to_window(transform, width: int, height: int, bbox) -> Tuple[int, int, int, int]:
    """(xmin, ymin, xmax, ymax) in the raster's coordinates -> pixel window (col_off, row_off, width, height): the offsets
    are floored, the far edges ceiled, and the result clipped to the raster.  ValueError when nothing is left."""
    import math
    a, b, c, d, e, f = (float(v) for v in transform[:6])
    if b != 0.0 or d != 0.0 or a == 0.0 or e == 0.0:
        raise ValueError("bbox reads need a north-up transform without rotation")
    xmin, ymin, xmax, ymax = (float(v) for v in bbox)
    cx = sorted(((xmin - c) / a, (xmax - c) / a))
    ry = sorted(((ymin - f) / e, (ymax - f) / e))
    c0, c1 = max(math.floor(cx[0]), 0), min(math.ceil(cx[1]), int(width))
    r0, r1 = max(math.floor(ry[0]), 0), min(math.ceil(ry[1]), int(height))
    if c1 <= c0 or r1 <= r0:
        raise ValueError(f"bbox {tuple(bbox)} does not intersect the raster")
    return c0, r0, c1 - c0, r1 - r0


def _stream_table(byte_offsets, byte_lengths, n_samples, sample_rates, channels: int, blocksize: int):
    """Whole streams as DECODE_STREAM_DTYPE records, and where each stream's frames start in the batch (n_streams + 1
    entries, the last one the batch's frame count).  frame_base and audio_base are the exclusive scans of the streams'
    frame and sample counts."""
    n_samples = np.asarray(n_samples, dtype=np.int64)
    fstart = np.zeros(len(n_samples) + 1, dtype=np.int64)
    np.cumsum((n_samples + blocksize - 1) // blocksize, out=fstart[1:])
    st = np.zeros(len(n_samples), dtype=nat.DECODE_STREAM_DTYPE)
    st["byte_offset"] = byte_offsets
    st["byte_length"] = byte_lengths
    st["n_samples"] = n_samples
    st["audio_base"][1:] = np.cumsum(n_samples[:-1] * channels)
    st["sample_rate"] = sample_rates
    st["frame_base"] = fstart[:-1]
    return st, fstart


def _index_fits(index, total_frames: int, channels: int) -> bool:
    """Whether index = (frame_bytes, sub_bitoff) has the shape of the seek index of `total_frames` frames: one frame size per
    frame and, for more than one channel, one subframe bit offset per subframe (sub_bitoff is not used for one channel)."""
    def size(x):
        return -1 if x is None else x.numel() if isinstance(x, torch.Tensor) else np.size(x)

    return index is not None and size(index[0]) == total_frames and (channels == 1 or size(index[1]) == total_frames * channels)


def _fused_default(bps: int, dtype: str, scale: float) -> bool:
    """Whether decode_tiles and decode_window denormalise inside the decode launch when the caller does not say.  The fused
    launch pays off where the pixel mapping is the exact integer form (8/16-bit rasters behind 16-bit audio).  Wider dtypes
    need the fp64 formula per sample, which is cheaper in the bandwidth-bound mapping kernel than inside the issue-bound
    decode kernel (C4 float32: 129 vs 97 GSamples/s), so they stay two-step."""
    return bps == 16 and dtype in ("uint8", "int8", "uint16", "int16") and float(scale) == 32767.0


def decode_ladder(attempt, has_index: bool, allow_scan: bool, where: str):
    """The decodes every device decode call tries, which decide what a damaged, foreign or wrongly indexed stream turns into.
    attempt(max_order, use_index) decodes once and returns the host status words; the status words of the last attempt are
    returned.  Order: seek index at LPC order <= 12, index at order 32, sync scan at 12, scan at 32.  Index attempts need an
    index, and damage under it drops it: the index does not describe the bytes, so decode again by scanning -- unless
    `allow_scan` is False (the bytes hold only some frames of each stream), where the damaged words come back for the caller
    to judge.  Rejected tiles raise NativeError: they are the caller's error, not the stream's."""
    status = None
    for max_order, use_index in ((12, True), (32, True), (12, False), (32, False)):
        if use_index and not has_index:
            continue
        if not use_index and not allow_scan:
            break
        status = attempt(max_order, use_index)
        if status[nat.ST_TILES_REJECTED]:
            raise nat.NativeError(nat.ERR_INVALID_ARG, where, f"{int(status[nat.ST_TILES_REJECTED])} tile(s) do not hold as many "
                                  "pixels as their stream has samples, or lie outside the raster")
        if use_index and nat.status_damaged(status):
            has_index = False
            continue
        if status[nat.ST_LPC_ORDER_ABOVE_12] == 0:
            break
    return status


def _stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def _dev_bytes(n: int, device) -> torch.Tensor:
    return torch.empty(max(int(n), 1), dtype=torch.uint8, device=device)


@dataclass
class EncodedTiles:
    """Frames of a batch of tiles, still on the device."""
    payload: torch.Tensor          # uint8, concatenated frame payloads (no metadata blocks)
    offsets: np.ndarray            # int64 [n_tiles] start of each tile's frames in payload
    sizes: np.ndarray              # int64 [n_tiles] bytes of frames per tile
    minmax: np.ndarray             # float64 [n_tiles, 2] data_min/data_max per tile (normalization.py:149-153)
    n_samples: np.ndarray          # int64 [n_tiles] samples per channel
    sample_rates: np.ndarray       # uint32 [n_tiles]
    channels: int
    bps: int                       # FLAC bits per sample (16 or 32)
    bits_per_sample: int           # the reference's notion (16 or 24)
    blocksize: int
    # seek index of the frames (frb_encode_index): byte size of every frame and bit offset of every subframe inside its
    # frame, tiles and frames in payload order; int32 views of uint32 data, on the payload's device (CPU for the host path)
    frame_bytes: Optional[torch.Tensor] = None
    sub_bitoff: Optional[torch.Tensor] = None
    sizes_all: Optional[np.ndarray] = None   # sharded path: frame bytes of EVERY tile of the scene (all ranks), see encode_tiles

    def frames_per_tile(self) -> np.ndarray:
        return (np.asarray(self.n_samples, dtype=np.int64) + self.blocksize - 1) // self.blocksize

    def index(self):
        """(frame_bytes, sub_bitoff) for Engine.decode_tiles / decode_streams, or None."""
        return None if self.frame_bytes is None else (self.frame_bytes, self.sub_bitoff)


class Engine:
    """One per process / per GPU.  Keeps grow-only workspaces so steady-state calls do not allocate."""

    def __init__(self, device: Optional[torch.device | int | str] = None):
        nat.require_cuda()
        if not torch.cuda.is_available():
            raise nat.NativeError(nat.ERR_NO_DEVICE, "Engine", "torch sees no CUDA device")
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.L = nat.lib()
        self._ws: dict[str, torch.Tensor] = {}
        # scan-path decode of multi-channel streams: False = skim CTAs inside the decode launch (in-order CTA dispatch assumed),
        # True = skim as its own launch.  Switched on for good the first time a decode thread reports that it gave up waiting
        # for a subframe offset (ST_OFFSET_WAIT_TIMEOUTS): the device is shared or does not dispatch in order.  See _decode.
        self._two_launch = False

    # ---------------------------------------------------------------- helpers
    def _buf(self, name: str, nbytes: int) -> torch.Tensor:
        t = self._ws.get(name)
        if t is None or t.numel() < nbytes:
            t = None
            self._ws.pop(name, None)
            t = torch.empty(int(nbytes * 1.125) + 4096, dtype=torch.uint8, device=self.device)
            self._ws[name] = t
        return t

    def _map_ws(self, n_tiles: int) -> torch.Tensor:
        nbytes = C.c_size_t(0)
        nat.check(self.L.frb_sample_map_workspace_size(n_tiles, C.byref(nbytes)), "frb_sample_map_workspace_size")
        return self._buf("map_ws", nbytes.value)

    def release(self):
        self._ws.clear()

    @staticmethod
    def audio_elem_bytes(bits_per_sample: int, dtype_code: int) -> int:
        """Bytes per sample of the planar audio buffer between the mapping kernels and the codec kernels: int16 for
        16-bit audio of 8/16-bit rasters (the tile path of C2/C3/C5), int32 otherwise."""
        return 2 if (bits_per_sample == 16 and dtype_code <= nat.DTYPE_CODES["int16"]) else 4

    def _upload(self, arr: np.ndarray) -> torch.Tensor:
        """A small host array -> a fresh device tensor (uint8 view) on the current stream, through the library's pinned
        staging + copy kernel: torch's .to(device) is a DMA transfer and would queue behind the bulk copies of the host
        pipelines (see frb_small_upload)."""
        a = np.ascontiguousarray(arr)
        nbytes = a.nbytes
        t = torch.empty((nbytes + 15) & ~15, dtype=torch.uint8, device=self.device)
        nat.check(self.L.frb_small_upload(t.data_ptr(), a.ctypes.data, nbytes, _stream_ptr()), "frb_small_upload")
        return t

    def _download(self, t: torch.Tensor, dtype, count: int) -> np.ndarray:
        """A small device tensor -> numpy (synchronises the current stream), off the copy engines as well."""
        out = np.empty(count, dtype=dtype)
        nat.check(self.L.frb_small_download(out.ctypes.data, t.data_ptr(), out.nbytes, _stream_ptr()), "frb_small_download")
        return out

    # ------------------------------------------------------------------ encode
    def normalize_tiles(self, raster: torch.Tensor, tiles: np.ndarray, bits_per_sample: Optional[int] = None,
                        d_minmax: Optional[torch.Tensor] = None, audio_i16: bool = False):
        """(bands,H,W) device raster -> (planar audio per tile, audio_base, n_px, minmax_dev, bits).  The audio is int32
        in a uint8 workspace buffer; with `audio_i16` (encode_tiles asks for it) it is an int16 tensor whenever
        audio_elem_bytes allows (encode_audio takes either; denormalize_tiles takes int32 only)."""
        assert raster.is_cuda and raster.is_contiguous() and raster.dim() == 3
        bands, H, W = raster.shape
        dt = str(raster.dtype).replace("torch.", "")
        code = nat.DTYPE_CODES[dt]
        if bits_per_sample is None:
            bits_per_sample = 16 if dt in ("uint8", "int8", "uint16", "int16") else 24
        n_tiles = len(tiles)
        npx = tiles["h"].astype(np.int64) * tiles["w"].astype(np.int64)
        _check_tile_sizes(npx)
        base = np.zeros(n_tiles, dtype=np.int64)
        np.cumsum(npx[:-1] * bands, out=base[1:])
        total = int((npx * bands).sum())
        with torch.cuda.device(self.device):
            s = _stream_ptr()
            d_tiles = self._upload(tiles.view(np.uint8))
            d_base = self._upload(base)
            if d_minmax is None:
                d_minmax = torch.empty(2 * n_tiles, dtype=torch.float64, device=self.device)
            esz = self.audio_elem_bytes(bits_per_sample, code) if audio_i16 else 4
            audio = self._buf("audio", total * esz)
            if esz == 2:
                audio = audio[: total * 2].view(torch.int16)
            nat.check(self.L.frb_minmax_tiles(raster.data_ptr(), code, bands, H, W, d_tiles.data_ptr(), n_tiles,
                                              d_minmax.data_ptr(), s), "frb_minmax_tiles")
            mws = self._map_ws(n_tiles)
            if esz == 2:
                nat.check(self.L.frb_normalize_tiles_i16(raster.data_ptr(), code, bands, H, W, d_tiles.data_ptr(), n_tiles,
                                                         d_minmax.data_ptr(), audio.data_ptr(),
                                                         d_base.data_ptr(), mws.data_ptr(), mws.numel(), s), "frb_normalize_tiles_i16")
            else:
                nat.check(self.L.frb_normalize_tiles(raster.data_ptr(), code, bands, H, W, d_tiles.data_ptr(), n_tiles,
                                                     d_minmax.data_ptr(), bits_per_sample, audio.data_ptr(),
                                                     d_base.data_ptr(), mws.data_ptr(), mws.numel(), s), "frb_normalize_tiles")
        return audio, base, npx, d_minmax, bits_per_sample

    def encode_audio(self, audio: torch.Tensor, n_samples: np.ndarray, audio_base: np.ndarray, sample_rates: np.ndarray,
                     channels: int, bps: int, level: int = 5, blocksize: int = 4096, payload_name: str = "payload",
                     fetch=None, range30: bool = False):
        """planar audio on the device (int32, or int16 for 16-bps streams: the element type is taken from the tensor) ->
        (payload uint8 tensor, offsets, sizes, frame sizes, subframe offsets).
        One host synchronisation: the per-stream sizes, which fix where every stream's frames go.  `fetch(d_sizes)`
        (optional) replaces the plain size download: it gets the device tensor of the sizes (int64[n_streams], filled by the
        analysis, stream-ordered) and returns them on the host -- encode_tiles uses it to bring the min/max pairs and the
        other ranks' sizes back in the SAME transfer."""
        n_streams = len(n_samples)
        a16 = audio.dtype == torch.int16
        if a16 and bps != 16:
            raise ValueError("int16 audio is for 16-bps streams")
        # range30: the caller vouches that a 32-bps stream holds samples below 2^30 in magnitude (24-bit audio of the tile path), which
        # lets two-channel streams use libFLAC's mid/side search there too (the 33-bit side channel then fits the int32 audio)
        p = nat.EncodeParams(n_streams, channels, bps, blocksize, level,
                             (nat.ENC_AUDIO_I16 if a16 else 0) | (nat.ENC_RANGE_30 if (range30 and bps == 32) else 0))
        frames = int(((n_samples + blocksize - 1) // blocksize).sum())
        ws_bytes = C.c_size_t(0)
        nat.check(self.L.frb_encode_workspace_size(C.byref(p), frames, C.byref(ws_bytes)), "frb_encode_workspace_size")
        ws = self._buf("enc_ws", ws_bytes.value)
        hn = np.ascontiguousarray(n_samples, dtype=np.uint64)
        hr = np.ascontiguousarray(sample_rates, dtype=np.uint32)
        hb = np.ascontiguousarray(audio_base, dtype=np.int64)
        sizes = np.zeros(n_streams, dtype=np.uint64)
        with torch.cuda.device(self.device):
            s = _stream_ptr()
            fb = torch.empty(frames, dtype=torch.int32, device=self.device)
            sb = torch.empty(frames * channels, dtype=torch.int32, device=self.device)
            if fetch is None:
                nat.check(self.L.frb_encode_analyse(C.byref(p), audio.data_ptr(), hn.ctypes.data, hr.ctypes.data, hb.ctypes.data,
                                                    ws.data_ptr(), ws.numel(), None, sizes.ctypes.data, s), "frb_encode_analyse")
                offsets = np.zeros(n_streams, dtype=np.uint64)
                np.cumsum(sizes[:-1], out=offsets[1:])
                total = int(sizes.sum())
                payload = self._buf(payload_name, total + 16)
                nat.check(self.L.frb_encode_emit(C.byref(p), ws.data_ptr(), ws.numel(), offsets.ctypes.data,
                                                 payload.data_ptr(), payload.numel(), None, s), "frb_encode_emit")
            else:
                # No host round trip between analysis and frame assembly: the streams are packed back to back by a device-side
                # scan of their sizes (frb_encode_emit with no host offsets) into a buffer sized for the worst case (VERBATIM
                # subframes), and the sizes come back in the step's single download afterwards.
                d_sizes = fetch.d_sizes
                nat.check(self.L.frb_encode_analyse(C.byref(p), audio.data_ptr(), hn.ctypes.data, hr.ctypes.data, hb.ctypes.data,
                                                    ws.data_ptr(), ws.numel(), d_sizes.data_ptr(), None, s), "frb_encode_analyse")
                if hasattr(fetch, "start"):
                    fetch.start()                         # e.g. the multi-GPU size exchange: overlaps the frame assembly
                bound = int(n_samples.sum()) * channels * (bps // 8) + frames * (24 + 8 * channels) + 64
                if channels == 2:
                    bound += frames * blocksize // 4          # a side subframe carries one more bit per sample
                payload = self._buf(payload_name, bound + 16)
                nat.check(self.L.frb_encode_emit(C.byref(p), ws.data_ptr(), ws.numel(), None,
                                                 payload.data_ptr(), payload.numel(), None, s), "frb_encode_emit")
            # seek index (frame sizes + subframe bit offsets): what lets a decoder skip the sync scan and the subframe walk
            nat.check(self.L.frb_encode_index(C.byref(p), ws.data_ptr(), ws.numel(), fb.data_ptr(), sb.data_ptr(), s), "frb_encode_index")
            if fetch is not None:
                sizes = np.ascontiguousarray(fetch(), dtype=np.uint64)
                offsets = np.zeros(n_streams, dtype=np.uint64)
                np.cumsum(sizes[:-1], out=offsets[1:])
                total = int(sizes.sum())
        return payload[:total], offsets.astype(np.int64), sizes.astype(np.int64), fb, sb

    def encode_tiles(self, raster: torch.Tensor, tiles: np.ndarray, level: int = 5, blocksize: int = 4096,
                     payload_name: str = "payload", size_exchange=None) -> EncodedTiles:
        """Whole pipeline for a batch of tiles of one device-resident raster.

        The step has ONE host round trip in the middle (frame assembly needs every stream's byte size for the output
        offsets): the tiles' min/max pairs ride along in that transfer, and with `size_exchange`
        (distributed.SizeExchange: the all-gather of per-tile sizes of the sharded path, cli.py:615-621) the other ranks'
        sizes do as well -- the collective is enqueued on the stream between analysis and download, so the multi-GPU
        path costs no extra synchronisation.  The gathered sizes come back as EncodedTiles.sizes_all."""
        bands = raster.shape[0]
        if not (1 <= bands <= 8):
            raise ValueError("FLAC carries at most 8 channels (bands)")
        n = len(tiles)
        extra = size_exchange.recv_count if size_exchange is not None else 0
        with torch.cuda.device(self.device):
            combo = torch.empty(3 * n + extra, dtype=torch.float64, device=self.device)     # [sizes int64 n | min/max 2n | gathered sizes]
        d_sizes = combo[:n].view(torch.int64)
        d_minmax = combo[n:3 * n]
        audio, base, npx, d_minmax, bits = self.normalize_tiles(raster, tiles, d_minmax=d_minmax, audio_i16=True)
        bps = 16 if bits == 16 else 32            # pyflac derives bps from the array dtype (docs/sonos-pyflac.txt:1988-1991)
        rates = sample_rates_for_pixel_counts(npx)                # one vector expression (4096 tiles: 5 ms of Python before)
        got = {}

        def start():          # called by encode_audio between analysis and frame assembly
            if size_exchange is not None:
                size_exchange.start(d_sizes, combo[3 * n:].view(torch.int64))

        def fetch():
            if size_exchange is not None:
                size_exchange.wait()
            host = self._download(combo.view(torch.uint8), np.uint8, combo.numel() * 8)
            got["minmax"] = host[8 * n:24 * n].view(np.float64).reshape(-1, 2).copy()
            if size_exchange is not None:
                got["sizes_all"] = size_exchange.unpack(host[24 * n:].view(np.int64))
            return host[:8 * n].view(np.int64)

        fetch.d_sizes = d_sizes
        fetch.start = start
        payload, offsets, sizes, fb, sb = self.encode_audio(audio, npx, base, rates, bands, bps, level, blocksize, payload_name, fetch=fetch,
                                                            range30=(bits == 24))
        enc = EncodedTiles(payload, offsets, sizes, got["minmax"], npx, rates, bands, bps, bits, blocksize, fb, sb)
        enc.sizes_all = got.get("sizes_all")
        return enc

    # ------------------------------------------------------------------ encode, host buffers (pipelined)
    @staticmethod
    def _row_groups(tiles: np.ndarray, row_bytes: int = 0, target_bytes: int = 0) -> List[Tuple[int, int, int, int]]:
        """Consecutive runs of tiles that cover one band of rows: [(first, last+1, row0, row1)].  A row-major tile
        grid (cli.py:553-556) gives one run per tile row; vertically adjacent runs are merged until a group holds
        about `target_bytes` of raster (many small tiles would otherwise mean many tiny pipeline stages)."""
        ro = tiles["row_off"].astype(np.int64)
        re = ro + tiles["h"].astype(np.int64)
        groups: List[Tuple[int, int, int, int]] = []
        i, n = 0, len(tiles)
        while i < n:
            j = i + 1
            while j < n and ro[j] == ro[i] and re[j] == re[i]:
                j += 1
            g = (i, j, int(ro[i]), int(re[i]))
            if groups and target_bytes and groups[-1][3] == g[2] and (groups[-1][3] - groups[-1][2]) * row_bytes < target_bytes:
                p = groups[-1]
                groups[-1] = (p[0], j, p[2], g[3])
            else:
                groups.append(g)
            i = j
        return groups

    def _pinned(self, name: str, nbytes: int) -> torch.Tensor:
        t = self._ws.get(name)
        if t is None or t.numel() < nbytes:
            self._ws.pop(name, None)
            t = torch.empty(int(nbytes) + 4096, dtype=torch.uint8, pin_memory=True)     # straight from the pinned allocator (no pageable detour)
            self._ws[name] = t
        return t

    def encode_tiles_host(self, host_raster: torch.Tensor, tiles: np.ndarray, level: int = 5, blocksize: int = 4096,
                          host_out: Optional[torch.Tensor] = None, group_bytes: Optional[int] = None,
                          timeline: Optional[list] = None) -> EncodedTiles:
        """Host (bands,H,W) raster in, host frames out: the end-to-end form of encode_tiles.

        The reference walks tiles serially (cli.py:553-622).  Here the tile rows are pipelined over three
        streams so PCIe and the GPU work concurrently: H2D of tile row g+1 (double-buffered slab) overlaps
        the encode of row g, which overlaps the D2H of row g-1's frames (double-buffered payload).
        `host_raster` and `host_out` should be pinned; the returned EncodedTiles.payload is a CPU tensor
        (a view of host_out, or of an engine-owned pinned buffer that the next call reuses).  `group_bytes`: raster
        bytes per pipeline stage (default: a twelfth of the raster, at least 32 MiB; 0 = one stage per tile row)."""
        assert not host_raster.is_cuda and host_raster.is_contiguous() and host_raster.dim() == 3
        bands, H, W = host_raster.shape
        esize = host_raster.element_size()
        total_bytes = int(host_raster.numel()) * esize
        groups = self._row_groups(tiles, bands * W * esize, group_bytes if group_bytes is not None else max(total_bytes // 12, 32 << 20))
        max_rows = max(r1 - r0 for _, _, r0, r1 in groups)
        if host_out is None:
            frames = int(sum((int(t["h"]) * int(t["w"]) + blocksize - 1) // blocksize for t in tiles))
            cap = int(host_raster.numel()) * (2 if esize <= 2 else 4) + frames * (32 + 8 * bands) + 4096
            host_out = self._pinned("host_out", cap)
        with torch.cuda.device(self.device):
            if not hasattr(self, "_streams"):
                self._streams = (torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream())
            s_h2d, s_comp, s_d2h = self._streams
            entry = torch.cuda.current_stream()
            for st in self._streams:
                st.wait_stream(entry)
            slabs = [self._buf(f"slab{k}", bands * max_rows * W * esize) for k in range(2)]
            ev_h2d: List[torch.cuda.Event] = []
            ev_comp: List[torch.cuda.Event] = []
            ev_d2h: List[torch.cuda.Event] = []
            timed = timeline is not None          # debug: per-stage device timestamps (tools/e2e_timeline.py)
            if timed:
                t_origin = torch.cuda.Event(enable_timing=True)
                t_origin.record(entry)
                marks = []
                host_marks = []
                import time

            def mark(stream, name, g):
                if timed:
                    e = torch.cuda.Event(enable_timing=True)
                    e.record(stream)
                    marks.append((name, g, e))
                    host_marks.append((name, g, time.perf_counter()))

            def slab_view(g):
                _, _, r0, r1 = groups[g]
                return slabs[g % 2][: bands * (r1 - r0) * W * esize].view(host_raster.dtype).reshape(bands, r1 - r0, W)

            def enqueue_h2d(g):
                _, _, r0, r1 = groups[g]
                with torch.cuda.stream(s_h2d):
                    if g >= 2:
                        s_h2d.wait_event(ev_comp[g - 2])          # slab g%2 is free once row g-2 has been encoded
                    dst = slab_view(g)
                    mark(s_h2d, "h2d_begin", g)
                    for b in range(bands):                          # each band's rows are one contiguous block
                        dst[b].copy_(host_raster[b, r0:r1], non_blocking=True)
                    e = torch.cuda.Event()
                    e.record(s_h2d)
                    ev_h2d.append(e)
                    mark(s_h2d, "h2d_end", g)

            parts: List[EncodedTiles] = []
            total = 0
            enqueue_h2d(0)
            for g, (i0, i1, r0, r1) in enumerate(groups):
                if g + 1 < len(groups):
                    enqueue_h2d(g + 1)
                local = tiles[i0:i1].copy()
                local["row_off"] -= r0
                with torch.cuda.stream(s_comp):
                    s_comp.wait_event(ev_h2d[g])
                    if g >= 2:
                        s_comp.wait_event(ev_d2h[g - 2])          # payload g%2 has left the device
                    mark(s_comp, "enc_begin", g)
                    enc = self.encode_tiles(slab_view(g), local, level, blocksize, payload_name=f"payload{g % 2}")
                    e = torch.cuda.Event()
                    e.record(s_comp)
                    ev_comp.append(e)
                    mark(s_comp, "enc_end", g)
                n = int(enc.payload.numel())
                if total + n > host_out.numel():
                    raise nat.NativeError(nat.ERR_OVERFLOW, "encode_tiles_host", "host_out too small")
                with torch.cuda.stream(s_d2h):
                    s_d2h.wait_event(ev_comp[g])
                    mark(s_d2h, "d2h_begin", g)
                    host_out[total:total + n].copy_(enc.payload, non_blocking=True)
                    e = torch.cuda.Event()
                    e.record(s_d2h)
                    ev_d2h.append(e)
                    mark(s_d2h, "d2h_end", g)
                enc.offsets = enc.offsets + total
                parts.append(enc)
                total += n
            for st in self._streams:
                entry.wait_stream(st)
            s_d2h.synchronize()
            if timed:
                torch.cuda.synchronize()
                timeline.extend((name, g, t_origin.elapsed_time(e)) for name, g, e in marks)
                h0 = host_marks[0][2]
                timeline.extend(("host_" + name, g, (t - h0) * 1e3) for name, g, t in host_marks)
        p0 = parts[0]
        fb = torch.cat([p.frame_bytes for p in parts]).cpu() if all(p.frame_bytes is not None for p in parts) else None
        sb = torch.cat([p.sub_bitoff for p in parts]).cpu() if fb is not None else None
        return EncodedTiles(host_out[:total], np.concatenate([p.offsets for p in parts]), np.concatenate([p.sizes for p in parts]),
                            np.concatenate([p.minmax for p in parts]), np.concatenate([p.n_samples for p in parts]),
                            np.concatenate([p.sample_rates for p in parts]), p0.channels, p0.bps, p0.bits_per_sample, p0.blocksize, fb, sb)

    # ------------------------------------------------------------------ decode
    def _decode_params(self, n_streams: int, channels: int, bps: int, blocksize: int, verify_crc: bool, max_order: int,
                       total_frames: int, ws_name: str):
        """DecodeParams of one decode attempt in the engine's current launch mode, and its workspace."""
        p = nat.DecodeParams(n_streams, channels, bps, blocksize, (1 if verify_crc else 0) | (2 if self._two_launch else 0), max_order)
        ws_bytes = C.c_size_t(0)
        nat.check(self.L.frb_decode_workspace_size(C.byref(p), total_frames, C.byref(ws_bytes)), "frb_decode_workspace_size")
        return p, self._buf(ws_name, ws_bytes.value)

    def _decode(self, launch, d_status: torch.Tensor, has_index: bool, allow_scan: bool, where: str) -> np.ndarray:
        """Run decode_ladder over `launch(max_order, use_index)`, which enqueues one decode writing d_status.  When a decode
        thread gave up waiting for a subframe offset, the engine switches to two-launch mode for good and runs the ladder once
        more.  Every attempt ends in a synchronising status download, so the caller's staged tables are still alive then."""
        def attempt(max_order, use_index):
            launch(max_order, use_index)
            return self._download(d_status, np.int32, 8).astype(np.int64)

        status = decode_ladder(attempt, has_index, allow_scan, where)
        if status[nat.ST_OFFSET_WAIT_TIMEOUTS] and not self._two_launch:
            self._two_launch = True                  # offsets did not arrive inside the fused launch: separate skim launch from now on
            status = decode_ladder(attempt, has_index, allow_scan, where)
        return status

    def decode_streams(self, data: torch.Tensor, byte_offsets: np.ndarray, byte_lengths: np.ndarray, n_samples: np.ndarray,
                       sample_rates: np.ndarray, channels: int, bps: int, blocksize: int = 4096, verify_crc: bool = True,
                       sync: bool = True, name: str = "dec", index=None):
        """Frames of many streams (device bytes) -> int32 planar audio on the device.

        data must be readable 16 bytes past the last stream.  Returns (audio, audio_base, status words).  sync=False makes
        only the first attempt of decode_ladder, leaves it queued on the current stream and returns the status words as a
        device tensor (the caller checks them: ST_LPC_ORDER_ABOVE_12 means rerun with sync).  index = (frame_bytes,
        sub_bitoff) of these streams (EncodedTiles.index(), or the container's "frbI" blocks): the sync scan and the subframe
        walk are skipped; an index that does not fit the streams is detected while decoding and the call scans instead."""
        st, fstart = _stream_table(byte_offsets, byte_lengths, n_samples, sample_rates, channels, blocksize)
        total_frames = int(fstart[-1])
        base = st["audio_base"].copy()
        with torch.cuda.device(self.device):
            s = _stream_ptr()
            audio = self._buf(name + "_audio", int(st["n_samples"].sum()) * channels * 4)
            d_status = torch.zeros(8, dtype=torch.int32, device=self.device)
            idx = self._index_on_device(index, total_frames, channels)

            def launch(max_order, use_idx):
                p, ws = self._decode_params(len(st), channels, bps, blocksize, verify_crc, max_order, total_frames, name + "_ws")
                if use_idx:
                    nat.check(self.L.frb_decode_batch_indexed(C.byref(p), st.ctypes.data, data.data_ptr(), total_frames, idx[0].data_ptr(),
                                                              idx[1].data_ptr(), audio.data_ptr(), ws.data_ptr(), ws.numel(),
                                                              d_status.data_ptr(), s), "frb_decode_batch_indexed")
                else:
                    nat.check(self.L.frb_decode_batch(C.byref(p), st.ctypes.data, data.data_ptr(), total_frames, audio.data_ptr(),
                                                      ws.data_ptr(), ws.numel(), d_status.data_ptr(), s), "frb_decode_batch")

            if not sync:
                launch(12, idx is not None)
                return audio, base, d_status
            status = self._decode(launch, d_status, idx is not None, True, "frb_decode_batch")
        return audio, base, status

    def _index_on_device(self, index, total_frames: int, channels: int):
        """(frame_bytes, sub_bitoff) as int32 device tensors, or None when they do not have the index's shape (_index_fits)."""
        if not _index_fits(index, total_frames, channels):
            return None

        def dev(x):
            if isinstance(x, np.ndarray):
                return self._upload(np.ascontiguousarray(x, dtype=np.uint32).view(np.uint8))[:4 * x.size].view(torch.int32)
            return x.contiguous() if x.is_cuda else self._upload(x.contiguous().numpy().view(np.uint8))[:4 * x.numel()].view(torch.int32)

        d_fb = dev(index[0])
        return d_fb, dev(index[1]) if channels > 1 else d_fb

    def decode_tiles(self, data: torch.Tensor, byte_offsets: np.ndarray, byte_lengths: np.ndarray, tiles: np.ndarray,
                     sample_rates: np.ndarray, minmax: np.ndarray, scale: float, out: torch.Tensor, bps: int,
                     blocksize: int = 4096, verify_crc: bool = True, fused: Optional[bool] = None, index=None) -> np.ndarray:
        """Frames of a batch of tiles (device bytes) -> windows of the (bands,H,W) device raster `out`, decoded and
        denormalised in one launch (frb_decode_tiles); what `extract` + flac_to_tiff do per tile (cli.py:297-315,
        converter.py:181-253).  Returns the status words.  Two-band rasters go through decode_streams +
        denormalize_tiles (their frames may be mid/side coded); `fused` forces (True) or forbids (False) the one-launch
        form, None picks it where it is the faster one (_fused_default)."""
        bands, H, W = out.shape
        n_tiles = len(tiles)
        n_samples = tiles["h"].astype(np.int64) * tiles["w"].astype(np.int64)
        _check_tile_sizes(n_samples)
        dt = str(out.dtype).replace("torch.", "")
        if bands == 2 or not (_fused_default(bps, dt, scale) if fused is None else fused):
            audio, base, status = self.decode_streams(data, byte_offsets, byte_lengths, n_samples, sample_rates, bands, bps, blocksize,
                                                      verify_crc, index=index)
            self.denormalize_tiles(audio, base, tiles, minmax, scale, out)
            return status
        st, fstart = _stream_table(byte_offsets, byte_lengths, n_samples, sample_rates, bands, blocksize)
        total_frames = int(fstart[-1])
        with torch.cuda.device(self.device):
            s = _stream_ptr()
            # one staging buffer, one copy: tile table followed by the min/max pairs
            stage = np.zeros(n_tiles * 16 + n_tiles * 16, dtype=np.uint8)
            stage[: n_tiles * 16] = np.ascontiguousarray(tiles).view(np.uint8)
            stage[n_tiles * 16:] = np.ascontiguousarray(minmax, dtype=np.float64).reshape(-1).view(np.uint8)
            d_stage = self._upload(stage)
            d_status = torch.zeros(8, dtype=torch.int32, device=self.device)
            idx = self._index_on_device(index, total_frames, bands)

            def launch(max_order, use_idx):
                p, ws = self._decode_params(n_tiles, bands, bps, blocksize, verify_crc, max_order, total_frames, "dec_ws")
                if use_idx:
                    nat.check(self.L.frb_decode_tiles_indexed(C.byref(p), st.ctypes.data, data.data_ptr(), total_frames,
                                                              idx[0].data_ptr(), idx[1].data_ptr(),
                                                              d_stage.data_ptr(), d_stage.data_ptr() + n_tiles * 16, float(scale),
                                                              out.data_ptr(), nat.DTYPE_CODES[dt], bands, H, W,
                                                              ws.data_ptr(), ws.numel(), d_status.data_ptr(), s), "frb_decode_tiles_indexed")
                else:
                    nat.check(self.L.frb_decode_tiles(C.byref(p), st.ctypes.data, data.data_ptr(), total_frames,
                                                      d_stage.data_ptr(), d_stage.data_ptr() + n_tiles * 16, float(scale),
                                                      out.data_ptr(), nat.DTYPE_CODES[dt], bands, H, W,
                                                      ws.data_ptr(), ws.numel(), d_status.data_ptr(), s), "frb_decode_tiles")

            return self._decode(launch, d_status, idx is not None, True, "frb_decode_tiles")

    def decode_window(self, data: torch.Tensor, byte_offsets: np.ndarray, byte_lengths: np.ndarray, tiles: np.ndarray,
                      sample_rates: np.ndarray, minmax: np.ndarray, scale: float, window, out: torch.Tensor, bps: int,
                      blocksize: int = 4096, index=None, runs_only: bool = False, verify_crc: bool = True,
                      fused: Optional[bool] = None) -> np.ndarray:
        """The pixels of `window` (col_off, row_off, width, height, image coordinates) from the frames of the tiles that
        cover it (image coordinates) -> the (bands, height, width) device array `out`.  Only the frames each tile's part of
        the window needs are decoded (window_frames).  Returns the status words; ST_FRAMES_DECODED counts the decoded frames.
        byte_offsets / byte_lengths: where each tile's frames are in `data` -- all of them, or with `runs_only` only the
        run's frames (a partial read; then the seek index is required, and a rejected index is reported in the status words
        instead of falling back to a scan, which would need every frame).  index: (frame_bytes, sub_bitoff) of all the
        tiles' frames in tile order (host arrays), or None (scan path).  `fused` as decode_tiles."""
        bands = out.shape[0]
        col0, row0, width, height = (int(v) for v in window)
        if tuple(out.shape[1:]) != (height, width):
            raise ValueError("out must have the window's shape")
        n_samples = tiles["h"].astype(np.int64) * tiles["w"].astype(np.int64)
        _check_tile_sizes(n_samples)
        fstart = _stream_table(byte_offsets, byte_lengths, n_samples, sample_rates, bands, blocksize)[1]
        fits = _index_fits(index, int(fstart[-1]), bands)
        fb_all = np.asarray(index[0]).view(np.uint32).reshape(-1) if fits else None
        sb_all = np.asarray(index[1]).view(np.uint32).reshape(-1) if fits and bands > 1 else None
        if runs_only and fb_all is None:
            raise ValueError("decode_window(runs_only=True) needs the tiles' seek index")
        runs = window_frames(tiles, window, blocksize,
                             None if fb_all is None else [fb_all[fstart[i]:fstart[i + 1]] for i in range(len(tiles))])
        if len(runs) == 0:
            raise ValueError(f"window {tuple(window)} covers no tile")
        sel = runs["tile"]
        n_runs = len(runs)
        dt = str(out.dtype).replace("torch.", "")
        two_step = bands == 2 or not (_fused_default(bps, dt, scale) if fused is None else fused)
        run_n = np.minimum((runs["first_frame"] + runs["n_frames"]) * blocksize, n_samples[sel]) - runs["first_frame"] * blocksize
        st = np.zeros(n_runs, dtype=nat.WINDOW_STREAM_DTYPE)
        st["total_samples"] = n_samples[sel]
        st["sample_rate"] = np.asarray(sample_rates)[sel]
        st["first_frame"] = runs["first_frame"]
        st["n_frames"] = runs["n_frames"]
        st["frame_base"][1:] = np.cumsum(runs["n_frames"][:-1])
        st["audio_base"][1:] = np.cumsum(run_n[:-1] * bands)
        total_frames = int(runs["n_frames"].sum())
        idx_host = None
        if fb_all is not None:
            parts_fb = [fb_all[fstart[t] + f0:fstart[t] + f0 + n] for t, f0, n in zip(sel, runs["first_frame"], runs["n_frames"])]
            parts_sb = [sb_all[(fstart[t] + f0) * bands:(fstart[t] + f0 + n) * bands]
                        for t, f0, n in zip(sel, runs["first_frame"], runs["n_frames"])] if bands > 1 else None
            idx_host = (np.concatenate(parts_fb), np.concatenate(parts_sb) if bands > 1 else None)
        offs = np.asarray(byte_offsets, dtype=np.int64)[sel]
        lens = np.asarray(byte_lengths, dtype=np.int64)[sel]
        with torch.cuda.device(self.device):
            s = _stream_ptr()
            stage = np.zeros(n_runs * 32, dtype=np.uint8)
            stage[: n_runs * 16] = np.ascontiguousarray(tiles[sel]).view(np.uint8)
            stage[n_runs * 16:] = np.ascontiguousarray(np.asarray(minmax, dtype=np.float64).reshape(-1, 2)[sel]).reshape(-1).view(np.uint8)
            d_stage = self._upload(stage)
            d_status = torch.zeros(8, dtype=torch.int32, device=self.device)
            idx = None if idx_host is None else self._index_on_device(idx_host, total_frames, bands)
            audio = self._buf("win_audio", int(run_n.sum()) * bands * 4) if two_step else None
            win = nat.Tile(row0, col0, height, width)

            def launch(max_order, use_idx):
                if use_idx:
                    st["byte_offset"] = offs if runs_only else offs + runs["byte_offset"]
                    st["byte_length"] = lens if runs_only else runs["byte_length"]
                else:
                    st["byte_offset"], st["byte_length"] = offs, lens
                p, ws = self._decode_params(n_runs, bands, bps, blocksize, verify_crc, max_order, total_frames, "dec_ws")
                nat.check(self.L.frb_decode_window(C.byref(p), st.ctypes.data, data.data_ptr(), total_frames,
                                                   idx[0].data_ptr() if use_idx else None, idx[1].data_ptr() if use_idx else None,
                                                   d_stage.data_ptr(), d_stage.data_ptr() + n_runs * 16, float(scale), win,
                                                   audio.data_ptr() if two_step else out.data_ptr(), -1 if two_step else nat.DTYPE_CODES[dt],
                                                   ws.data_ptr(), ws.numel(), d_status.data_ptr(), s), "frb_decode_window")

            # the scan path needs every frame of the streams: with runs_only the caller decides what a rejected index means
            status = self._decode(launch, d_status, idx is not None, not runs_only, "frb_decode_window")
            if two_step and not (nat.status_damaged(status) or status[nat.ST_LPC_ORDER_ABOVE_12] or status[nat.ST_OFFSET_WAIT_TIMEOUTS]):
                d_st = self._upload(st)
                nat.check(self.L.frb_denormalize_window(audio.data_ptr(), d_st.data_ptr(), n_runs, blocksize, d_stage.data_ptr(),
                                                        d_stage.data_ptr() + n_runs * 16, float(scale), win, out.data_ptr(),
                                                        nat.DTYPE_CODES[dt], bands, s), "frb_denormalize_window")
                torch.cuda.current_stream().synchronize()
        return status

    def decode_tiles_host(self, host_payload: torch.Tensor, byte_offsets: np.ndarray, byte_lengths: np.ndarray, tiles: np.ndarray,
                          sample_rates: np.ndarray, minmax: np.ndarray, scale: float, host_out: torch.Tensor, bps: int,
                          blocksize: int = 4096, group_bytes: Optional[int] = None, index=None) -> np.ndarray:
        """Host frames in, host (bands,H,W) raster out: the end-to-end form of decode_tiles and the mirror of
        encode_tiles_host.  Tile rows are pipelined over three streams: H2D of the frames of rows g+1 (double-buffered),
        the fused decode of rows g into a device slab, D2H of the pixels of rows g-1.  `host_payload` (uint8, the tiles'
        frames in row-major tile order) and `host_out` should be pinned.  Returns the summed status words."""
        assert not host_out.is_cuda and host_out.is_contiguous() and host_out.dim() == 3 and not host_payload.is_cuda
        bands, H, W = host_out.shape
        esize = host_out.element_size()
        total_bytes = int(host_out.numel()) * esize
        groups = self._row_groups(tiles, bands * W * esize, group_bytes if group_bytes is not None else max(total_bytes // 12, 32 << 20))
        max_rows = max(r1 - r0 for _, _, r0, r1 in groups)
        byte_offsets = np.asarray(byte_offsets, dtype=np.int64)
        byte_lengths = np.asarray(byte_lengths, dtype=np.int64)
        # seek index: uploaded once, sliced per stage by frame range (tiles and frames are in payload order)
        frame_start = _stream_table(byte_offsets, byte_lengths, tiles["h"].astype(np.int64) * tiles["w"].astype(np.int64), sample_rates,
                                    bands, blocksize)[1]
        with torch.cuda.device(self.device):
            d_index = self._index_on_device(index, int(frame_start[-1]), bands)
        spans = [(int(byte_offsets[i0]), int(byte_offsets[i1 - 1] + byte_lengths[i1 - 1])) for i0, i1, _, _ in groups]
        max_span = max(b - a for a, b in spans)
        status = np.zeros(8, dtype=np.int64)
        with torch.cuda.device(self.device):
            if not hasattr(self, "_streams"):
                self._streams = (torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream())
            s_h2d, s_comp, s_d2h = self._streams
            entry = torch.cuda.current_stream()
            for st in self._streams:
                st.wait_stream(entry)
            frames_dev = [self._buf(f"dec_frames{k}", max_span + 64 + 16) for k in range(2)]
            slabs = [self._buf(f"dec_slab{k}", bands * max_rows * W * esize) for k in range(2)]
            ev_h2d: List[torch.cuda.Event] = []
            ev_comp: List[torch.cuda.Event] = []
            ev_d2h: List[torch.cuda.Event] = []

            def enqueue_h2d(g):
                a, b = spans[g]
                with torch.cuda.stream(s_h2d):
                    if g >= 2:
                        s_h2d.wait_event(ev_comp[g - 2])          # frames buffer g%2 has been decoded
                    buf = frames_dev[g % 2]
                    buf[:b - a].copy_(host_payload[a:b], non_blocking=True)
                    buf[b - a:b - a + 64].zero_()                  # readable slack behind the last frame
                    e = torch.cuda.Event()
                    e.record(s_h2d)
                    ev_h2d.append(e)

            enqueue_h2d(0)
            for g, (i0, i1, r0, r1) in enumerate(groups):
                if g + 1 < len(groups):
                    enqueue_h2d(g + 1)
                local = tiles[i0:i1].copy()
                local["row_off"] -= r0
                slab = slabs[g % 2][: bands * (r1 - r0) * W * esize].view(host_out.dtype).reshape(bands, r1 - r0, W)
                with torch.cuda.stream(s_comp):
                    s_comp.wait_event(ev_h2d[g])
                    if g >= 2:
                        s_comp.wait_event(ev_d2h[g - 2])          # slab g%2 has left the device
                    a, b = spans[g]
                    f0, f1 = int(frame_start[i0]), int(frame_start[i1])
                    gidx = None if d_index is None else (d_index[0][f0:f1], d_index[1][f0 * bands:f1 * bands] if bands > 1 else d_index[0][f0:f1])
                    st = self.decode_tiles(frames_dev[g % 2][:b - a + 64], byte_offsets[i0:i1] - a, byte_lengths[i0:i1], local,
                                           sample_rates[i0:i1], minmax[i0:i1], scale, slab, bps, blocksize, index=gidx)
                    status += st
                    e = torch.cuda.Event()
                    e.record(s_comp)
                    ev_comp.append(e)
                with torch.cuda.stream(s_d2h):
                    s_d2h.wait_event(ev_comp[g])
                    for b_ in range(bands):
                        host_out[b_, r0:r1].copy_(slab[b_], non_blocking=True)
                    e = torch.cuda.Event()
                    e.record(s_d2h)
                    ev_d2h.append(e)
            for st_ in self._streams:
                entry.wait_stream(st_)
            s_d2h.synchronize()
        return status

    def denormalize_tiles(self, audio: torch.Tensor, audio_base: np.ndarray, tiles: np.ndarray, minmax: np.ndarray,
                          scale: float, out: torch.Tensor, sync: bool = True):
        """int32 planar audio -> windows of the (bands,H,W) device raster `out` (denormalize_from_audio, int path)."""
        bands, H, W = out.shape
        dt = str(out.dtype).replace("torch.", "")
        _check_tile_sizes(tiles["h"].astype(np.int64) * tiles["w"].astype(np.int64))
        with torch.cuda.device(self.device):
            s = _stream_ptr()
            d_tiles = self._upload(tiles.view(np.uint8))
            d_base = self._upload(np.ascontiguousarray(audio_base, dtype=np.int64))
            d_mm = self._upload(np.ascontiguousarray(minmax, dtype=np.float64).reshape(-1))
            mws = self._map_ws(len(tiles))
            nat.check(self.L.frb_denormalize_tiles(audio.data_ptr(), d_base.data_ptr(), d_tiles.data_ptr(), len(tiles),
                                                   d_mm.data_ptr(), float(scale), out.data_ptr(), nat.DTYPE_CODES[dt],
                                                   bands, H, W, mws.data_ptr(), mws.numel(), s), "frb_denormalize_tiles")
            # keep the staging tensors alive until the kernel has consumed them
            if sync:
                torch.cuda.current_stream().synchronize()
            else:
                for t in (d_tiles, d_base, d_mm):
                    t.record_stream(torch.cuda.current_stream())
        return out


_default_engine: Optional[Engine] = None


def default_engine() -> Engine:
    global _default_engine
    if _default_engine is None:
        _default_engine = Engine()
    return _default_engine
