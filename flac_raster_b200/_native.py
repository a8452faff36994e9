"""ctypes binding of libflacraster_b200.so (include/flacraster_b200.h).

The CUDA library is the product; there is no CPU fallback.  Importing this
module on a machine where the library has not been built raises, and every
compute call fails loudly when no CUDA device is present.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

_PKG = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ["FRB_LIB_PATH"]) if os.environ.get("FRB_LIB_PATH") else _PKG / "lib" / "libflacraster_b200.so"   # override: kernel variant experiments
CSRC = _PKG / "csrc"

FRB_OK = 0
ERR_INVALID_ARG, ERR_CUDA, ERR_UNSUPPORTED, ERR_BAD_STREAM, ERR_CRC, ERR_OVERFLOW, ERR_NO_DEVICE = range(1, 8)

DTYPE_CODES = {
    "uint8": 0, "int8": 1, "uint16": 2, "int16": 3,
    "uint32": 4, "int32": 5, "float32": 6, "float64": 7,
}


class NativeError(RuntimeError):
    def __init__(self, status: int, where: str, detail: str = ""):
        self.status = status
        super().__init__(f"{where}: status {status}" + (f" ({detail})" if detail else ""))


class Tile(C.Structure):
    _fields_ = [("row_off", C.c_uint32), ("col_off", C.c_uint32), ("h", C.c_uint32), ("w", C.c_uint32)]


TILE_DTYPE = np.dtype([("row_off", "<u4"), ("col_off", "<u4"), ("h", "<u4"), ("w", "<u4")])


class EncodeParams(C.Structure):
    _fields_ = [("n_streams", C.c_uint32), ("channels", C.c_uint32), ("bps", C.c_uint32),
                ("blocksize", C.c_uint32), ("level", C.c_uint32), ("reserved", C.c_uint32)]


ENC_AUDIO_I16 = 1          # frb_encode_params.reserved flag (FRB_ENC_AUDIO_I16): d_audio holds int16 elements
ENC_RANGE_30 = 2           # FRB_ENC_RANGE_30: every sample of a 32-bps stream is below 2^30 in magnitude (mid/side is then allowed)


class DecodeParams(C.Structure):
    _fields_ = [("n_streams", C.c_uint32), ("channels", C.c_uint32), ("bps", C.c_uint32),
                ("blocksize", C.c_uint32), ("verify_crc16", C.c_uint32), ("reserved", C.c_uint32)]


# the eight status words every decode call writes (d_status of frb_decode_batch), in order; the eighth is always 0
(ST_FRAMES_MISSING, ST_CRC16_ERRORS, ST_PARSE_ERRORS, ST_FRAMES_DECODED, ST_LPC_ORDER_ABOVE_12, ST_OFFSET_WAIT_TIMEOUTS,
 ST_TILES_REJECTED, ST_RESERVED) = range(8)


def status_damaged(status) -> bool:
    """Frames missing, a CRC-16 mismatch or a parse error: the bytes (or their seek index) do not hold the frames asked for."""
    return bool(status[ST_FRAMES_MISSING] or status[ST_CRC16_ERRORS] or status[ST_PARSE_ERRORS])


TILE_HEADER_DTYPE = np.dtype([
    ("first_frame_offset", "<u4"), ("sample_rate", "<u4"), ("channels", "<u4"), ("bps", "<u4"), ("min_blocksize", "<u4"),
    ("max_blocksize", "<u4"), ("width", "<u4"), ("height", "<u4"), ("count", "<u4"), ("dtype", "<i4"), ("flags", "<u4"),
    ("index_offset", "<u4"), ("index_len", "<u4"), ("_pad", "<u4"), ("total_samples", "<u8"),
    ("data_min", "<f8"), ("data_max", "<f8"), ("nodata", "<f8"),
])

# frb_window_stream: a run of frames [first_frame, first_frame + n_frames) of a stream of total_samples samples
WINDOW_STREAM_DTYPE = np.dtype([
    ("byte_offset", "<u8"), ("byte_length", "<u8"), ("total_samples", "<u8"), ("audio_base", "<i8"),
    ("sample_rate", "<u4"), ("frame_base", "<u4"), ("first_frame", "<u4"), ("n_frames", "<u4"),
])

DECODE_STREAM_DTYPE = np.dtype([
    ("byte_offset", "<u8"), ("byte_length", "<u8"), ("n_samples", "<u8"), ("audio_base", "<i8"),
    ("sample_rate", "<u4"), ("frame_base", "<u4"),
])

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC"]


def build(force: bool = False, verbose: bool = False) -> Path:
    """Compile the unity build for sm_100a in-tree (nvcc cross-compiles without a GPU)."""
    srcs = sorted(CSRC.glob("*.cu")) + sorted(CSRC.glob("*.cuh")) + [_PKG.parent / "include" / "flacraster_b200.h"]
    newest = max(p.stat().st_mtime for p in srcs)
    if not force and LIB_PATH.exists() and LIB_PATH.stat().st_mtime >= newest:
        return LIB_PATH
    LIB_PATH.parent.mkdir(exist_ok=True)
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = [nvcc, *NVCC_FLAGS, "-o", str(LIB_PATH), str(CSRC / "flacraster_b200.cu")]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    subprocess.check_call(cmd)
    return LIB_PATH


_lib = None

_EXPORTS = [
    "frb_version", "frb_error_string", "frb_last_cuda_error", "frb_device_count", "frb_launch_count", "frb_selftest_crc16",
    "frb_profile_enable", "frb_profile_last_ms", "frb_small_upload", "frb_small_download",
    "frb_minmax_tiles", "frb_normalize_tiles", "frb_normalize_tiles_i16", "frb_denormalize_tiles", "frb_sample_map_workspace_size",
    "frb_minmax_flat", "frb_normalize_flat", "frb_denormalize_flat", "frb_selftest_division",
    "frb_encode_workspace_size", "frb_encode_analyse", "frb_encode_emit", "frb_encode_index",
    "frb_decode_workspace_size", "frb_decode_batch", "frb_decode_tiles", "frb_decode_batch_indexed", "frb_decode_tiles_indexed",
    "frb_decode_window", "frb_denormalize_window",
    "frb_probe_stream", "frb_debug_spin", "frb_parse_tile_headers", "frb_gather_seek_index",
    "frb_host_encode", "frb_host_decode",
    "frb_stream_encoder_new", "frb_stream_encoder_delete", "frb_stream_encoder_set_channels",
    "frb_stream_encoder_set_bits_per_sample", "frb_stream_encoder_set_sample_rate",
    "frb_stream_encoder_set_compression_level", "frb_stream_encoder_set_blocksize",
    "frb_stream_encoder_set_total_samples_estimate", "frb_stream_encoder_init_stream",
    "frb_stream_encoder_process_interleaved", "frb_stream_encoder_process", "frb_stream_encoder_finish",
    "frb_stream_encoder_get_state", "frb_stream_encoder_set_verify", "frb_stream_encoder_set_streamable_subset",
    "frb_stream_encoder_set_limit_min_bitrate", "frb_stream_encoder_get_verify",
    "frb_stream_decoder_new", "frb_stream_decoder_delete", "frb_stream_decoder_init_stream", "frb_stream_decoder_init_file",
    "frb_stream_decoder_process_until_end_of_metadata", "frb_stream_decoder_process_until_end_of_stream",
    "frb_stream_decoder_finish", "frb_stream_decoder_get_state", "frb_stream_decoder_get_channels",
    "frb_stream_decoder_get_bits_per_sample", "frb_stream_decoder_get_sample_rate", "frb_stream_decoder_get_blocksize",
    "frb_stream_decoder_get_total_samples",
]


class StreamInfoC(C.Structure):
    _fields_ = [("min_blocksize", C.c_uint32), ("max_blocksize", C.c_uint32), ("min_framesize", C.c_uint32),
                ("max_framesize", C.c_uint32), ("sample_rate", C.c_uint32), ("channels", C.c_uint32),
                ("bits_per_sample", C.c_uint32), ("total_samples", C.c_uint64), ("md5sum", C.c_uint8 * 16)]


class StreamMetadataC(C.Structure):
    _fields_ = [("type", C.c_int), ("is_last", C.c_int), ("length", C.c_uint32), ("stream_info", StreamInfoC)]


class _FrameNumber(C.Union):
    _fields_ = [("frame_number", C.c_uint32), ("sample_number", C.c_uint64)]


class FrameHeaderC(C.Structure):
    _fields_ = [("blocksize", C.c_uint32), ("sample_rate", C.c_uint32), ("channels", C.c_uint32),
                ("channel_assignment", C.c_int), ("bits_per_sample", C.c_uint32), ("number_type", C.c_int),
                ("number", _FrameNumber), ("crc", C.c_uint8)]


class FrameC(C.Structure):
    _fields_ = [("header", FrameHeaderC)]


# callback types of the handle API (include/flacraster_b200.h section 6)
WRITE_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(C.c_uint8), C.c_size_t, C.c_uint32, C.c_uint32, C.c_void_p)
ENC_SEEK_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_uint64, C.c_void_p)
ENC_TELL_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(C.c_uint64), C.c_void_p)
ENC_METADATA_CB = C.CFUNCTYPE(None, C.c_void_p, C.POINTER(StreamMetadataC), C.c_void_p)
DEC_WRITE_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(FrameC), C.POINTER(C.POINTER(C.c_int32)), C.c_void_p)
DEC_METADATA_CB = C.CFUNCTYPE(None, C.c_void_p, C.POINTER(StreamMetadataC), C.c_void_p)
DEC_ERROR_CB = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.c_void_p)
DEC_READ_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(C.c_uint8), C.POINTER(C.c_size_t), C.c_void_p)


def lib():
    """Load the CUDA library (raises if it is not built: no CPU fallback exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(flac_raster_b200 has no CPU fallback)")
    L = C.CDLL(str(LIB_PATH))
    if os.environ.get("FRB_LIB_PATH"):
        # kernel-variant experiments (tools/var_sweep.sh) may load an older build: symbols it lacks resolve to a stub that raises
        class _Tolerant:
            def __init__(self, lib):
                object.__setattr__(self, "_l", lib)

            def __getattr__(self, name):
                try:
                    return getattr(self._l, name)
                except AttributeError:
                    def missing(*a, **k):
                        raise NativeError(ERR_UNSUPPORTED, name, "not exported by the FRB_LIB_PATH variant build")
                    return missing
        L = _Tolerant(L)
    vp, u32, u64, i32, sz = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int, C.c_size_t
    L.frb_version.restype = i32
    L.frb_error_string.restype = C.c_char_p
    L.frb_error_string.argtypes = [i32]
    L.frb_last_cuda_error.restype = C.c_char_p
    L.frb_device_count.argtypes = [C.POINTER(i32)]
    L.frb_launch_count.restype = u64
    L.frb_selftest_crc16.argtypes = [vp, u64, u64, i32, C.POINTER(u32)]
    L.frb_profile_enable.argtypes = [i32]
    L.frb_profile_last_ms.argtypes = [i32, C.POINTER(C.c_float)]
    L.frb_minmax_tiles.argtypes = [vp, i32, u32, u32, u32, vp, u32, vp, vp]
    L.frb_normalize_tiles.argtypes = [vp, i32, u32, u32, u32, vp, u32, vp, i32, vp, vp, vp, sz, vp]
    L.frb_normalize_tiles_i16.argtypes = [vp, i32, u32, u32, u32, vp, u32, vp, vp, vp, vp, sz, vp]
    L.frb_sample_map_workspace_size.argtypes = [u32, C.POINTER(sz)]
    L.frb_denormalize_tiles.argtypes = [vp, vp, vp, u32, vp, C.c_double, vp, i32, u32, u32, u32, vp, sz, vp]
    L.frb_selftest_division.argtypes = [C.c_double, C.c_int64, C.c_int64, C.POINTER(C.c_uint64), vp]
    L.frb_minmax_flat.argtypes = [vp, i32, u64, vp, vp]
    L.frb_normalize_flat.argtypes = [vp, i32, u64, C.c_double, C.c_double, i32, vp, i32, vp]
    L.frb_denormalize_flat.argtypes = [vp, i32, u64, C.c_double, C.c_double, C.c_double, vp, i32, vp]
    L.frb_encode_workspace_size.argtypes = [C.POINTER(EncodeParams), u64, C.POINTER(sz)]
    L.frb_encode_analyse.argtypes = [C.POINTER(EncodeParams), vp, vp, vp, vp, vp, sz, vp, vp, vp]
    L.frb_encode_emit.argtypes = [C.POINTER(EncodeParams), vp, sz, vp, vp, sz, vp, vp]
    L.frb_encode_index.argtypes = [C.POINTER(EncodeParams), vp, sz, vp, vp, vp]
    L.frb_decode_batch_indexed.argtypes = [C.POINTER(DecodeParams), vp, vp, u64, vp, vp, vp, vp, sz, vp, vp]
    L.frb_decode_tiles_indexed.argtypes = [C.POINTER(DecodeParams), vp, vp, u64, vp, vp, vp, vp, C.c_double, vp, C.c_int, u32, u32, u32, vp, sz, vp, vp]
    L.frb_decode_window.argtypes = [C.POINTER(DecodeParams), vp, vp, u64, vp, vp, vp, vp, C.c_double, Tile, vp, C.c_int, vp, sz, vp, vp]
    L.frb_denormalize_window.argtypes = [vp, vp, u32, u32, vp, vp, C.c_double, Tile, vp, C.c_int, u32, vp]
    L.frb_debug_spin.argtypes = [u32, u32, u64, vp]
    L.frb_parse_tile_headers.argtypes = [vp, vp, vp, u32, vp]
    L.frb_gather_seek_index.argtypes = [vp, vp, vp, u32, u32, u32, vp, vp, vp]
    L.frb_decode_workspace_size.argtypes = [C.POINTER(DecodeParams), u64, C.POINTER(sz)]
    L.frb_decode_batch.argtypes = [C.POINTER(DecodeParams), vp, vp, u64, vp, vp, sz, vp, vp]
    L.frb_decode_tiles.argtypes = [C.POINTER(DecodeParams), vp, vp, u64, vp, vp, C.c_double, vp, C.c_int, u32, u32, u32, vp, sz, vp, vp]
    L.frb_small_upload.argtypes = [vp, vp, sz, vp]
    L.frb_small_download.argtypes = [vp, vp, sz, vp]
    L.frb_probe_stream.argtypes = [vp, u64, u64, u32, u32, u32, u32, C.POINTER(u64), C.POINTER(u64), vp]
    L.frb_host_encode.argtypes = [vp, u64, u32, u32, u32, u32, u32, u64, vp, sz, C.POINTER(sz), vp, sz, C.POINTER(sz)]
    L.frb_host_decode.argtypes = [vp, sz, u32, u32, u32, u32, u64, vp, sz, C.POINTER(u64)]
    L.frb_stream_encoder_new.restype = vp
    L.frb_stream_encoder_delete.argtypes = [vp]
    L.frb_stream_encoder_delete.restype = None
    for name in ("channels", "bits_per_sample", "sample_rate", "compression_level", "blocksize"):
        getattr(L, f"frb_stream_encoder_set_{name}").argtypes = [vp, u32]
    L.frb_stream_encoder_set_total_samples_estimate.argtypes = [vp, u64]
    for name in ("verify", "streamable_subset", "limit_min_bitrate"):
        getattr(L, f"frb_stream_encoder_set_{name}").argtypes = [vp, i32]
    L.frb_stream_encoder_init_stream.argtypes = [vp, vp, vp, vp, vp, vp]      # callbacks may be NULL: pass cb_ptr(cb)
    L.frb_stream_encoder_process_interleaved.argtypes = [vp, vp, u32]
    L.frb_stream_encoder_process.argtypes = [vp, vp, u32]
    L.frb_stream_encoder_finish.argtypes = [vp]
    L.frb_stream_encoder_get_state.argtypes = [vp]
    L.frb_stream_encoder_get_verify.argtypes = [vp]
    L.frb_stream_decoder_new.restype = vp
    L.frb_stream_decoder_delete.argtypes = [vp]
    L.frb_stream_decoder_delete.restype = None
    L.frb_stream_decoder_init_stream.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.frb_stream_decoder_init_file.argtypes = [vp, C.c_char_p, vp, vp, vp, vp]
    for name in ("process_until_end_of_metadata", "process_until_end_of_stream", "finish", "get_state"):
        getattr(L, f"frb_stream_decoder_{name}").argtypes = [vp]
    for name in ("get_channels", "get_bits_per_sample", "get_sample_rate", "get_blocksize"):
        getattr(L, f"frb_stream_decoder_{name}").argtypes = [vp]
        getattr(L, f"frb_stream_decoder_{name}").restype = u32
    L.frb_stream_decoder_get_total_samples.argtypes = [vp]
    L.frb_stream_decoder_get_total_samples.restype = u64
    for name in _EXPORTS:
        getattr(L, name)          # AttributeError if a declared symbol is not exported
    _lib = L
    return L


def cb_ptr(cb):
    """A ctypes callback object (or None) as the void* the handle API takes (NULL = callback not given)."""
    return None if cb is None else C.cast(cb, C.c_void_p)


def check(status: int, where: str):
    if status != FRB_OK:
        L = lib()
        detail = L.frb_error_string(status).decode()
        if status == ERR_CUDA:
            detail += ": " + L.frb_last_cuda_error().decode()
        raise NativeError(status, where, detail)


def require_cuda():
    """Fail loudly when there is no usable GPU (there is no CPU path)."""
    n = C.c_int(0)
    st = lib().frb_device_count(C.byref(n))
    if st != FRB_OK or n.value < 1:
        raise NativeError(ERR_NO_DEVICE, "flac_raster_b200", "no CUDA device: the engine has no CPU fallback")
    return n.value


# --------------------------------------------------------------------- host API
def host_encode(samples: np.ndarray, bps: int, sample_rate: int, level: int = 5, blocksize: int = 4096):
    """(N,C) int array (host) -> (frame payload bytes, per-frame sizes uint32[N_frames])."""
    require_cuda()
    a = np.ascontiguousarray(samples)
    if a.ndim == 1:
        a = a.reshape(-1, 1)
    if a.dtype != np.int32:
        a = a.astype(np.int32)
    n, ch = a.shape
    nf = (n + blocksize - 1) // blocksize
    cap = n * ch * 5 + nf * 64 + 4096
    out = np.empty(cap, dtype=np.uint8)
    fs = np.empty(max(nf, 1), dtype=np.uint32)
    ob, got = C.c_size_t(0), C.c_size_t(0)
    st = lib().frb_host_encode(a.ctypes.data, n, ch, bps, sample_rate, level, blocksize, 0,
                               out.ctypes.data, cap, C.byref(ob), fs.ctypes.data, fs.size, C.byref(got))
    check(st, "frb_host_encode")
    return out[:ob.value], fs[:got.value]


def host_decode(frames: bytes | np.ndarray, channels: int, bps: int, blocksize: int, sample_rate: int,
                n_samples: int = 0) -> np.ndarray:
    """Frame bytes of one stream (host) -> (N,C) int32 samples."""
    require_cuda()
    b = np.frombuffer(frames, dtype=np.uint8) if not isinstance(frames, np.ndarray) else frames
    ns = C.c_uint64(0)
    L = lib()
    if n_samples == 0:
        st = L.frb_host_decode(b.ctypes.data, b.size, channels, bps, blocksize, sample_rate, 0, None, 0, C.byref(ns))
        check(st, "frb_host_decode(probe)")
        n_samples = ns.value
    out = np.empty((n_samples, channels), dtype=np.int32)
    st = L.frb_host_decode(b.ctypes.data, b.size, channels, bps, blocksize, sample_rate, n_samples,
                           out.ctypes.data, out.size, C.byref(ns))
    check(st, "frb_host_decode")
    return out
