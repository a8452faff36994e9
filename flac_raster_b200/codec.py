"""pyflac-shaped codec objects backed by the CUDA engine (the plugin seam of the reference).

The reference touches pyflac in exactly two ways:
  * pyflac.StreamEncoder(write_callback=, sample_rate=, compression_level=, blocksize=)
    .process(samples) / .finish()            converter.py:139-154, spatial_encoder.py:291-304
  * pyflac.FileDecoder(path).process() -> (audio, sample_rate)     converter.py:181-182
These classes keep pyflac 3.0.0's constructor/method signatures, exceptions and
callback contract (docs/sonos-pyflac.txt:1881-2378, :1326-1877): header chunks
first with num_samples == 0, then one callback per frame with
num_samples == blocksize and current_frame == frame index.
"""
from __future__ import annotations

from pathlib import Path
from typing import Callable, Optional, Tuple

import numpy as np

from . import _native as nat
from . import flacfmt


class EncoderInitException(Exception):
    """docs/sonos-pyflac.txt:1909-1938"""

    def __init__(self, code):
        self.code = code
        super().__init__(f"FLAC encoder failed to initialise (code {code})")


class EncoderProcessException(Exception):
    pass


class DecoderInitException(Exception):
    def __init__(self, code):
        self.code = code
        super().__init__(f"FLAC decoder failed to initialise (code {code})")


class DecoderProcessException(Exception):
    pass


class StreamEncoder:
    """Same surface as pyflac.StreamEncoder (docs/sonos-pyflac.txt:2175-2198)."""

    def __init__(self,
                 sample_rate: int,
                 write_callback: Callable[[bytes, int, int, int], None],
                 seek_callback: Callable[[int], None] = None,
                 tell_callback: Callable[[], int] = None,
                 metadata_callback: Callable[[int], None] = None,
                 compression_level: int = 5,
                 blocksize: int = 0,
                 streamable_subset: bool = True,
                 verify: bool = False,
                 limit_min_bitrate: bool = False):
        self.write_callback = write_callback
        self.seek_callback = seek_callback
        self.tell_callback = tell_callback
        self.metadata_callback = metadata_callback
        self._sample_rate = int(sample_rate)
        self._compression_level = int(compression_level)
        self._blocksize = int(blocksize)
        self._streamable_subset = streamable_subset
        self._verify = verify
        self._limit_min_bitrate = limit_min_bitrate
        # attributes the reference assigns (converter.py:147-148); overwritten on first process()
        self._channels = 0
        self._bits_per_sample = 0
        self._initialised = False
        self._pending = []
        self._frames_out = 0

    # -- pyflac derives channels/bps from the first array (docs/sonos-pyflac.txt:1986-1992)
    def _init(self):
        if not (0 <= self._compression_level <= 8):
            self._compression_level = 8 if self._compression_level > 8 else 0
        # blocksize 0 (pyflac's default) follows libFLAC's init_stream: 1152 for the presets without LPC (levels 0-2,
        # max_lpc_order == 0), 4096 otherwise
        bs = self._blocksize or (1152 if self._compression_level <= 2 else 4096)
        if not (16 <= bs <= 4096):
            raise EncoderInitException("FLAC__STREAM_ENCODER_INIT_STATUS_INVALID_BLOCK_SIZE")
        if not (1 <= self._channels <= 8):
            raise EncoderInitException("FLAC__STREAM_ENCODER_INIT_STATUS_INVALID_NUMBER_OF_CHANNELS")
        if self._bits_per_sample not in (16, 32):
            raise EncoderInitException("FLAC__STREAM_ENCODER_INIT_STATUS_INVALID_BITS_PER_SAMPLE")
        if not (0 < self._sample_rate <= 1048575):
            raise EncoderInitException("FLAC__STREAM_ENCODER_INIT_STATUS_INVALID_SAMPLE_RATE")
        self._blocksize = bs
        # libFLAC emits the stream header through the write callback right away
        # ("fLaC", STREAMINFO, VORBIS_COMMENT(vendor)); STREAMINFO stays unfinalised
        # because no seek callback is given (reference files: total_samples == 0).
        si = flacfmt.StreamInfo(bs, bs, 0, 0, self._sample_rate, self._channels, self._bits_per_sample, 0)
        hdr = flacfmt.build_header(si)
        for chunk in (hdr[:4], hdr[4:42], hdr[42:]):
            self.write_callback(chunk, len(chunk), 0, 0)
        self._initialised = True

    def process(self, samples: np.ndarray):
        if not isinstance(samples, np.ndarray):
            raise TypeError("Processing only supports numpy arrays")
        if samples.ndim == 1:
            samples = samples.reshape(-1, 1)
        if not self._initialised:
            self._channels = samples.shape[1]
            self._bits_per_sample = samples.dtype.itemsize * 8
            self._init()
        elif samples.shape[1] != self._channels:
            raise EncoderProcessException("FLAC__STREAM_ENCODER_CLIENT_ERROR")
        self._pending.append(np.ascontiguousarray(samples).astype(np.int32))

    def finish(self) -> bool:
        if not self._initialised:
            return False
        ok = True
        if self._pending:
            x = self._pending[0] if len(self._pending) == 1 else np.concatenate(self._pending, axis=0)
            self._pending = []
            if x.shape[0]:
                try:
                    payload, fsizes = nat.host_encode(x, self._bits_per_sample, self._sample_rate,
                                                      self._compression_level, self._blocksize)
                except nat.NativeError as e:
                    raise EncoderProcessException(str(e)) from e
                if self._verify:
                    # libFLAC's verify mode (FLAC__stream_encoder_set_verify, docs/sonos-pyflac.txt:6810-6824): decode the
                    # frames just produced -- on the GPU decoder -- and compare them with the input samples
                    try:
                        back = nat.host_decode(payload, self._channels, self._bits_per_sample, self._blocksize,
                                               self._sample_rate, x.shape[0])
                    except nat.NativeError as e:
                        raise EncoderProcessException("FLAC__STREAM_ENCODER_VERIFY_DECODER_ERROR: " + str(e)) from e
                    if not np.array_equal(back, x):
                        raise EncoderProcessException("FLAC__STREAM_ENCODER_VERIFY_MISMATCH_IN_AUDIO_DATA")
                mv = memoryview(payload)
                off = 0
                n = x.shape[0]
                for f, sz in enumerate(fsizes):
                    sz = int(sz)
                    nsamp = min(self._blocksize, n - f * self._blocksize)
                    self.write_callback(bytes(mv[off:off + sz]), sz, nsamp, f)
                    off += sz
        self._initialised = False
        return ok


class FileDecoder:
    """Same surface as pyflac.FileDecoder (docs/sonos-pyflac.txt:1584-1640).

    process() returns (samples, sample_rate).  pyflac returns float64 in [-1,1)
    after a PCM_16 WAV round trip (SURVEY Q3); pass compat_pyflac_float=True to
    reproduce that, default is the exact integer samples (int16 for 16-bps
    streams, int32 otherwise) -- what the reference's denormalize_from_audio
    documents as its integer path.
    """

    def __init__(self, input_file, output_file=None, compat_pyflac_float: bool = False):
        self._path = Path(input_file)
        self._output_file = output_file
        self._compat = compat_pyflac_float
        if not self._path.exists():
            raise DecoderInitException("FLAC__STREAM_DECODER_INIT_STATUS_ERROR_OPENING_FILE")
        self.header: Optional[flacfmt.FlacHeader] = None

    def process(self) -> Tuple[np.ndarray, int]:
        data = self._path.read_bytes()
        try:
            audio, hdr = decode_bytes(data)
        except (ValueError, nat.NativeError) as e:
            raise DecoderProcessException(str(e)) from e
        self.header = hdr
        si = hdr.streaminfo
        if self._compat:
            if si.bits_per_sample == 16:
                out = audio.astype(np.float64) / 32768.0
            else:
                out = (audio >> 16).astype(np.float64) / 32768.0
            return out, si.sample_rate
        if si.bits_per_sample == 16:
            return audio.astype(np.int16), si.sample_rate
        return audio, si.sample_rate


def decode_bytes(data: bytes, n_samples: int = 0):
    """One complete FLAC stream in memory -> ((N,C) int32 samples, FlacHeader)."""
    hdr = flacfmt.parse_header(data)
    si = hdr.streaminfo
    if si.bits_per_sample not in (8, 12, 16, 20, 24, 32):
        raise ValueError(f"unsupported bits per sample {si.bits_per_sample}")
    if si.min_blocksize != si.max_blocksize and si.total_samples > si.max_blocksize:
        raise ValueError("variable-blocksize FLAC streams are not supported")
    frames = np.frombuffer(data, dtype=np.uint8, offset=hdr.first_frame_offset)
    # legacy --spatial files concatenate streams: stop at the next "fLaC" marker
    n = n_samples or si.total_samples
    audio = nat.host_decode(frames, si.channels, si.bits_per_sample, si.max_blocksize, si.sample_rate, n)
    return audio, hdr
