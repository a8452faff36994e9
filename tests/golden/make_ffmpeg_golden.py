"""Generate tests/golden/ffmpeg_decoded.json: the streams FFmpeg's libavcodec FLAC decoder accepted.

Needs the FFmpeg libraries that opencv-python-headless bundles (oracle/ffmpeg_flac.py):
    python tests/golden/make_ffmpeg_golden.py
For every case of conftest.signal_cases (tiny3 excepted: FFmpeg refuses blocksize < 16) it encodes the
streams the two FFmpeg tests check with the C oracle, has FFmpeg decode them, requires the input samples
back, and records the md5 of each stream and of FFmpeg's int32 output.  A test that produces a stream with
the same md5 produces a stream this FFmpeg decoded to those samples, with or without FFmpeg installed.
  oracle_level5: oracle.encode(x, bps, 48000, 5, finalize=True), the whole file
  gpu_level8:    flacfmt.build_header(StreamInfo(..., 48000, ch, bps, n)) + the level-8 frames that
                 nat.host_encode must emit (byte-identical to the oracle's, mid/side for 16-bit input)
  oracle_stream_params: oracle.encode(x, bits, rate, level, blocksize=B, finalize=True) over stream_param_cases(), a
                 subset of tests/test_gpu_stream_params.py's parameters: blocksizes 192-65535, full-range 8- to 24-bit
                 audio, 1, 2 and 8 channels, rates with every kind of header code.  FFmpeg hands 8- to 16-bit audio out
                 as s16 and wider audio as s32, shifted left to the top bits; ffmpeg_samples() shifts it back.  A stream
                 FFmpeg refuses, or decodes to anything but its input, is left out (and printed): the CPU test only
                 holds the oracle to the streams recorded here.
"""
import hashlib
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

from conftest import signal_cases  # noqa: E402
from test_gpu_stream_params import full_range  # noqa: E402
from flac_raster_b200 import flacfmt  # noqa: E402
from oracle import ffmpeg_flac as ff, flac_oracle as fo  # noqa: E402


def md5_samples(x: np.ndarray) -> str:
    return hashlib.md5(np.ascontiguousarray(x, dtype="<i4").tobytes()).hexdigest()


def record(stream: bytes, x: np.ndarray) -> dict:
    out = ff.decode_bytes(stream, x.shape[1])
    assert np.array_equal(out, x), "FFmpeg does not decode the stream to its input"
    return {"stream_md5": hashlib.md5(stream).hexdigest(), "decoded_md5": md5_samples(out)}


def stream_param_cases():
    """(name, (x, bits, rate, level, blocksize)) of the oracle_stream_params section."""
    blocksizes = [192, 576, 1000, 1152, 2304, 4095, 4608, 16384, 65535]
    rates = [8000, 37800, 44100, 65535, 655350, 700001, 1048575, 96000]
    for j, B in enumerate(blocksizes):
        for q, bits in enumerate([8, 10, 12, 16, 18, 20, 24]):
            if (j + q) % 2:
                continue
            rate, ch, level = rates[(j + q) % len(rates)], [1, 2, 8][(j + 2 * q) % 3], [0, 5, 8][(j + q) % 3]
            x = full_range(2 * B + B // 3 + 1, ch, bits, seed=1000 + 10 * j + q)
            yield f"b{B}_s{bits}_r{rate}_c{ch}_l{level}", (x, bits, rate, level, B)


def ffmpeg_samples(stream: bytes, channels: int, bits: int) -> np.ndarray:
    """FFmpeg's decode of the stream as the integer samples: its s16 / s32 output carries them in the top bits."""
    out = ff.decode_bytes(stream, channels)
    shift = (16 if bits <= 16 else 32) - bits
    assert not (out & ((1 << shift) - 1)).any()
    return out >> shift


def main():
    if not ff.available():
        sys.exit("the bundled FFmpeg libraries are not installed")
    fo.build()
    res = {"decoder": "FFmpeg libavcodec flac (" + ", ".join(sorted(Path(p._name).name for p in ff._load())) + ")",
           "oracle_level5": {}, "gpu_level8": {}, "oracle_stream_params": {}}
    for name, (x, bps) in signal_cases().items():
        if name == "tiny3":
            continue
        enc, _ = fo.encode(x, bps, 48000, 5, finalize=True)
        res["oracle_level5"][name] = record(enc, x)
        enc8, fs8 = fo.encode(x, bps, 48000, 8, mid_side=(bps == 16))
        frames = enc8[len(enc8) - int(fs8.sum()):]
        si = flacfmt.StreamInfo(4096, 4096, 0, 0, 48000, x.shape[1], bps, x.shape[0])
        res["gpu_level8"][name] = record(flacfmt.build_header(si) + frames, x)
    for name, (x, bits, rate, level, B) in stream_param_cases():
        enc, _ = fo.encode(x, bits, rate, level, blocksize=B, finalize=True)
        try:
            ok = np.array_equal(ffmpeg_samples(enc, x.shape[1], bits), x)
        except (ValueError, AssertionError) as e:
            ok = False
            print("FFmpeg refuses", name, e)
        if not ok:
            # this FFmpeg build hands back no samples at all for the 8-channel 20- and 24-bit streams at blocksizes 16384
            # and 65535 (frames of several hundred kilobytes); the oracle's own decoder reads them back exactly
            print("left out (FFmpeg does not give the input back):", name)
            continue
        res["oracle_stream_params"][name] = {"stream_md5": hashlib.md5(enc).hexdigest(), "decoded_md5": md5_samples(x)}
    dst = Path(__file__).with_name("ffmpeg_decoded.json")
    dst.write_text(json.dumps(res, indent=1) + "\n")
    print("wrote", dst, dst.stat().st_size, "bytes")


if __name__ == "__main__":
    main()
