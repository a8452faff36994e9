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
from flac_raster_b200 import flacfmt  # noqa: E402
from oracle import ffmpeg_flac as ff, flac_oracle as fo  # noqa: E402


def md5_samples(x: np.ndarray) -> str:
    return hashlib.md5(np.ascontiguousarray(x, dtype="<i4").tobytes()).hexdigest()


def record(stream: bytes, x: np.ndarray) -> dict:
    out = ff.decode_bytes(stream, x.shape[1])
    assert np.array_equal(out, x), "FFmpeg does not decode the stream to its input"
    return {"stream_md5": hashlib.md5(stream).hexdigest(), "decoded_md5": md5_samples(out)}


def main():
    if not ff.available():
        sys.exit("the bundled FFmpeg libraries are not installed")
    fo.build()
    res = {"decoder": "FFmpeg libavcodec flac (" + ", ".join(sorted(Path(p._name).name for p in ff._load())) + ")",
           "oracle_level5": {}, "gpu_level8": {}}
    for name, (x, bps) in signal_cases().items():
        if name == "tiny3":
            continue
        enc, _ = fo.encode(x, bps, 48000, 5, finalize=True)
        res["oracle_level5"][name] = record(enc, x)
        enc8, fs8 = fo.encode(x, bps, 48000, 8, mid_side=(bps == 16))
        frames = enc8[len(enc8) - int(fs8.sum()):]
        si = flacfmt.StreamInfo(4096, 4096, 0, 0, 48000, x.shape[1], bps, x.shape[0])
        res["gpu_level8"][name] = record(flacfmt.build_header(si) + frames, x)
    dst = Path(__file__).with_name("ffmpeg_decoded.json")
    dst.write_text(json.dumps(res, indent=1) + "\n")
    print("wrote", dst, dst.stat().st_size, "bytes")


if __name__ == "__main__":
    main()
