"""GPU suite (-m gpu): the warp-per-subframe statistics kernel against the CTA kernel it replaces for 16-bit subframes.

FRB_STATS_CTA=1 selects the CTA kernel (k_enc_stats + k_enc_fixed) for every subframe; the setting is read once per process, so
each variant encodes in a subprocess of its own.  Both must produce the same bytes, frame sizes and subframe bit offsets: the
warp kernel forms every partial sum of the CTA kernel in the same order, and applies the wasted-bits shift afterwards.
The inputs reach its special cases: wasted bits (from 1 to 15), constant and all-zero subframes, near-pure tones (Levinson
is sensitive to the last bit of the autocorrelation), channels that start 8-byte but not 16-byte aligned, int32 audio and
two-channel mid/side streams (whose 17-bit side channel stays on the CTA kernel).
"""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parents[1]
LEVELS = [0, 3, 5, 6, 8]

CHILD = r"""
import sys
import numpy as np
import torch
sys.path.insert(0, sys.argv[1])
from flac_raster_b200.engine import Engine

BS = 4096


def signals(channels, seed):
    # per stream (n_samples, audio_base): 3 full frames + a tail, bases at 4 mod 8 samples (8-byte, not 16-byte aligned)
    rng = np.random.default_rng(seed)
    layout = [(3 * BS + 4, 4), (2 * BS, 0), (4 * BS + 1, 12)]
    streams = []
    for k, (n, _) in enumerate(layout):
        t = np.arange(n)
        chans = []
        for c in range(channels):
            kind = (k * channels + c) % 6
            if kind == 0:      # tone and noise
                x = 9000 * np.sin(2 * np.pi * t * (0.003 + 0.001 * c)) + rng.normal(0, 40, n)
            elif kind == 1:    # near-pure tone
                x = 30000 * np.sin(2 * np.pi * t * 0.0021 + 0.3 * c)
            elif kind == 2:    # wasted bits: 3 in the first frame, 1 in the second, 15 later
                x = rng.integers(-500, 500, n)
                x[:BS] <<= 3
                x[BS:2 * BS] <<= 1
                x[2 * BS:] = np.where(rng.random(n - 2 * BS) < 0.5, -32768, 0)
            elif kind == 3:    # constant frame, all-zero frame, then a slow ramp
                x = np.full(n, 1234.0)
                x[BS:2 * BS] = 0
                x[2 * BS:] = (t[2 * BS:] // 7) % 3000 - 1500
            elif kind == 4:    # full-scale noise
                x = rng.integers(-32768, 32768, n)
            else:              # low-amplitude noise with a step
                x = rng.integers(-3, 4, n) + np.where(t > n // 2, 20000, -20000)
            chans.append(np.clip(np.round(x), -32768, 32767).astype(np.int16))
        streams.append(np.stack(chans))
    return layout, streams


def run(eng, channels, level, i16, seed):
    layout, streams = signals(channels, seed)
    bases, total = [], 0
    for (n, pad), s in zip(layout, streams):
        total += pad
        bases.append(total)
        total += channels * n
    buf = np.zeros(total + 8, dtype=np.int16 if i16 else np.int32)
    for b, (n, _), s in zip(bases, layout, streams):
        buf[b:b + channels * n] = s.reshape(-1)
    audio = torch.from_numpy(buf).cuda()
    ns = np.array([n for n, _ in layout], dtype=np.int64)
    payload, offs, sizes, fb, sb = eng.encode_audio(audio, ns, np.array(bases, dtype=np.int64), np.full(len(ns), 44100),
                                                    channels, 16, level)
    torch.cuda.synchronize()
    return payload.cpu().numpy().copy(), sizes, fb.cpu().numpy().copy(), sb.cpu().numpy().copy()


eng = Engine(0)
out = {}
for level in [int(v) for v in sys.argv[3].split(",")]:
    for channels, i16 in ((1, True), (3, True), (8, True), (2, True), (2, False), (5, False)):
        key = f"l{level}_c{channels}_{'i16' if i16 else 'i32'}"
        p, s, f, b = run(eng, channels, level, i16, 1000 * level + 10 * channels + int(i16))
        out[key + "_payload"], out[key + "_sizes"], out[key + "_frame_bytes"], out[key + "_sub_bitoff"] = p, s, f, b
np.savez(sys.argv[2], **out)
"""


def _encode(tmp_path, name, cta):
    env = dict(os.environ)
    env.pop("FRB_STATS_CTA", None)
    if cta:
        env["FRB_STATS_CTA"] = "1"
    out = tmp_path / f"{name}.npz"
    subprocess.run([sys.executable, "-c", CHILD, str(ROOT), str(out), ",".join(map(str, LEVELS))], env=env, check=True,
                   timeout=600)
    return np.load(out)


def test_warp_stats_match_cta_stats(tmp_path):
    warp = _encode(tmp_path, "warp", cta=False)
    cta = _encode(tmp_path, "cta", cta=True)
    assert sorted(warp.files) == sorted(cta.files)
    assert len(warp.files) == 4 * 6 * len(LEVELS)
    for k in sorted(warp.files):
        assert np.array_equal(warp[k], cta[k]), f"{k}: warp-per-subframe statistics change the encoding"
