"""GPU parity suite (-m gpu): the CUDA path through the C ABI vs the oracle and the golden fixtures."""
import json
import os
import struct

import numpy as np
import pytest

from conftest import GOLDEN, signal_cases

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def nat():
    from flac_raster_b200 import _native
    _native.require_cuda()
    return _native


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available()
    return torch


def _full_stream(payload, x, bps, rate):
    from flac_raster_b200 import flacfmt
    si = flacfmt.StreamInfo(4096, 4096, 0, 0, rate, x.shape[1], bps, x.shape[0])
    return flacfmt.build_header(si) + bytes(payload)


# ------------------------------------------------------------------ sample mapping
def test_normalize_kernels_match_reference_vectors(nat, torch_cuda):
    """Bit-identical to the real reference module's outputs for all 8 dtypes, NaN, constant arrays."""
    from flac_raster_b200 import NormalizationParams, denormalize_from_audio, normalize_to_audio
    z = np.load(GOLDEN / "normalization_vectors.npz")
    keys = sorted(set(k.rsplit("__", 1)[0] for k in z.files if k.endswith("__in")))
    for k in keys:
        x, a, b, p = z[k + "__in"], z[k + "__audio"], z[k + "__back"], z[k + "__params"]
        audio, params = normalize_to_audio(x.reshape(-1, 3), int(p[2]))
        assert audio.dtype == a.dtype and np.array_equal(audio, a), k
        assert params.scale_factor == int(p[3]) and params.original_dtype == str(x.dtype)
        assert params.data_min == p[0] or (np.isnan(params.data_min) and np.isnan(p[0]))
        assert params.data_max == p[1] or (np.isnan(params.data_max) and np.isnan(p[1]))
        back = denormalize_from_audio(audio, params)
        assert back.dtype == b.dtype and np.array_equal(back, b, equal_nan=True), k


def test_normalize_large_random_vs_oracle(nat, torch_cuda):
    from flac_raster_b200 import denormalize_from_audio, normalize_to_audio
    from oracle import normalization_oracle as no
    rng = np.random.default_rng(3)
    for dt, bits in (("uint16", 16), ("int16", 16), ("float32", 24), ("int32", 24), ("uint8", 16), ("float64", 24)):
        if dt.startswith("float"):
            x = (rng.standard_normal((700, 1031)) * 1e3).astype(dt)
            x[5, 7] = np.nan
            x[9, 9] = np.inf if dt == "float64" else x[9, 9]
        else:
            info = np.iinfo(dt)
            x = rng.integers(info.min, info.max, size=(700, 1031), endpoint=True).astype(dt)
        a, p = normalize_to_audio(x, bits)
        a2, p2 = no.normalize_to_audio(x, bits)
        assert np.array_equal(a, a2) and p.data_min == p2["data_min"] and p.data_max == p2["data_max"], dt
        if not np.isinf(p.data_max):
            b = denormalize_from_audio(a, p)
            b2 = no.denormalize_from_audio(a2, p2["data_min"], p2["data_max"], dt, p2["scale_factor"])
            assert np.array_equal(b, b2, equal_nan=True), dt
    # explicit min/max override and the float (pyflac WAV) branch of denormalize
    x = rng.integers(0, 4000, size=5000).astype(np.uint16)
    a, p = normalize_to_audio(x, 16, data_min=0.0, data_max=11672.0)
    a2, _ = no.normalize_to_audio(x, 16, 0.0, 11672.0)
    assert np.array_equal(a, a2)
    f = a.astype(np.float64) / 32768.0
    assert np.array_equal(denormalize_from_audio(f, p), no.denormalize_from_audio(f, 0.0, 11672.0, "uint16", 32767))


# ------------------------------------------------------------------ decode
def test_decode_reference_goldens(nat, oracle):
    """Reference-encoded files decode bit-exactly through the GPU decoder (north_star part 2)."""
    from flac_raster_b200 import flacfmt
    data = (GOLDEN / "sample_rgb.flac").read_bytes()
    hdr = flacfmt.parse_header(data)
    ref, _ = oracle.decode(data)
    si = hdr.streaminfo
    for hint in (65536, 0):           # with and without the sample count (STREAMINFO total is 0 in reference files)
        out = nat.host_decode(data[hdr.first_frame_offset:], si.channels, si.bits_per_sample, si.max_blocksize, si.sample_rate, hint)
        assert np.array_equal(out, ref)
    data = (GOLDEN / "sample_dem.flac").read_bytes()
    pos = 0
    while pos < len(data):
        ref, info = oracle.decode(data[pos:])
        h = flacfmt.parse_header(data[pos:])
        seg = data[pos + h.first_frame_offset: pos + int(info.bytes_consumed)]
        out = nat.host_decode(seg, 1, 32, 4096, 44100, 0)
        assert np.array_equal(out, ref)
        pos += int(info.bytes_consumed)


@pytest.mark.parametrize("level", [0, 5, 8])
def test_decode_oracle_encoded_streams(nat, oracle, level):
    from flac_raster_b200 import flacfmt
    for name, (x, bps) in signal_cases().items():
        enc, _ = oracle.encode(x, bps, 48000, level)
        h = flacfmt.parse_header(enc)
        out = nat.host_decode(enc[h.first_frame_offset:], x.shape[1], bps, 4096, 48000, x.shape[0])
        assert np.array_equal(out, x), (name, level)


def test_decode_survives_a_false_frame_header_before_the_real_one(nat, oracle):
    """The scan path keeps the two earliest header candidates per frame number and drops a first candidate that lies at or
    before the previous frame's (frb_decode.cuh k_sync_resolve): bytes that look like frame k's header (sync code, matching
    fields, correct CRC-8) placed ahead of the real frame must not shadow it.  libFLAC never sees such bytes (it walks the
    frames in order); the keep-the-first scan of round 1 reported a malformed stream here."""
    from flac_raster_b200 import flacfmt
    for case, ch in (("sine16_1ch", 1), ("smooth16_8ch", 8)):
        x, bps = signal_cases()[case]
        enc, fsz = oracle.encode(x, bps, 44100, 5)
        off = flacfmt.parse_header(enc).first_frame_offset
        frames = enc[off:]
        starts = np.concatenate([[0], np.cumsum(fsz)]).astype(np.int64)
        assert len(fsz) >= 3
        for k in (1, len(fsz) - 2):
            fake = frames[starts[k]:starts[k] + 16]                 # frame k's own header (CRC-8 included) + a few payload bytes
            got = nat.host_decode(fake + frames, ch, bps, 4096, 44100, x.shape[0])
            assert np.array_equal(got, x), (case, k)


def test_decode_detects_corruption(nat, oracle):
    x, bps = signal_cases()["sine16_1ch"]
    enc, _ = oracle.encode(x, bps, 44100, 5)
    from flac_raster_b200 import flacfmt
    off = flacfmt.parse_header(enc).first_frame_offset
    bad = bytearray(enc[off:])
    bad[len(bad) // 2] ^= 0x04
    with pytest.raises(nat.NativeError) as ei:
        nat.host_decode(bytes(bad), 1, 16, 4096, 44100, x.shape[0])
    assert ei.value.status in (nat.ERR_CRC, nat.ERR_BAD_STREAM)
    with pytest.raises(nat.NativeError):                      # truncated stream: frames missing
        nat.host_decode(bytes(enc[off:off + 3000]), 1, 16, 4096, 44100, x.shape[0])


def test_decode_handcrafted_stream_big_orders_rice2_escapes(nat, oracle, torch_cuda):
    """Syntax no libFLAC preset emits, written by tests/flac_handcraft.py and checked against the oracle decoder first:
    LPC orders 20, 32 and 13 (the > 12 kernel instantiation and the automatic rerun), Rice2 parameters, an escape-coded
    partition, partition orders 3/0/2, a short last frame with a 16-bit blocksize field.  Decoded through the host API and
    through the fused decode-to-raster launch."""
    torch = torch_cuda
    import flac_handcraft as hc
    from flac_raster_b200 import flacfmt, _native as natmod
    from flac_raster_b200.engine import default_engine
    from oracle import normalization_oracle as no
    rng = np.random.default_rng(4)
    n_total, bs = 4096 * 2 + 1000, 4096
    t = np.arange(n_total)
    x = (9000 * np.sin(t / 40.0) + 3000 * np.sin(t / 7.3) + rng.integers(-40, 40, size=n_total)).astype(np.int64)
    frames = b""
    for f, a in enumerate(range(0, n_total, bs)):
        order = [20, 32, 13][f]
        coefs = rng.integers(-300, 300, size=order); coefs[0] = 1900; coefs[1] = -900
        frames += hc.frame(x[a:a + bs], 16, 9, f, bs, oracle.crc8, oracle.crc16, order=order, coefs=coefs, shift=10, precision=12,
                           partition_order=[3, 0, 2][f], rice2=(f == 1), escape_partitions=((2,) if f == 0 else ()))
    si = flacfmt.StreamInfo(bs, bs, 0, 0, 44100, 1, 16, n_total)
    ref, _ = oracle.decode(flacfmt.build_header(si) + frames)
    assert np.array_equal(ref[:, 0], x)
    got = nat.host_decode(frames, 1, 16, bs, 44100, n_total)
    assert np.array_equal(got[:, 0], x)
    # the same frames as one "tile" of 8 x 1149 pixels, straight into an int16 raster
    eng = default_engine()
    data = torch.cat([torch.from_numpy(np.frombuffer(frames, dtype=np.uint8).copy()), torch.zeros(64, dtype=torch.uint8)]).cuda()
    tiles = np.zeros(1, dtype=natmod.TILE_DTYPE)
    tiles[0] = (0, 0, 8, 1149)
    mn, mx = -12345.0, 20000.0
    out = torch.zeros(1, 8, 1149, dtype=torch.int16, device="cuda")
    st = eng.decode_tiles(data, np.array([0]), np.array([len(frames)]), tiles, np.array([44100], dtype=np.uint32),
                          np.array([[mn, mx]]), 32767.0, out, 16, bs, fused=True)
    assert list(st[:3]) == [0, 0, 0] and st[4] == 0, st
    want = no.denormalize_from_audio(x.astype(np.int16), mn, mx, "int16", 32767.0).reshape(8, 1149)
    assert np.array_equal(out.cpu().numpy()[0], want)


def test_decode_handcrafted_multichannel_skim_paths(nat, oracle):
    """Three-channel frames whose FIRST subframes hold what the skim walk has to step over without decoding it: escape-coded
    partitions (raw words), Rice2 parameters, LPC order 32 warm-up and coefficient blocks, partition order 5."""
    import flac_handcraft as hc
    from flac_raster_b200 import flacfmt
    rng = np.random.default_rng(8)
    n_total, bs = 4096 * 3, 4096
    t = np.arange(n_total)
    x = np.stack([(7000 * np.sin(t / (23.0 + 9 * c)) + rng.integers(-60, 60, size=n_total)).astype(np.int64) for c in range(3)], axis=1)
    x[5000:5200, 1] = rng.integers(-30000, 30000, size=200)          # a burst: long codes in one partition
    frames = b""
    for f, a in enumerate(range(0, n_total, bs)):
        subs = []
        for c in range(3):
            order = [[32, 4, 8], [13, 20, 2], [8, 8, 31]][f][c]
            coefs = rng.integers(-200, 200, size=order); coefs[0] = 1800; 
            if order > 1: coefs[1] = -800
            subs.append(dict(order=order, coefs=coefs, shift=10, precision=12, partition_order=[5, 2, 0][c],
                             rice2=(c == 1), escape_partitions=((0, 3) if (c + f) % 2 == 0 and c < 2 else ())))
        frames += hc.frame(x[a:a + bs], 16, 9, f, bs, oracle.crc8, oracle.crc16, subs=subs)
    si = flacfmt.StreamInfo(bs, bs, 0, 0, 44100, 3, 16, n_total)
    ref, _ = oracle.decode(flacfmt.build_header(si) + frames)
    assert np.array_equal(ref, x)
    got = nat.host_decode(frames, 3, 16, bs, 44100, n_total)
    assert np.array_equal(got, x)


def test_decode_fuzzed_multichannel_streams_fail_cleanly(nat, oracle):
    """Random single-byte damage anywhere in an 8-channel stream (frame headers, subframe headers, Rice data, CRC bytes):
    the fused skim + decode launch must come back promptly with CRC / malformed-stream status -- never hang on an offset
    that is no longer published, never return damaged samples as good."""
    x, bps = signal_cases()["smooth16_8ch"]
    enc, _ = oracle.encode(x, bps, 44100, 5)
    from flac_raster_b200 import flacfmt
    off = flacfmt.parse_header(enc).first_frame_offset
    good = bytearray(enc[off:])
    assert np.array_equal(nat.host_decode(bytes(good), 8, 16, 4096, 44100, x.shape[0]), x)
    rng = np.random.default_rng(99)
    for trial in range(24):
        bad = bytearray(good)
        pos = int(rng.integers(0, len(bad)))
        bad[pos] ^= int(rng.integers(1, 256))
        if trial % 6 == 5:                                   # also a burst: a run of zero bytes (long unary runs)
            bad[pos:pos + 64] = bytes(min(64, len(bad) - pos))
        with pytest.raises(nat.NativeError) as ei:
            nat.host_decode(bytes(bad), 8, 16, 4096, 44100, x.shape[0])
        assert ei.value.status in (nat.ERR_CRC, nat.ERR_BAD_STREAM), (trial, pos, ei.value.status)
    assert np.array_equal(nat.host_decode(bytes(good), 8, 16, 4096, 44100, x.shape[0]), x)   # and the engine is still healthy


def test_stream_encoder_verify_mode(nat):
    """pyflac's verify=True (libFLAC set_verify): the shim decodes its own frames on the GPU and compares."""
    from flac_raster_b200 import codec
    x = signal_cases()["stereo16_corr"][0].astype(np.int16)
    chunks = []
    enc = codec.StreamEncoder(44100, lambda b, n, s, f: chunks.append(bytes(b)), compression_level=5, blocksize=4096, verify=True)
    enc.process(x)
    assert enc.finish() is True
    assert len(chunks) == 3 + (x.shape[0] + 4095) // 4096


# ------------------------------------------------------------------ encode
@pytest.mark.parametrize("level", [0, 1, 2, 3, 4, 5, 6, 7, 8])
def test_encode_matches_oracle_and_roundtrips(nat, oracle, level):
    """GPU frames: decoded bit-exactly by the oracle decoder, byte-identical to the libFLAC-procedure
    oracle encoder, and (as a size gate) never more than 1 % larger."""
    for name, (x, bps) in signal_cases().items():
        payload, fs = nat.host_encode(x, bps, 44100, level)
        assert int(fs.sum()) == len(payload)
        dec, info = oracle.decode(_full_stream(payload, x, bps, 44100))
        assert np.array_equal(dec, x), (name, level)
        # two-channel input: libFLAC's mid/side search runs on the GPU for 16-bit streams; 32-bit ones would need a
        # 33-bit side channel and are coded as independent channels (DESIGN.md section 2)
        oenc, ofs = oracle.encode(x, bps, 44100, level, mid_side=(bps == 16))
        osz = int(ofs.sum())
        assert len(payload) <= 1.01 * osz + 16, (name, level, len(payload), osz)
        assert bytes(payload) == oenc[len(oenc) - osz:], (name, level)
        assert list(fs) == list(ofs)
        back = nat.host_decode(payload, x.shape[1], bps, 4096, 44100, x.shape[0])
        assert np.array_equal(back, x)


def _random_signal(rng, n, ch, bps):
    """A seeded signal with segments of different character (smooth, noisy, sparse, constant, full scale, wasted bits)."""
    lim = 32767 if bps == 16 else 8388607
    x = np.zeros((n, ch), dtype=np.int64)
    base = np.cumsum(rng.integers(-lim // 400 - 1, lim // 400 + 2, size=n))
    kinds = []
    for c in range(ch):
        kind = int(rng.integers(0, 6))
        kinds.append(kind)
        if kind == 0:
            v = base + rng.integers(-8, 9, size=n) + (c * 37)                          # correlated with the other channels
        elif kind == 1:
            v = rng.integers(-lim, lim + 1, size=n)                                     # white noise, full scale
        elif kind == 2:
            v = (lim * 0.6 * np.sin(np.arange(n) / rng.uniform(3, 90))).astype(np.int64) + rng.integers(-30, 31, size=n)
        elif kind == 3:
            v = np.where(rng.random(n) < 0.01, rng.integers(-lim, lim + 1, size=n), 0)  # sparse spikes (long unary runs / escapes)
        elif kind == 4:
            v = np.full(n, int(rng.integers(-lim, lim + 1)))                            # constant
        else:
            v = (base // 3) * (1 << int(rng.integers(1, 6)))                            # wasted bits
        x[:, c] = np.clip(v, -lim, lim)
    if n > 6000 and rng.random() < 0.5:
        a = int(rng.integers(0, n - 5000))
        x[a:a + 4500] = x[a, :]                                                         # a constant stretch: CONSTANT subframes
    return x.astype(np.int32), kinds


def test_random_streams_match_oracle_and_roundtrip(nat, oracle):
    """Seeded sweep over lengths (tail frames, sub-block streams), channel counts 1-8 (2 -> mid/side), both bit depths and
    all levels: GPU frames decode back exactly, are never more than 1 % larger than the oracle's, and are byte-identical to
    the oracle's libFLAC procedure -- except for one documented class: a nearly pure tone at 24-bit amplitude makes the
    autocorrelation matrix close to singular, and there the GPU's summation tree (per-thread partial sums + butterfly)
    and libFLAC's sample-order sum round differently in the last bits, which moves a quantised LPC coefficient by 1-2
    steps (DESIGN.md section 4, "Encoder exactness").  Those streams must differ in nothing but LPC subframes."""
    rng = np.random.default_rng(20261018)
    from flac_raster_b200 import flacfmt
    mismatched = 0
    for case in range(36):
        ch = int(rng.integers(1, 9)) if case % 3 else 2
        bps = 16 if rng.random() < 0.7 else 32
        n = int(rng.choice([17, 4095, 4096, 4097, 8192, 12289, 20000, 33000]))
        level = int(rng.integers(0, 9))
        x, kinds = _random_signal(rng, n, ch, bps)
        payload, fs = nat.host_encode(x, bps, 48000, level)
        oenc, ofs, od = oracle.encode(x, bps, 48000, level, mid_side=(bps == 16), want_descs=True)
        osz = int(ofs.sum())
        back = nat.host_decode(payload, ch, bps, 4096, 48000, n)
        assert np.array_equal(back, x), (case, n, ch, bps, level)
        assert len(payload) <= 1.01 * osz + 16, (case, len(payload), osz)
        if bytes(payload) == oenc[len(oenc) - osz:]:
            continue
        mismatched += 1
        assert bps == 32 and 2 in kinds and level >= 3, (case, n, ch, bps, level, kinds)
        si = flacfmt.StreamInfo(4096, 4096, 0, 0, 48000, ch, bps, n)
        dec, info, gd = oracle.decode(flacfmt.build_header(si) + bytes(payload), want_descs=True)
        assert np.array_equal(dec, x)
        for a, b in zip(gd, od):
            if any(a[k] != b[k] for k in ("type", "order", "coefs", "partition_order", "params", "shift", "precision")):
                assert a["type"] == 3 and b["type"] == 3 and kinds[a["channel"]] == 2, (case, a["frame"], a["channel"])
    assert mismatched <= 6


def test_encode_golden_rgb_is_byte_identical_to_libflac(nat, rgb_pcm):
    """Level 5 on normalize_to_audio(sample_rgb.tif): the GPU emits libFLAC 1.4.3's exact frame bytes."""
    golden = (GOLDEN / "sample_rgb.flac").read_bytes()
    payload, fs = nat.host_encode(rgb_pcm, 16, 44100, 5)
    assert len(payload) == 178857 <= 1.01 * 178857
    assert bytes(payload) == golden[86:]


def test_gpu_streams_accepted_by_ffmpeg(nat):
    """FFmpeg libavcodec accepts the GPU's level-8 streams: every stream is byte for byte one that FFmpeg decoded to the
    input samples (tests/golden/ffmpeg_decoded.json, made by make_ffmpeg_golden.py), and where the bundled FFmpeg
    libraries are installed they decode it again."""
    import hashlib
    from flac_raster_b200 import flacfmt
    from oracle import ffmpeg_flac as ff
    golden = json.loads((GOLDEN / "ffmpeg_decoded.json").read_text())["gpu_level8"]
    live = ff.available()
    cases = {k: v for k, v in signal_cases().items() if k != "tiny3"}        # FFmpeg refuses blocksize < 16
    assert set(golden) == set(cases)
    for name, (x, bps) in cases.items():
        payload, _ = nat.host_encode(x, bps, 48000, 8)
        si = flacfmt.StreamInfo(4096, 4096, 0, 0, 48000, x.shape[1], bps, x.shape[0])
        stream = flacfmt.build_header(si) + bytes(payload)
        assert hashlib.md5(stream).hexdigest() == golden[name]["stream_md5"], name
        assert hashlib.md5(np.ascontiguousarray(x, dtype="<i4").tobytes()).hexdigest() == golden[name]["decoded_md5"], name
        if live:
            assert np.array_equal(ff.decode_bytes(stream, x.shape[1]), x), name


def test_pyflac_shim_callback_contract(nat, oracle, tmp_path):
    """StreamEncoder/FileDecoder behave like pyflac's (header chunks with num_samples == 0 first, then
    one callback per frame with current_frame == index), and the written file decodes everywhere."""
    from flac_raster_b200 import codec
    x = signal_cases()["smooth16_8ch"][0].astype(np.int16)
    calls = []
    path = tmp_path / "shim.flac"
    fh = open(path, "wb")

    def cb(data, num_bytes, num_samples, current_frame):
        calls.append((num_bytes, num_samples, current_frame))
        fh.write(data[:num_bytes])

    enc = codec.StreamEncoder(write_callback=cb, sample_rate=48000, compression_level=5, blocksize=4096)
    enc._channels, enc._bits_per_sample = 8, 16
    enc.process(x)
    assert enc.finish() is True
    fh.close()
    hdr_calls = [c for c in calls if c[1] == 0]
    frame_calls = [c for c in calls if c[1] != 0]
    assert calls[:len(hdr_calls)] == hdr_calls and hdr_calls[0][0] == 4
    assert [c[2] for c in frame_calls] == list(range(len(frame_calls))) == list(range((len(x) + 4095) // 4096))
    assert frame_calls[-1][1] == len(x) - 4096 * (len(frame_calls) - 1)
    dec, info = oracle.decode(path.read_bytes())
    assert np.array_equal(dec, x.astype(np.int32)) and info.total_samples_streaminfo == 0
    audio, rate = codec.FileDecoder(str(path)).process()
    assert rate == 48000 and audio.dtype == np.int16 and np.array_equal(audio, x)
    f64, _ = codec.FileDecoder(str(path), compat_pyflac_float=True).process()
    assert f64.dtype == np.float64 and np.array_equal(f64, x / 32768.0)
    # reference-made file through the shim
    g, r = codec.FileDecoder(str(GOLDEN / "sample_rgb.flac")).process()
    assert r == 44100 and g.shape == (65536, 3)


# ------------------------------------------------------------------ public API (configs C1, C2)
def test_config1_dem_roundtrip(nat, oracle, tmp_path):
    """BASELINE config 1: sample_dem.tif -> FLAC -> TIFF, level 5, bit-exact; file is a valid tagged FLAC."""
    from flac_raster_b200 import RasterFLACConverter, flacfmt
    from flac_raster_b200.tiffio import read_geotiff
    from oracle import normalization_oracle as no
    conv = RasterFLACConverter()
    flac, tif = tmp_path / "dem.flac", tmp_path / "dem.tif"
    conv.tiff_to_flac(GOLDEN / "sample_dem.tif", flac, compression_level=5)
    conv.flac_to_tiff(flac, tif)
    a, b = read_geotiff(GOLDEN / "sample_dem.tif"), read_geotiff(tif)
    assert np.array_equal(a.data, b.data) and a.data.dtype == b.data.dtype
    assert a.transform == b.transform and a.crs == b.crs
    blob = flac.read_bytes()
    h = flacfmt.parse_header(blob)
    assert h.tags["GEOSPATIAL_WIDTH"] == ["512"] and h.tags["GEOSPATIAL_DTYPE"] == ["int16"]
    assert h.tags["GEOSPATIAL_DATA_MIN"] == ["577.0"] and h.tags["GEOSPATIAL_DATA_MAX"] == ["1492.0"]
    dec, info = oracle.decode(blob)                       # samples == reference normalisation of the raster
    want, _ = no.normalize_to_audio(a.data.reshape(-1, 1), 16)
    assert np.array_equal(dec, want.astype(np.int32)) and (info.sample_rate, info.bps) == (44100, 16)
    # byte-identical frames to the libFLAC-procedure oracle on the same samples
    oenc, ofs = oracle.encode(want, 16, 44100, 5)
    assert blob[h.first_frame_offset:] == oenc[len(oenc) - int(ofs.sum()):]
    with pytest.raises(ValueError, match="No metadata found"):
        bare = tmp_path / "bare.flac"
        bare.write_bytes(oenc)
        conv.flac_to_tiff(bare, tmp_path / "x.tif")


def test_config2_rgb_streaming_tile512(nat, oracle, tmp_path):
    """BASELINE config 2: sample_rgb.tif, streaming, tile_size 512, encode + get_tile_by_id."""
    from flac_raster_b200 import SpatialFLACEncoder, SpatialFLACStreamer
    from flac_raster_b200.tiffio import read_geotiff
    out = tmp_path / "rgb_stream.flac"
    SpatialFLACEncoder(tile_size=512).encode(GOLDEN / "sample_rgb.tif", out, streaming=True)
    blob = out.read_bytes()
    (n,) = struct.unpack(">I", blob[:4])
    index = json.loads(blob[4:4 + n])
    assert index["width"] == 256 and index["bands"] == 3 and index["dtype"] == "uint8" and index["tile_size"] == 512
    assert len(index["frames"]) == 1 and index["frames"][0]["byte_offset"] == 0
    f0 = index["frames"][0]
    tile_file = blob[4 + n: 4 + n + f0["byte_size"]]
    assert 4 + n + f0["byte_size"] == len(blob) and tile_file[:4] == b"fLaC"
    golden = (GOLDEN / "sample_rgb.flac").read_bytes()
    from flac_raster_b200 import flacfmt
    off = flacfmt.parse_header(tile_file).first_frame_offset
    assert tile_file[off:] == golden[86:]                 # same frames libFLAC produced for this raster
    tile, meta = SpatialFLACStreamer(out).get_tile_by_id(0)
    src = read_geotiff(GOLDEN / "sample_rgb.tif")
    assert np.array_equal(tile, src.data) and tile.dtype == np.uint8
    assert meta["width"] == 256 and meta["count"] == 3 and meta["frame_id"] == 0
    with pytest.raises(KeyError):
        SpatialFLACStreamer(out).get_tile_by_id(7)


def test_streaming_small_tiles_bbox_and_center(nat, oracle, tmp_path):
    """CI smoke of the reference (--streaming --tile-size 128 + extract) plus multi-tile bbox decode."""
    from flac_raster_b200 import SpatialFLACEncoder, SpatialFLACStreamer
    from flac_raster_b200.tiffio import read_geotiff
    from oracle import normalization_oracle as no
    src = read_geotiff(GOLDEN / "sample_dem.tif")
    out = tmp_path / "dem_stream.flac"
    idx = SpatialFLACEncoder(tile_size=200).encode(GOLDEN / "sample_dem.tif", out, streaming=True, compression_level=8)
    assert len(idx.frames) == 9                          # 3x3 grid with 112-wide edge tiles
    s = SpatialFLACStreamer(out)
    blob = out.read_bytes()
    total = 0
    for f in s.spatial_index.frames:
        w = f.window
        tile_file = blob[s.header_size + f.byte_offset: s.header_size + f.byte_offset + f.byte_size]
        dec, info = oracle.decode(tile_file)              # every tile is a standalone FLAC file
        win = src.data[:, w.row_off:w.row_off + w.height, w.col_off:w.col_off + w.width]
        want, _ = no.normalize_to_audio(win.transpose(1, 2, 0).reshape(-1, 1), 16)     # per-tile min/max (SURVEY Q5)
        assert np.array_equal(dec, want.astype(np.int32)) and info.sample_rate == 44100
        assert f.byte_offset == total
        total += f.byte_size
    assert s.header_size + total == len(blob)
    t = src.transform
    res = s.get_tiles_by_bbox(t[2] + 150 * t[0], t[5] + 450 * t[4], t[2] + 450 * t[0], t[5] + 150 * t[4])
    assert sorted(m["frame_id"] for _, m in res) == [0, 1, 2, 3, 4, 5, 6, 7, 8]
    for tile, m in res:
        w = m["window"]
        assert np.array_equal(tile, src.data[:, w["row_off"]:w["row_off"] + w["height"], w["col_off"]:w["col_off"] + w["width"]])
    res = s.get_tiles_by_bbox(t[2] + 10 * t[0], t[5] + 190 * t[4], t[2] + 190 * t[0], t[5] + 10 * t[4])
    assert [m["frame_id"] for _, m in res] == [0]
    assert s.get_tiles_by_bbox(1e6, 1e6, 2e6, 2e6) == []
    tile, m = s.get_center_tile()
    assert m["frame_id"] == 4
    # legacy --spatial layout: concatenated streams with a valid embedded index
    leg = tmp_path / "legacy.flac"
    SpatialFLACEncoder(tile_size=256).encode(GOLDEN / "sample_dem.tif", leg, streaming=False)
    ls = SpatialFLACStreamer(leg)
    lblob = leg.read_bytes()
    for f in ls.spatial_index.frames:
        assert lblob[f.byte_offset:f.byte_offset + 4] == b"fLaC"
    tile, m = ls.get_tile_by_id(3)
    assert np.array_equal(tile, src.data[:, 256:, 256:])


@pytest.mark.parametrize("dt", ["uint8", "int8", "uint16", "int16", "uint32", "int32", "float32", "float64"])
def test_all_dtypes_roundtrip_equals_reference_semantics(nat, tmp_path, dt):
    """Reconstruction equals denormalize(normalize(x)) of the reference for every dtype (SURVEY Q4)."""
    from flac_raster_b200 import RasterFLACConverter
    from oracle import normalization_oracle as no
    rng = np.random.default_rng(11)
    if dt.startswith("float"):
        x = (500 + 300 * np.sin(np.arange(3 * 130 * 170) / 50.0) + rng.standard_normal(3 * 130 * 170)).astype(dt)
    else:
        info = np.iinfo(dt)
        lo, hi = max(info.min, -8000), min(info.max, 8000)    # range < 32767: exact under truncation (SURVEY Q3)
        x = rng.integers(lo, hi, size=3 * 130 * 170, endpoint=True).astype(dt)
    x = x.reshape(3, 130, 170)
    conv = RasterFLACConverter()
    p = tmp_path / f"{dt}.flac"
    conv.array_to_flac(x, p, 5, transform=(1.0, 0.0, 0.0, 0.0, -1.0, 0.0), crs="EPSG:4326")
    back, md = conv.flac_to_array(p)
    bits = 16 if dt in ("uint8", "int8", "uint16", "int16") else 24
    a, prm = no.normalize_to_audio(x.transpose(1, 2, 0).reshape(-1, 3), bits)
    want = no.denormalize_from_audio(a, prm["data_min"], prm["data_max"], dt, prm["scale_factor"])
    want = want.reshape(130, 170, 3).transpose(2, 0, 1)
    assert back.dtype == x.dtype and np.array_equal(back, want)
    if bits == 16:
        assert np.array_equal(back, x)        # 8/16-bit rasters with range <= 32767 are lossless


# ------------------------------------------------------------------ full-size properties
def _roundtrip_on_device(torch, raster, tile_size, level):
    from flac_raster_b200.engine import default_engine, tile_grid
    eng = default_engine()
    bands, H, W = raster.shape
    tiles = tile_grid(H, W, tile_size)
    enc = eng.encode_tiles(raster, tiles, level)
    payload = torch.cat([enc.payload, torch.zeros(64, dtype=torch.uint8, device=raster.device)])
    audio, base, status = eng.decode_streams(payload, enc.offsets, enc.sizes, enc.n_samples, enc.sample_rates,
                                             bands, enc.bps, enc.blocksize)
    assert status[0] == 0 and status[1] == 0 and status[2] == 0, status
    assert status[3] == int(((enc.n_samples + 4095) // 4096).sum())
    out = torch.zeros_like(raster)
    scale = 32767.0 if enc.bits_per_sample == 16 else 8388607.0
    eng.denormalize_tiles(audio, base, tiles, enc.minmax, scale, out)
    # the fused decode + denormalise launch must write exactly the same raster
    fused = torch.zeros_like(raster)
    st2 = eng.decode_tiles(payload, enc.offsets, enc.sizes, tiles, enc.sample_rates, enc.minmax, scale, fused, enc.bps, enc.blocksize, fused=True)
    assert list(st2[:3]) == [0, 0, 0] and st2[3] == status[3] and st2[5] == 0, st2
    assert torch.equal(fused.reshape(-1).view(torch.uint8), out.reshape(-1).view(torch.uint8))
    return enc, out


def test_fullsize_c5_tiles_int16_roundtrip(nat, torch_cuda):
    """Config 5 corpus (4096 tiles of 512x512 int16, or FRB_TEST_TILES): encode -> decode -> raster identical."""
    torch = torch_cuda
    from flac_raster_b200.synth import dem_int16_tiles
    n = int(os.environ.get("FRB_TEST_TILES", "4096"))
    raster = dem_int16_tiles(n, 512)
    enc, out = _roundtrip_on_device(torch, raster, 512, 5)
    assert torch.equal(out, raster)
    assert len(enc.sizes) == n and int(enc.sizes.sum()) < raster.numel() * 2 * 0.8


def test_fullsize_c3_sentinel_like_roundtrip(nat, torch_cuda):
    """Config 3 (10980^2 x 8 uint16, tile 1024 -> 121 tiles incl. 740-wide edges): lossless on device."""
    torch = torch_cuda
    from flac_raster_b200.synth import sentinel2_like
    side = int(os.environ.get("FRB_TEST_C3_SIDE", "10980"))
    raster = sentinel2_like(side, side, 8)
    enc, out = _roundtrip_on_device(torch, raster, 1024, 5)
    assert torch.equal(out.view(torch.int16), raster.view(torch.int16))
    if side == 10980:
        assert len(enc.sizes) == 121 and set(enc.sample_rates.tolist()) == {44100, 48000}


def test_fullsize_c4_float32_level8_roundtrip(nat, torch_cuda):
    """Config 4 at its BASELINE size (float32 DEM 32768^2, level 8, one 32-bps stream of 2^30 samples; FRB_TEST_C4_SIDE
    shrinks it for debugging): decode(encode(x)) == normalise(x) sample-for-sample, and the reconstruction equals the
    reference's 24-bit quantisation (normalize_to_audio -> denormalize_from_audio in numpy) on sampled rows."""
    torch = torch_cuda
    from flac_raster_b200.engine import default_engine, tile_grid
    from flac_raster_b200.synth import dem_float32
    from oracle import normalization_oracle as no
    side = int(os.environ.get("FRB_TEST_C4_SIDE", "32768"))
    raster = dem_float32(side, side)
    eng = default_engine()
    tiles = tile_grid(side, side, side)
    enc = eng.encode_tiles(raster, tiles, 8)
    assert enc.bps == 32 and enc.sample_rates[0] == (96000 if side * side < 100_000_000 else 192000)
    audio_ref, base_ref, npx, d_mm, bits = eng.normalize_tiles(raster, tiles)
    ref = audio_ref[:side * side * 4].view(torch.int32).clone()
    payload = torch.cat([enc.payload, torch.zeros(64, dtype=torch.uint8, device=raster.device)])
    audio, base, status = eng.decode_streams(payload, enc.offsets, enc.sizes, enc.n_samples, enc.sample_rates, 1, 32, 4096)
    assert list(status[:3]) == [0, 0, 0]
    assert status[3] == (side * side + 4095) // 4096
    assert torch.equal(audio[:side * side * 4].view(torch.int32), ref)
    assert int(enc.sizes.sum()) < side * side * 4 * 0.75
    # reconstruction: the GPU denormalise of the decoded samples against the reference formula on a few row bands
    out = torch.zeros_like(raster)
    eng.denormalize_tiles(audio, base, tiles, enc.minmax, 8388607.0, out)
    dmin, dmax = float(enc.minmax[0, 0]), float(enc.minmax[0, 1])
    for r0 in (0, side // 2 - 3, side - 8):
        rows = raster[0, r0:r0 + 8].cpu().numpy()
        a, prm = no.normalize_to_audio(rows.reshape(-1, 1), 24, dmin, dmax)
        back = no.denormalize_from_audio(a, dmin, dmax, "float32", 8388607)
        assert np.array_equal(out[0, r0:r0 + 8].cpu().numpy().reshape(-1, 1), back)
        assert np.abs(back.reshape(rows.shape).astype(np.float64) - rows).max() <= (dmax - dmin) / 8388607.0


def test_two_band_raster_mid_side_tiles(nat, oracle, torch_cuda):
    """A 2-band raster through the tile engine: frames equal the oracle's libFLAC procedure WITH its stereo decorrelation
    (correlated bands make left/side or mid/side win), and the mid/side frames decode back to the raster."""
    torch = torch_cuda
    from flac_raster_b200 import flacfmt
    from flac_raster_b200.engine import default_engine, tile_grid
    from oracle import normalization_oracle as no
    rng = np.random.default_rng(21)
    H, W = 300, 420
    yy, xx = np.mgrid[0:H, 0:W]
    b0 = (3000 + 1500 * np.sin(xx / 31.0) * np.cos(yy / 19.0) + rng.integers(-20, 20, size=(H, W))).astype(np.uint16)
    b1 = (b0.astype(np.int32) + 40 + rng.integers(-5, 5, size=(H, W))).astype(np.uint16)
    x = np.stack([b0, b1])
    raster = torch.from_numpy(x.view(np.int16)).cuda().view(torch.uint16)
    eng = default_engine()
    tiles = tile_grid(H, W, 160)
    enc = eng.encode_tiles(raster, tiles, 5)
    payload = enc.payload.cpu().numpy()
    assigns = set()
    for i, t in enumerate(tiles):
        r, c, h, w = (int(t[k]) for k in ("row_off", "col_off", "h", "w"))
        want, prm = no.normalize_to_audio(x[:, r:r + h, c:c + w].transpose(1, 2, 0).reshape(-1, 2), 16)
        oenc, ofs, descs = oracle.encode(want, 16, int(enc.sample_rates[i]), 5, want_descs=True)
        assigns.update(d["ch_assign"] for d in descs)
        frames = payload[enc.offsets[i]:enc.offsets[i] + enc.sizes[i]].tobytes()
        assert frames == oenc[len(oenc) - int(ofs.sum()):], i
    assert assigns & {8, 9, 10}, assigns                      # the decorrelated forms were actually chosen
    dev_payload = torch.cat([enc.payload, torch.zeros(64, dtype=torch.uint8, device=raster.device)])
    out = torch.zeros_like(raster)
    st = eng.decode_tiles(dev_payload, enc.offsets, enc.sizes, tiles, enc.sample_rates, enc.minmax, 32767.0, out, 16, 4096)
    assert list(st[:3]) == [0, 0, 0], st
    assert torch.equal(out.view(torch.int16), raster.view(torch.int16))


@pytest.mark.parametrize("dt", ["float32", "int32"])
def test_two_band_32bit_raster_mid_side_with_33bit_side(nat, oracle, torch_cuda, dt):
    """A 2-band float32 / int32 raster: the reference hands libFLAC a two-channel 32-bps stream, and libFLAC's presets run the
    mid/side search there too, with a 33-bit side subframe (docs/sonos-pyflac.txt:6926-6934).  The tile path's audio is 24-bit
    (scale 8388607), so L - R fits the int32 planar audio and the GPU encoder runs the same search (FRB_ENC_RANGE_30): frames
    equal the oracle's at levels 0-8 (tail frames through the one-kernel encoder included), the decorrelated forms are
    actually chosen, the frames are smaller than independent coding and decode back on the GPU (33-bit warm-up samples,
    side reconstruction)."""
    torch = torch_cuda
    from flac_raster_b200 import flacfmt
    from flac_raster_b200.engine import Engine, tile_grid
    from oracle import normalization_oracle as no
    rng = np.random.default_rng(31)
    H, W = 200, 330
    yy, xx = np.mgrid[0:H, 0:W]
    base = 1200.0 + 700.0 * np.sin(xx / 37.0) * np.cos(yy / 23.0) + rng.normal(0, 0.4, size=(H, W))
    other = base * 0.98 + 11.0 + rng.normal(0, 0.05, size=(H, W))
    x = np.stack([base, other])
    x = x.astype(np.float32) if dt == "float32" else np.round(x * 1000).astype(np.int32)
    raster = torch.from_numpy(x).cuda()
    eng = Engine()
    tiles = tile_grid(H, W, 128)
    for level in (0, 1, 5, 8):
        enc = eng.encode_tiles(raster, tiles, level)
        assert enc.bps == 32 and enc.bits_per_sample == 24
        payload = enc.payload.cpu().numpy()
        assigns, indep = set(), 0
        for i, t in enumerate(tiles):
            r, c, h, w = (int(t[k]) for k in ("row_off", "col_off", "h", "w"))
            want, prm = no.normalize_to_audio(x[:, r:r + h, c:c + w].transpose(1, 2, 0).reshape(-1, 2), 24)
            oenc, ofs, descs = oracle.encode(want.astype(np.int32), 32, int(enc.sample_rates[i]), level, want_descs=True)
            assigns.update(d["ch_assign"] for d in descs)
            frames = payload[enc.offsets[i]:enc.offsets[i] + enc.sizes[i]].tobytes()
            assert frames == oenc[len(oenc) - int(ofs.sum()):], (level, i)
            plain, pfs = oracle.encode(want.astype(np.int32), 32, int(enc.sample_rates[i]), level, mid_side=False)
            indep += int(pfs.sum())
        if level:                                              # level 0 has no stereo search
            assert assigns & {8, 9, 10}, (level, assigns)
            assert int(enc.sizes.sum()) < 0.97 * indep, (level, int(enc.sizes.sum()), indep)
        dev_payload = torch.cat([enc.payload, torch.zeros(64, dtype=torch.uint8, device=raster.device)])
        audio, abase, st = eng.decode_streams(dev_payload, enc.offsets, enc.sizes, enc.n_samples, enc.sample_rates, 2, 32, 4096)
        assert list(st[:3]) == [0, 0, 0], st
        out = torch.zeros_like(raster)
        eng.denormalize_tiles(audio, abase, tiles, enc.minmax, 8388607.0, out)
        want_px = np.zeros_like(x)
        for i, t in enumerate(tiles):
            r, c, h, w = (int(t[k]) for k in ("row_off", "col_off", "h", "w"))
            a, prm = no.normalize_to_audio(x[:, r:r + h, c:c + w].transpose(1, 2, 0).reshape(-1, 2), 24)
            back = no.denormalize_from_audio(a, prm["data_min"], prm["data_max"], dt, prm["scale_factor"])
            want_px[:, r:r + h, c:c + w] = back.T.reshape(2, h, w)
        assert np.array_equal(out.cpu().numpy(), want_px), level
    # the other direction: a foreign two-channel 32-bps stream whose side channel really needs 33 bits (full-range audio, never
    # made by the reference) cannot be held by the int32 sample path: the decoder must say so, not hand out wrapped samples
    t = np.arange(12000)
    wob = (900 * np.sin(t / 50.0)).astype(np.int64) + rng.integers(-40, 40, size=t.size)
    wide = np.stack([(1 << 30) + 1000 + wob, -(1 << 30) - 1000 + wob], axis=1).astype(np.int32)
    oenc, ofs, descs = oracle.encode(wide, 32, 44100, 5, want_descs=True)
    assert {d["ch_assign"] for d in descs} & {8, 9, 10}
    ref, _ = oracle.decode(oenc)
    assert np.array_equal(ref, wide)
    with pytest.raises(nat.NativeError) as ei:
        nat.host_decode(oenc[len(oenc) - int(ofs.sum()):], 2, 32, 4096, 44100, wide.shape[0])
    assert ei.value.status == nat.ERR_BAD_STREAM
    # a stream that breaks the range promise is refused, not mis-coded
    big = torch.tensor([[2 ** 30 + 5] * 5000, [-(2 ** 30) - 9] * 5000], dtype=torch.int32).cuda().reshape(-1)
    n = np.array([5000], dtype=np.int64)
    with pytest.raises(nat.NativeError) as ei:
        eng.encode_audio(big, n, np.array([0], dtype=np.int64), np.array([44100], dtype=np.uint32), 2, 32, 5, 4096, range30=True)
    assert ei.value.status == nat.ERR_INVALID_ARG
    eng.encode_audio(big, n, np.array([0], dtype=np.int64), np.array([44100], dtype=np.uint32), 2, 32, 5, 4096)    # independent: fine


def test_host_pipeline_equals_device_path(nat, torch_cuda):
    """encode_tiles_host (tile rows pipelined over copy/compute/copy streams, host buffers) produces exactly the
    bytes, offsets and min/max of the one-shot device path, including ragged edge tiles."""
    torch = torch_cuda
    from flac_raster_b200.engine import default_engine, tile_grid
    from flac_raster_b200.synth import sentinel2_like
    raster = sentinel2_like(1500, 1300, 3)
    eng = default_engine()
    tiles = tile_grid(1500, 1300, 512)              # 3 x 3 tiles, last row/col ragged (476 / 276)
    ref = eng.encode_tiles(raster, tiles, 5)
    ref_bytes = ref.payload.cpu().numpy().copy()
    host = raster.cpu().pin_memory()
    for gb in (0, 0, None):                          # 0: one stage per tile row (second pass reuses slabs/payload buffers)
        got = eng.encode_tiles_host(host, tiles, 5, group_bytes=gb)
        assert not got.payload.is_cuda
        assert np.array_equal(got.sizes, ref.sizes) and np.array_equal(got.offsets, ref.offsets)
        assert np.array_equal(got.minmax, ref.minmax)
        assert np.array_equal(got.payload.numpy(), ref_bytes)


def test_host_decode_pipeline_equals_raster(nat, torch_cuda):
    """decode_tiles_host (frames of tile rows pipelined over copy/decode/copy streams, host buffers) reproduces the raster,
    ragged edge tiles included, whatever the stage size."""
    torch = torch_cuda
    from flac_raster_b200.engine import default_engine, tile_grid
    from flac_raster_b200.synth import sentinel2_like
    raster = sentinel2_like(1500, 1300, 3)
    eng = default_engine()
    tiles = tile_grid(1500, 1300, 512)
    enc = eng.encode_tiles(raster, tiles, 5)
    host_payload = enc.payload.cpu().pin_memory()
    want = raster.cpu()
    for gb in (0, 0, None):
        out = torch.zeros(raster.shape, dtype=raster.dtype).pin_memory()
        st = eng.decode_tiles_host(host_payload, enc.offsets, enc.sizes, tiles, enc.sample_rates, enc.minmax, 32767.0, out, enc.bps,
                                   group_bytes=gb)
        assert list(st[:3]) == [0, 0, 0] and st[3] == int(((enc.n_samples + 4095) // 4096).sum()), st
        assert torch.equal(out.view(torch.int16), want.view(torch.int16))


@pytest.mark.parametrize("dt", ["uint8", "int8", "uint16", "int16"])
def test_int16_audio_equals_int32_audio(nat, oracle, torch_cuda, dt):
    """The tile path keeps 16-bit audio as int16 between the mapping kernel and the analysis kernels
    (frb_normalize_tiles_i16 + FRB_ENC_AUDIO_I16): same samples as the int32 buffer on aligned and ragged windows, and
    the frames coded from either buffer are the same bytes (fast kernels on aligned full blocks, the one-kernel
    encoder on unaligned channels and tail frames)."""
    torch = torch_cuda
    from flac_raster_b200.engine import Engine
    from flac_raster_b200 import _native as natmod
    from flac_raster_b200.normalization import sample_rates_for_pixel_counts
    rng = np.random.default_rng(11)
    bands, H, W = 3, 300, 523
    info = np.iinfo(dt)
    yy, xx = np.mgrid[0:H, 0:W]
    x = np.stack([np.clip(info.min // 2 + (info.max - info.min) // 3 * (1 + np.sin(xx / 19.0 + b) * np.cos(yy / 13.0)) / 2
                          + rng.integers(-3, 4, xx.shape), info.min, info.max).astype(dt) for b in range(bands)])
    tiles = np.zeros(7, dtype=natmod.TILE_DTYPE)
    tiles[0] = (0, 0, 128, 128); tiles[1] = (1, 3, 67, 211); tiles[2] = (7, 13, 33, 37); tiles[3] = (44, 1, 256, 512); tiles[4] = (2, 5, 5, 1)
    # 250 x 250 = 4 mod 8 pixels: every other band starts 8-byte (not 16-byte) aligned in the int16 audio -- still the fast kernels;
    # twice, so that the second one starts at a different alignment of the running base
    tiles[5] = (10, 10, 250, 250); tiles[6] = (30, 200, 250, 250)
    eng = Engine()
    dev = torch.from_numpy(x.view(np.uint8).reshape(-1)).cuda().view(getattr(torch, dt)).reshape(bands, H, W)
    a32, base, npx, d_mm, bits = eng.normalize_tiles(dev, tiles)
    total = int((npx * bands).sum())
    a32 = a32[: total * 4].view(torch.int32).clone()
    a16, base16, _, _, _ = eng.normalize_tiles(dev, tiles, audio_i16=True)
    assert a16.dtype == torch.int16 and a16.numel() == total and np.array_equal(base, base16)
    assert torch.equal(a16.to(torch.int32), a32)
    rates = sample_rates_for_pixel_counts(npx)
    for level in (0, 5, 8):
        p16, o16, s16, fb16, sb16 = eng.encode_audio(a16, npx, base, rates, bands, 16, level, 4096, payload_name="p16")
        p32, o32, s32, fb32, sb32 = eng.encode_audio(a32, npx, base, rates, bands, 16, level, 4096, payload_name="p32")
        assert np.array_equal(s16, s32) and torch.equal(p16, p32) and torch.equal(fb16, fb32) and torch.equal(sb16, sb32), level
    with pytest.raises(ValueError):
        eng.encode_audio(a16, npx, base, rates, bands, 32, 5, 4096)


@pytest.mark.parametrize("dt", ["uint8", "int16", "uint16", "float32", "float64", "int32"])
def test_tile_mapping_odd_alignment_vs_oracle(nat, torch_cuda, dt):
    """Per-tile min/max, normalise and denormalise on windows whose rows start at odd element offsets and
    have widths that are not multiples of the 16-byte vector (head/tail lanes, scalar audio accesses)."""
    torch = torch_cuda
    from flac_raster_b200.engine import default_engine
    from flac_raster_b200 import _native as natmod
    from oracle import normalization_oracle as no
    rng = np.random.default_rng(5)
    bands, H, W = 2, 67, 211
    if dt.startswith("float"):
        x = (rng.standard_normal((bands, H, W)) * 1000).astype(dt)
        x[0, 3, 5] = np.nan
    else:
        info = np.iinfo(dt)
        x = rng.integers(max(info.min, -30000), min(info.max, 30000), size=(bands, H, W), endpoint=True).astype(dt)
    tiles = np.zeros(4, dtype=natmod.TILE_DTYPE)
    tiles[0] = (0, 0, 67, 211); tiles[1] = (1, 3, 5, 1); tiles[2] = (7, 13, 33, 37); tiles[3] = (2, 1, 60, 209)
    eng = default_engine()
    dev = torch.from_numpy(x.view(np.uint8).reshape(-1)).cuda().view(getattr(torch, dt)).reshape(bands, H, W)
    audio, base, npx, d_mm, bits = eng.normalize_tiles(dev, tiles)
    mm = d_mm.cpu().numpy().reshape(-1, 2)
    a = audio[: int((npx * bands).sum()) * 4].view(torch.int32).cpu().numpy()
    out = torch.zeros_like(dev)
    scale = 32767.0 if bits == 16 else 8388607.0
    for i, t in enumerate(tiles):
        r, c, h, w = (int(t[k]) for k in ("row_off", "col_off", "h", "w"))
        win = x[:, r:r + h, c:c + w]
        assert mm[i, 0] == np.nanmin(win) and mm[i, 1] == np.nanmax(win)
        want, prm = no.normalize_to_audio(win.reshape(bands, -1).T, bits)
        got = a[base[i]: base[i] + bands * h * w].reshape(bands, h * w).T
        assert np.array_equal(got, want.astype(np.int32)), (dt, i)
    # denormalise tile by tile (tiles overlap) and compare with the reference semantics
    for i, t in enumerate(tiles):
        r, c, h, w = (int(t[k]) for k in ("row_off", "col_off", "h", "w"))
        out.zero_()
        eng.denormalize_tiles(audio, base[i:i + 1], tiles[i:i + 1], mm[i:i + 1], scale, out)
        win = x[:, r:r + h, c:c + w]
        an, prm = no.normalize_to_audio(win.reshape(bands, -1).T, bits)
        want = no.denormalize_from_audio(an, prm["data_min"], prm["data_max"], dt, prm["scale_factor"]).T.reshape(bands, h, w)
        got = out.cpu().numpy()[:, r:r + h, c:c + w]
        assert np.array_equal(got, want, equal_nan=True), (dt, i)


@pytest.mark.parametrize("dt", ["uint8", "int8", "uint16", "int16", "uint32", "int32", "float32", "float64"])
@pytest.mark.parametrize("bands", [1, 3])
def test_fused_decode_to_raster_equals_two_step_path(nat, torch_cuda, dt, bands):
    """frb_decode_tiles (decode threads write denormalised pixels straight into the tile windows) against
    frb_decode_batch + frb_denormalize_tiles on ragged tiles: odd widths (batches straddle rows), a raster width that
    leaves rows at every store alignment, tail frames, constant and wasted-bits bands."""
    torch = torch_cuda
    from flac_raster_b200.engine import default_engine, tile_grid
    rng = np.random.default_rng(11)
    H, W = 301, 1037
    yy, xx = np.mgrid[0:H, 0:W]
    planes = []
    for b in range(bands):
        base_sig = 900 * np.sin(xx / (13.0 + b)) * np.cos(yy / 17.0) + rng.integers(-40, 40, size=(H, W))
        if dt.startswith("float"):
            planes.append((base_sig * 1.37 + 0.25).astype(dt))
        elif dt in ("uint8", "int8"):
            info = np.iinfo(dt)
            planes.append(np.clip(base_sig / 9 + (info.max + info.min) // 2, info.min, info.max).astype(dt))
        else:
            info = np.iinfo(dt)
            planes.append(np.clip(base_sig * 8 + 20000, max(info.min, -32000), min(info.max, 32000)).astype(dt))
    x = np.stack(planes)
    if bands == 3:
        x[2, :, :] = x[2, 0, 0]                              # a constant band: CONSTANT subframes
    raster = torch.from_numpy(x.view(np.uint8).reshape(-1)).cuda().view(getattr(torch, dt)).reshape(bands, H, W)
    eng = default_engine()
    for tile in (128, 97):
        tiles = tile_grid(H, W, tile)
        enc = eng.encode_tiles(raster, tiles, 5)
        payload = torch.cat([enc.payload, torch.zeros(64, dtype=torch.uint8, device=raster.device)])
        scale = 32767.0 if enc.bits_per_sample == 16 else 8388607.0
        audio, base, status = eng.decode_streams(payload, enc.offsets, enc.sizes, enc.n_samples, enc.sample_rates, bands, enc.bps, 4096)
        assert list(status[:3]) == [0, 0, 0]
        two = torch.zeros_like(raster)
        eng.denormalize_tiles(audio, base, tiles, enc.minmax, scale, two)
        one = torch.zeros_like(raster)
        st = eng.decode_tiles(payload, enc.offsets, enc.sizes, tiles, enc.sample_rates, enc.minmax, scale, one, enc.bps, 4096, fused=True)
        assert list(st[:3]) == [0, 0, 0] and st[5] == 0, st
        assert torch.equal(one.reshape(-1).view(torch.uint8), two.reshape(-1).view(torch.uint8)), (dt, bands, tile)
        if enc.bits_per_sample == 16:
            assert torch.equal(one.reshape(-1).view(torch.uint8), raster.reshape(-1).view(torch.uint8))


@pytest.mark.parametrize("dt", ["uint16", "int16", "uint8", "int8"])
def test_fused_integer_denormalise_is_exact_for_every_audio_value(nat, torch_cuda, dt):
    """The fused kernel maps 16-bit audio to integer pixels with exact integer arithmetic and only evaluates the fp64
    formula on exact ties.  Every audio value -32768..32767 (a foreign stream may hold any) under min/max pairs chosen to
    produce ties, zero range, full range and negative minima must equal the reference's fp64 formula + np.round."""
    torch = torch_cuda
    from flac_raster_b200.engine import default_engine
    from flac_raster_b200 import _native as natmod
    from oracle import normalization_oracle as no
    rng = np.random.default_rng(3)
    a = rng.permutation(np.arange(-32768, 32768, dtype=np.int32)).reshape(-1, 1)
    payload, _ = nat.host_encode(a, 16, 44100, 5)
    eng = default_engine()
    data = torch.cat([torch.from_numpy(np.frombuffer(bytes(payload), dtype=np.uint8).copy()), torch.zeros(64, dtype=torch.uint8)]).cuda()
    tiles = np.zeros(1, dtype=natmod.TILE_DTYPE)
    tiles[0] = (0, 0, 256, 256)
    info = np.iinfo(dt)
    pairs = [(info.min, info.max), (info.min, info.min + 1), (info.min + 3, info.min + 6), (info.max - 2, info.max),
             (info.min + 5, info.min + 5), (info.min, info.min + min(info.max - info.min, 32767)), (info.min + 1, info.max - 1),
             (info.min, info.min + 2), (info.min + 10, info.min + 10 + min(info.max - info.min - 10, 65533))]
    prng = np.random.default_rng(17)
    span = int(info.max) - int(info.min)
    for _ in range(24):                                   # seeded random windows, odd ranges (exact ties) over-represented
        r = int(prng.integers(0, min(span, 65535) + 1))
        if prng.random() < 0.5:
            r |= 1
        r = min(r, span)
        lo = int(prng.integers(int(info.min), int(info.max) - r + 1))
        pairs.append((lo, lo + r))
    for mn, mx in pairs:
        out = torch.zeros(1, 256, 256, dtype=getattr(torch, dt), device="cuda")
        st = eng.decode_tiles(data, np.array([0]), np.array([len(payload)]), tiles, np.array([44100], dtype=np.uint32),
                              np.array([[mn, mx]], dtype=np.float64), 32767.0, out, 16, 4096)
        assert list(st[:3]) == [0, 0, 0], st
        want = no.denormalize_from_audio(a.astype(np.int16), float(mn), float(mx), dt, 32767.0).reshape(256, 256)
        got = out.cpu().numpy()[0]
        assert np.array_equal(got, want), (dt, mn, mx, int((got != want).sum()))


def test_constant_division_is_exact(nat, torch_cuda):
    """The denormalise kernel divides by the constant scale with a reciprocal + one FMA correction; it must give the
    correctly rounded IEEE quotient for EVERY integer of the audio range (exhaustive, incl. all 2^32 int32 values)."""
    import ctypes as C
    L = nat.lib()
    for scale, lo, hi in ((32767.0, -32768, 32767), (8388607.0, -8388608, 8388607), (2147483647.0, -2147483648, 2147483647)):
        bad = C.c_uint64(123)
        nat.check(L.frb_selftest_division(scale, lo, hi, C.byref(bad), None), "frb_selftest_division")
        assert bad.value == 0, (scale, bad.value)


# ------------------------------------------------------------------ round 2: legacy reader, aliasing, big batches, C5 via the public API
def test_legacy_spatial_reader_on_reference_golden(nat, oracle):
    """SURVEY 8(f)4: the reference's own legacy --spatial file (gzip+base64 index without a marker tag, STALE byte offsets
    because mutagen grew stream 0 afterwards, SURVEY Q6) opens, and every tile equals oracle decode + reference denormalise
    with the file's global min/max (all the information a legacy file keeps)."""
    from flac_raster_b200 import SpatialFLACStreamer, flacfmt
    from oracle import normalization_oracle as no
    path = GOLDEN / "sample_dem.flac"
    blob = path.read_bytes()
    s = SpatialFLACStreamer(path)
    assert [(f.byte_offset, f.byte_size) for f in s.spatial_index.frames] == [(0, 10426), (10426, 8454), (18880, 8454), (27334, 8454)]
    for i, f in enumerate(s.spatial_index.frames):
        tile, meta = s.get_tile_by_id(i)
        pcm, info = oracle.decode(blob[f.byte_offset:f.byte_offset + f.byte_size])
        want = no.denormalize_from_audio(pcm.reshape(1, 256, 256), 577.0, 1493.0, "int16", 8388607)
        assert tile.dtype == np.int16 and tile.shape == (1, 256, 256) and np.array_equal(tile, want)
        assert meta["frame_id"] == i and meta["width"] == 256 and meta["data_min"] == 577.0
    allt = s.get_tiles_by_bbox(-200.0, -90.0, 200.0, 90.0)
    assert [m["frame_id"] for _, m in allt] == [0, 1, 2, 3]


def test_decoded_tiles_do_not_alias_the_staging_buffer(nat, tmp_path):
    """ADVICE r1 (high): arrays handed to the caller must survive the next decode call."""
    from flac_raster_b200 import SpatialFLACEncoder, SpatialFLACStreamer
    from flac_raster_b200.tiffio import read_geotiff
    src = read_geotiff(GOLDEN / "sample_dem.tif").data
    out = tmp_path / "s.flac"
    SpatialFLACEncoder(tile_size=256).encode(GOLDEN / "sample_dem.tif", out, streaming=True)
    s = SpatialFLACStreamer(out)
    a, _ = s.get_tile_by_id(1)
    a_copy = a.copy()
    b, _ = s.get_tile_by_id(2)
    assert not np.shares_memory(a, b)
    assert np.array_equal(a, a_copy) and np.array_equal(a, src[:, :256, 256:]) and np.array_equal(b, src[:, 256:, :256])
    res = s.get_tiles_by_bbox(-1e9, -1e9, 1e9, 1e9)
    keep = [t.copy() for t, _ in res]
    s.get_tile_by_id(3)
    assert all(np.array_equal(t, k) for (t, _), k in zip(res, keep))


def test_more_than_65535_tiles_in_one_batch(nat, torch_cuda):
    """ADVICE r1 (medium): the tile / stream index must not live in gridDim.y.  70 000 tiles of 16x16 in one batched call."""
    torch = torch_cuda
    from flac_raster_b200.engine import default_engine, tile_grid
    eng = default_engine()
    H, W = 16 * 280, 16 * 250
    g = torch.Generator(device="cuda").manual_seed(5)
    raster = (torch.randint(0, 4000, (1, H, W), generator=g, device="cuda", dtype=torch.int32)
              + (torch.arange(W, device="cuda", dtype=torch.int32) // 7)[None, None, :]).to(torch.int16)
    tiles = tile_grid(H, W, 16)
    assert len(tiles) == 70000
    enc = eng.encode_tiles(raster, tiles, 5)
    payload = torch.cat([enc.payload, torch.zeros(64, dtype=torch.uint8, device="cuda")])
    out = torch.zeros_like(raster)
    st = eng.decode_tiles(payload, enc.offsets, enc.sizes, tiles, enc.sample_rates, enc.minmax, 32767.0, out, 16, 4096)
    assert list(st[:3]) == [0, 0, 0] and st[3] == 70000
    assert torch.equal(out, raster)


def test_config5_bbox_over_4096_tiles_through_the_public_api(nat, torch_cuda, tmp_path):
    """BASELINE.json configs[4] through the product path: a 4096-tile container of 512x512 int16 written by the sharded
    writer, SpatialFLACStreamer.get_tiles_by_bbox over all of it (FRB_TEST_TILES shrinks it), every tile compared with the
    source, and the rank-split form (shard=(r, 4)) returning disjoint contiguous shares."""
    torch = torch_cuda
    import shutil
    import tempfile
    from flac_raster_b200 import SpatialFLACStreamer
    from flac_raster_b200.distributed import encode_streaming_sharded
    from flac_raster_b200.engine import default_engine
    from flac_raster_b200.synth import dem_int16_tiles
    n = int(os.environ.get("FRB_TEST_TILES", "4096"))
    T = 512
    raster = dem_int16_tiles(n, T)
    d = tempfile.mkdtemp(prefix="frb_c5_", dir="/dev/shm" if os.path.isdir("/dev/shm") else str(tmp_path))
    try:
        path = os.path.join(d, "c5.flac")
        H = n * T
        index, enc, _ = encode_streaming_sharded(raster, 0, (1, H, T), (1.0, 0.0, 0.0, 0.0, -1.0, float(H)), "EPSG:32633", None, "int16",
                                                 T, 5, path, 0, 1, engine=default_engine())
        s = SpatialFLACStreamer(path)
        res = s.get_tiles_by_bbox(-1.0, -1.0, T + 1.0, H + 1.0)
        assert [m["frame_id"] for _, m in res] == list(range(n))
        host = raster.cpu().numpy()
        for k, (tile, m) in enumerate(res):
            assert tile.shape == (1, T, T) and np.array_equal(tile, host[:, k * T:(k + 1) * T])
        del res
        shares = [s.get_tiles_by_bbox(-1.0, -1.0, T + 1.0, H + 1.0, shard=(r, 4)) for r in range(4)]
        ids = [m["frame_id"] for sh in shares for _, m in sh]
        assert ids == list(range(n)) and max(len(sh) for sh in shares) - min(len(sh) for sh in shares) <= 1
        # a bbox over part of the column: tiles 10..19 (strict intersection, cli.py:273-278)
        part = s.get_tiles_by_bbox(0.0, H - 20 * T + 0.5, T, H - 10 * T - 0.5)
        assert [m["frame_id"] for _, m in part] == list(range(10, 20))
    finally:
        shutil.rmtree(d, ignore_errors=True)


def test_seek_index_decode_equals_scan_path_and_bad_index_falls_back(nat, torch_cuda, tmp_path):
    """The encoder's seek index (frb_encode_index: frame sizes + subframe bit offsets) lets the decoder skip the sync scan and
    the subframe walk; results must be identical to the scanning path, an index that does not fit the bytes must be noticed and
    replaced by the scan, and containers must carry it in an APPLICATION block other decoders ignore."""
    torch = torch_cuda
    from flac_raster_b200 import SpatialFLACEncoder, SpatialFLACStreamer, flacfmt
    from flac_raster_b200.engine import default_engine, tile_grid
    from flac_raster_b200.synth import sentinel2_like
    eng = default_engine()
    for bands, side, ts in ((8, 1500, 512), (1, 1300, 512), (2, 700, 256)):
        raster = sentinel2_like(side, side, bands)
        tiles = tile_grid(side, side, ts)
        enc = eng.encode_tiles(raster, tiles, 5)
        assert enc.frame_bytes is not None and int(enc.frame_bytes.sum()) == int(enc.sizes.sum())
        fpt = enc.frames_per_tile()
        assert enc.frame_bytes.numel() == int(fpt.sum()) and enc.sub_bitoff.numel() == int(fpt.sum()) * bands
        payload = torch.cat([enc.payload, torch.zeros(64, dtype=torch.uint8, device="cuda")])
        outs = []
        for index in (None, enc.index(), (enc.frame_bytes.cpu().numpy().view(np.uint32), enc.sub_bitoff.cpu().numpy().view(np.uint32))):
            out = torch.zeros_like(raster)
            st = eng.decode_tiles(payload, enc.offsets, enc.sizes, tiles, enc.sample_rates, enc.minmax, 32767.0, out, 16, 4096, index=index)
            assert list(st[:3]) == [0, 0, 0] and st[3] == int(fpt.sum()), st
            outs.append(out)
        assert torch.equal(outs[0].view(torch.int16), raster.view(torch.int16))
        assert torch.equal(outs[1], outs[0]) and torch.equal(outs[2], outs[0])
        a0, b0, s0 = eng.decode_streams(payload, enc.offsets, enc.sizes, enc.n_samples, enc.sample_rates, bands, 16, 4096)
        ref_audio = a0[:int(enc.n_samples.sum()) * bands * 4].clone()
        a1, b1, s1 = eng.decode_streams(payload, enc.offsets, enc.sizes, enc.n_samples, enc.sample_rates, bands, 16, 4096, index=enc.index())
        assert list(s1[:3]) == [0, 0, 0] and torch.equal(a1[:ref_audio.numel()], ref_audio)
        # wrong index: one subframe offset moved, one frame size changed -> noticed, decoded by scanning, same pixels
        for which in ("sub", "frame"):
            fb, sb = enc.frame_bytes.clone(), enc.sub_bitoff.clone()
            if which == "sub" and bands > 1:
                sb[bands * 3 + 1] += 8
            else:
                fb[2] += 1
                fb[3] -= 1
            out = torch.zeros_like(raster)
            st = eng.decode_tiles(payload, enc.offsets, enc.sizes, tiles, enc.sample_rates, enc.minmax, 32767.0, out, 16, 4096, index=(fb, sb))
            assert list(st[:3]) == [0, 0, 0] and torch.equal(out, outs[0])
    # container: the block is there, is found again, and tiles decode through it
    out = tmp_path / "idx.flac"
    SpatialFLACEncoder(tile_size=256).encode(GOLDEN / "sample_rgb.tif", out, streaming=True)
    s = SpatialFLACStreamer(out)
    blob = out.read_bytes()
    f = s.spatial_index.frames[0]
    h = flacfmt.parse_header(blob[s.header_size + f.byte_offset: s.header_size + f.byte_offset + f.byte_size])
    got = flacfmt.unpack_seek_index(h.applications[flacfmt.SEEK_INDEX_ID], 3, 4096, 16)
    assert got is not None and int(got[0].sum()) == f.byte_size - h.first_frame_offset and got[1].size == 48


def test_scan_path_decode_under_sm_contention_and_two_launch_mode(nat, torch_cuda, monkeypatch):
    """VERDICT r1 item 9 / ADVICE: the fused skim + decode launch waits inside the grid for offsets that skim CTAs publish.
    (a) With most of the device held by a long-running filler kernel (so the decode grid becomes resident a few CTAs at a
    time) no thread may time out and the result must be right; (b) the separate-skim-launch mode gives the same pixels; (c) an
    engine that sees a time-out switches to that mode by itself."""
    torch = torch_cuda
    from flac_raster_b200.engine import Engine, tile_grid
    from flac_raster_b200.synth import sentinel2_like
    eng = Engine()
    raster = sentinel2_like(2048, 2048, 8)
    tiles = tile_grid(2048, 2048, 512)
    enc = eng.encode_tiles(raster, tiles, 5)
    payload = torch.cat([enc.payload, torch.zeros(64, dtype=torch.uint8, device="cuda")])

    def run():
        out = torch.zeros_like(raster)
        st = eng.decode_tiles(payload, enc.offsets, enc.sizes, tiles, enc.sample_rates, enc.minmax, 32767.0, out, 16, 4096)   # no index: scan path
        return st, out

    st, ref = run()
    assert list(st[:3]) == [0, 0, 0] and st[5] == 0 and torch.equal(ref.view(torch.int16), raster.view(torch.int16))
    # (a) 140 of the 148 SMs blocked for 30 ms by CTAs that take (almost) all the shared memory of an SM
    side = torch.cuda.Stream()
    nat.check(nat.lib().frb_debug_spin(140, 200 * 1024, 30_000_000, side.cuda_stream), "frb_debug_spin")
    st, out = run()
    side.synchronize()
    assert list(st[:3]) == [0, 0, 0] and st[5] == 0 and torch.equal(out, ref)
    # ... and with every SM taken for a while (the decode grid has to wait, then starts in whatever order the hardware picks)
    nat.check(nat.lib().frb_debug_spin(148, 200 * 1024, 5_000_000, side.cuda_stream), "frb_debug_spin")
    st, out = run()
    side.synchronize()
    assert list(st[:3]) == [0, 0, 0] and st[5] == 0 and torch.equal(out, ref)
    # (b) skim as its own launch
    eng._two_launch = True
    st, out = run()
    assert list(st[:3]) == [0, 0, 0] and st[5] == 0 and torch.equal(out, ref)
    a2, _, s2 = eng.decode_streams(payload, enc.offsets, enc.sizes, enc.n_samples, enc.sample_rates, 8, 16, 4096)
    eng._two_launch = False
    a1, _, s1 = Engine().decode_streams(payload, enc.offsets, enc.sizes, enc.n_samples, enc.sample_rates, 8, 16, 4096)
    n = int(enc.n_samples.sum()) * 8 * 4
    assert list(s2[:3]) == [0, 0, 0] and torch.equal(a1[:n], a2[:n])
    # (c) a reported time-out flips the engine into two-launch mode and the call is repeated
    real = eng._download
    calls = {"n": 0}

    def fake(t, dtype, count):
        r = real(t, dtype, count)
        if count == 8 and calls["n"] == 0:
            calls["n"] += 1
            r = r.copy()
            r[5] = 3
        return r

    monkeypatch.setattr(eng, "_download", fake)
    st, out = run()
    assert eng._two_launch and st[5] == 0 and torch.equal(out, ref)


def test_streamer_fast_path_equals_python_parse_path(nat, tmp_path, monkeypatch):
    """get_tiles_by_bbox: the C metadata walk + index gather + zero-copy result buffer must hand out exactly what the
    per-tile Python parse hands out (same pixels, same metadata dicts), for multi-band ragged tiles with a nodata value and
    for single-band equal tiles (which come back as views of one result buffer)."""
    from flac_raster_b200 import SpatialFLACEncoder, SpatialFLACStreamer
    from flac_raster_b200.tiffio import read_geotiff, write_geotiff
    rng = np.random.default_rng(11)
    yy, xx = np.mgrid[0:333, 0:420]
    rgb = np.stack([(1000 + 400 * np.sin(xx / 19.0 + b) * np.cos(yy / 13.0) + rng.integers(-9, 9, xx.shape)).astype(np.uint16) for b in range(3)])
    write_geotiff(tmp_path / "rgb.tif", rgb, (30.0, 0.0, 4e5, 0.0, -30.0, 5e6), "EPSG:32633", 65535.0)
    dem = (2000 * np.sin(xx[:256, :384] / 31.0)).astype(np.int16)[None]
    write_geotiff(tmp_path / "dem.tif", dem, None, None, None)
    # three bands, tiles all of one size: handed out as views of a (tile, band, h, w) result block
    uni = np.stack([(500 + 300 * np.cos(xx[:256, :384] / 11.0 + b) + rng.integers(-4, 4, (256, 384))).astype(np.int16) for b in range(3)])
    write_geotiff(tmp_path / "uni.tif", uni, (30.0, 0.0, 4e5, 0.0, -30.0, 5e6), "EPSG:32633", None)
    for name, ts, src in (("rgb", 128, rgb), ("dem", 128, dem), ("uni", 128, uni)):
        out = tmp_path / f"{name}.flac"
        SpatialFLACEncoder(tile_size=ts).encode(tmp_path / f"{name}.tif", out, streaming=True)
        s = SpatialFLACStreamer(out)
        fast = s.get_tiles_by_bbox(-1e12, -1e12, 1e12, 1e12)
        monkeypatch.setenv("FRB_SLOW_TILE_PARSE", "1")
        slow = s.get_tiles_by_bbox(-1e12, -1e12, 1e12, 1e12)
        monkeypatch.delenv("FRB_SLOW_TILE_PARSE")
        assert len(fast) == len(slow) == len(s.spatial_index.frames)
        for (a, ma), (b, mb) in zip(fast, slow):
            assert a.dtype == b.dtype and np.array_equal(a, b) and a.flags["C_CONTIGUOUS"]
            assert ma == mb, (ma, mb)
            w = ma["window"]
            assert np.array_equal(a, src[:, w["row_off"]:w["row_off"] + w["height"], w["col_off"]:w["col_off"] + w["width"]])
        one, m1 = s.get_tile_by_id(1)
        assert np.array_equal(one, fast[1][0]) and m1 == fast[1][1]
        again = s.get_tiles_by_bbox(-1e12, -1e12, 1e12, 1e12)          # earlier results must survive later calls
        assert all(np.array_equal(a, b) for (a, _), (b, _) in zip(fast, slow)) and len(again) == len(fast)


def test_grouped_bbox_decode_equals_one_batch(nat, tmp_path, monkeypatch):
    """Big bbox queries are cut into groups that are pipelined over two PCIe directions (SpatialFLACStreamer._decode_grouped: a
    background thread reads and uploads group g+1 on its own stream while group g is decoded and downloaded).  Forced here on a
    small container (tiny group size): same tiles, same order, same metadata as the one-batch path, also on a second call
    (buffer reuse) and for ragged multi-band tiles."""
    from flac_raster_b200 import SpatialFLACEncoder, SpatialFLACStreamer
    from flac_raster_b200.tiffio import write_geotiff
    rng = np.random.default_rng(23)
    yy, xx = np.mgrid[0:700, 0:900]
    for name, bands, dt in (("one", 1, np.int16), ("three", 3, np.uint16)):
        src = np.stack([(3000 + 900 * np.sin(xx / 23.0 + b) * np.cos(yy / 17.0) + rng.integers(-20, 20, xx.shape)).astype(dt) for b in range(bands)])
        write_geotiff(tmp_path / f"{name}.tif", src, (10.0, 0.0, 3e5, 0.0, -10.0, 4e6), "EPSG:32633", None)
        out = tmp_path / f"{name}.flac"
        SpatialFLACEncoder(tile_size=64).encode(tmp_path / f"{name}.tif", out, streaming=True)
        s = SpatialFLACStreamer(out)
        assert len(s.spatial_index.frames) == 11 * 15
        monkeypatch.setenv("FRB_NO_GROUPED_DECODE", "1")
        whole = s.get_tiles_by_bbox(-1e12, -1e12, 1e12, 1e12)
        monkeypatch.delenv("FRB_NO_GROUPED_DECODE")
        monkeypatch.setattr(SpatialFLACStreamer, "GROUP_BYTES", 64 << 10)
        calls = []
        orig = SpatialFLACStreamer._decode_grouped
        monkeypatch.setattr(SpatialFLACStreamer, "_decode_grouped", lambda self, fr: (calls.append(len(fr)), orig(self, fr))[1])
        for _ in range(2):
            grouped = s.get_tiles_by_bbox(-1e12, -1e12, 1e12, 1e12)
            assert len(grouped) == len(whole) == 165
            for (a, ma), (b, mb) in zip(grouped, whole):
                assert a.dtype == b.dtype and np.array_equal(a, b) and ma == mb
                w = ma["window"]
                assert np.array_equal(a, src[:, w["row_off"]:w["row_off"] + w["height"], w["col_off"]:w["col_off"] + w["width"]])
        assert calls == [165, 165]
        monkeypatch.undo()


def test_tiles_over_http_ranges(nat, tmp_path, range_http_server):
    """SURVEY 8(f)3: a container behind a URL -- the tile byte ranges are fetched with concurrent Range requests straight into
    the pinned staging buffer and handed to the GPU piece by piece; results equal the local-file path, also when the server
    ignores Range headers (remote.py:166-168)."""
    from flac_raster_b200 import SpatialFLACEncoder, SpatialFLACStreamer
    from flac_raster_b200.tiffio import read_geotiff
    base, d, log = range_http_server
    src = read_geotiff(GOLDEN / "sample_dem.tif")
    SpatialFLACEncoder(tile_size=100).encode(GOLDEN / "sample_dem.tif", d / "dem.flac", streaming=True)
    (d / "norange_dem.flac").write_bytes((d / "dem.flac").read_bytes())
    local = SpatialFLACStreamer(d / "dem.flac").get_tiles_by_bbox(-1e9, -1e9, 1e9, 1e9)
    for name in ("dem.flac", "norange_dem.flac"):
        s = SpatialFLACStreamer(f"{base}/{name}")
        got = s.get_tiles_by_bbox(-1e9, -1e9, 1e9, 1e9)
        assert len(got) == len(local) == 36
        for (a, ma), (b, mb) in zip(got, local):
            assert np.array_equal(a, b) and ma == mb
        t = src.transform
        part = s.get_tiles_by_bbox(t[2] + 250 * t[0], t[5] + 350 * t[4], t[2] + 350 * t[0], t[5] + 250 * t[4])    # tiles (2..3, 2..3)
        assert sorted(m["frame_id"] for _, m in part) == [14, 15, 20, 21]
        for tile, m in part:
            w = m["window"]
            assert np.array_equal(tile, src.data[:, w["row_off"]:w["row_off"] + w["height"], w["col_off"]:w["col_off"] + w["width"]])
        one, _ = s.get_tile_by_id(35)
        assert np.array_equal(one, src.data[:, 500:, 500:])
    assert any(r and r.startswith("bytes=") for r in log)
