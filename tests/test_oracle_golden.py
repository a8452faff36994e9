"""CPU suite part 1: the oracle is pinned against the reference's golden vectors (SURVEY.md 8c)."""
import hashlib
import json

import numpy as np
import pytest

from conftest import GOLDEN, signal_cases


def test_crc_known_answers(oracle):
    # CRC-8 (poly 0x07) and CRC-16 (poly 0x8005, init 0, MSB first) check values for "123456789"
    assert oracle.crc8(b"123456789") == 0xF4
    assert oracle.crc16(b"123456789") == 0xFEE8


def test_decode_golden_rgb_matches_kat(oracle):
    """sample_rgb.flac (libFLAC 1.4.3 via pyflac) decodes to the md5 recorded in SURVEY.md 8c."""
    data = (GOLDEN / "sample_rgb.flac").read_bytes()
    pcm, info, descs = oracle.decode(data, want_descs=True)
    assert (info.sample_rate, info.channels, info.bps, info.n_frames) == (44100, 3, 16, 16)
    assert info.first_frame_offset == 86 and info.total_samples_streaminfo == 0
    assert pcm.shape == (65536, 3)
    assert hashlib.md5(pcm.astype("<i2").tobytes()).hexdigest() == "4bf5483c1452f8c591c813b52db99491"
    assert len(descs) == 48


def test_golden_rgb_equals_reference_normalisation(oracle):
    """decode(sample_rgb.flac) == normalize_to_audio(sample_rgb.tif): the reference's own KAT."""
    from flac_raster_b200.tiffio import read_geotiff
    from oracle import normalization_oracle as no
    r = read_geotiff(GOLDEN / "sample_rgb.tif")
    interleaved = r.data.transpose(1, 2, 0).reshape(-1, 3)          # converter.py:99-110
    audio, params = no.normalize_to_audio(interleaved, 16)
    pcm, _ = oracle.decode((GOLDEN / "sample_rgb.flac").read_bytes())
    assert np.array_equal(audio.astype(np.int32), pcm)
    assert (params["data_min"], params["data_max"]) == (1.0, 255.0)


def test_oracle_encoder_reproduces_libflac_golden_bytes(oracle, rgb_pcm):
    """The libFLAC-1.4.3-procedure restatement emits the golden's 178 857 frame bytes exactly."""
    golden = (GOLDEN / "sample_rgb.flac").read_bytes()
    enc, fs, descs = oracle.encode(rgb_pcm, 16, 44100, 5, 4096, want_descs=True)
    payload = enc[len(enc) - int(fs.sum()):]
    assert int(fs.sum()) == 178857
    assert payload == golden[86:]
    _, _, gdescs = oracle.decode(golden, want_descs=True)
    for a, b in zip(gdescs, descs):
        for k in ("type", "order", "wasted", "precision", "shift", "coefs", "partition_order", "params", "nbits"):
            assert a[k] == b[k]


def test_decode_golden_dem_multistream(oracle):
    """sample_dem.flac: 4 concatenated 32-bps streams (legacy --spatial), tags + padding in stream 0."""
    data = (GOLDEN / "sample_dem.flac").read_bytes()
    pos, starts = 0, []
    while pos < len(data):
        pcm, info = oracle.decode(data[pos:])
        assert (info.channels, info.bps, info.n_frames) == (1, 32, 16)
        assert pcm.shape == (65536, 1) and not pcm.any()
        starts.append(pos)
        pos += int(info.bytes_consumed)
    assert starts == [0, 10426, 18880, 27334]


def test_normalization_oracle_matches_reference_vectors():
    """numpy restatement == outputs of the real reference module (tests/golden/make_golden.py)."""
    from oracle import normalization_oracle as no
    z = np.load(GOLDEN / "normalization_vectors.npz")
    keys = sorted(set(k.rsplit("__", 1)[0] for k in z.files if k.endswith("__in")))
    assert len(keys) == 26
    for k in keys:
        x, a, b, p = z[k + "__in"], z[k + "__audio"], z[k + "__back"], z[k + "__params"]
        a2, pp = no.normalize_to_audio(x.reshape(-1, 3), int(p[2]))
        assert a2.dtype == a.dtype and np.array_equal(a2, a), k
        assert pp["scale_factor"] == int(p[3])
        b2 = no.denormalize_from_audio(a2, pp["data_min"], pp["data_max"], pp["original_dtype"], pp["scale_factor"])
        assert b2.dtype == b.dtype and np.array_equal(b2, b, equal_nan=True), k
    rates = [no.calculate_audio_params(tuple(s), np.uint16)[0] for s in z["audio_params_shapes"]]
    assert rates == list(z["audio_params_rates"])


@pytest.mark.parametrize("level", [0, 1, 2, 3, 4, 5, 6, 7, 8])
def test_oracle_roundtrip_all_levels(oracle, level):
    for name, (x, bps) in signal_cases().items():
        enc, fs = oracle.encode(x, bps, 48000, level)
        dec, info = oracle.decode(enc)
        assert np.array_equal(dec, x), (name, level)
        assert info.crc16_errors == 0 and info.n_frames == len(fs)
        # never worse than VERBATIM + headers
        assert len(enc) <= x.size * (bps // 8) + 16 * x.shape[1] * len(fs) + 32 * len(fs) + 256


def test_oracle_streams_accepted_by_ffmpeg(oracle):
    """A second, unrelated production decoder (FFmpeg libavcodec) accepts the oracle's streams: every stream is byte for
    byte one that FFmpeg decoded to the input samples (tests/golden/ffmpeg_decoded.json, made by make_ffmpeg_golden.py),
    and where the bundled FFmpeg libraries are installed they decode it again."""
    from oracle import ffmpeg_flac as ff
    golden = json.loads((GOLDEN / "ffmpeg_decoded.json").read_text())["oracle_level5"]
    live = ff.available()
    cases = {k: v for k, v in signal_cases().items() if k != "tiny3"}        # FFmpeg refuses blocksize < 16
    assert set(golden) == set(cases)
    for name, (x, bps) in cases.items():
        enc, _ = oracle.encode(x, bps, 48000, 5, finalize=True)
        assert hashlib.md5(enc).hexdigest() == golden[name]["stream_md5"], name
        assert hashlib.md5(np.ascontiguousarray(x, dtype="<i4").tobytes()).hexdigest() == golden[name]["decoded_md5"], name
        if live:
            assert np.array_equal(ff.decode_bytes(enc, x.shape[1]), x), name


def test_oracle_rejects_corruption(oracle):
    data = bytearray((GOLDEN / "sample_rgb.flac").read_bytes())
    data[5000] ^= 0x10
    with pytest.raises(ValueError):
        oracle.decode(bytes(data))


def test_oracle_mid_side_presets(oracle):
    """The restated stereo decorrelation of libFLAC's presets: none at levels 0 and 3; levels 1 and 4 ("loose") decide
    every sample_rate*0.4/blocksize frames and keep independent or mid/side in between; the others choose among all four
    assignments per frame; turning the search off can only make the stream larger."""
    x, bps = signal_cases()["stereo16_corr"]
    for level in range(9):
        enc, fs, descs = oracle.encode(x, bps, 44100, level, want_descs=True)
        dec, _ = oracle.decode(enc)
        assert np.array_equal(dec, x)
        assign = [d["ch_assign"] for d in descs[::2]]
        if level in (0, 3):
            assert set(assign) == {1}, (level, assign)
            continue
        plain, _ = oracle.encode(x, bps, 44100, level, mid_side=False)
        assert len(enc) < len(plain), level
        if level in (1, 4):
            lf = int(44100 * 0.4 / 4096 + 0.5)                        # 4 frames per decision
            for k, a in enumerate(assign):
                if k % lf:
                    assert a in (1, 10) and a == (1 if assign[k - k % lf] == 1 else 10), (level, k, assign)
        else:
            assert {8, 9, 10} <= set(assign), (level, assign)           # left/side, right/side and mid/side all occur
