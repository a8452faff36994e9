"""CPU suite: the oracle's frame headers at every blocksize, sample-rate and bit-depth code, read field by field against the
tables of RFC 9639 section 9.1 by a parser of their own (not the oracle's decoder: an encoder and a decoder that share one
mistake pass each other's round trip).  The GPU encoder is held to the oracle's bytes, so these tables bind it too."""
import hashlib
import json

import numpy as np
import pytest

from conftest import GOLDEN
from test_gpu_stream_params import BLOCKSIZES, DEC_BLOCKSIZES, RATES, full_range, tone_noise

# RFC 9639 9.1.1 - 9.1.4
BS_CODE = {192: 1, 576: 2, 1152: 3, 2304: 4, 4608: 5, 256: 8, 512: 9, 1024: 10, 2048: 11, 4096: 12, 8192: 13, 16384: 14, 32768: 15}
RATE_CODE = {88200: 1, 176400: 2, 192000: 3, 8000: 4, 16000: 5, 22050: 6, 24000: 7, 32000: 8, 44100: 9, 48000: 10, 96000: 11}
BPS_CODE = {8: 1, 12: 2, 16: 4, 20: 5, 24: 6, 32: 7}


def crc8(data: bytes) -> int:
    """CRC-8, polynomial x^8 + x^2 + x + 1, initial value 0, bit by bit."""
    c = 0
    for b in data:
        c ^= b
        for _ in range(8):
            c = ((c << 1) ^ 0x07) & 0xFF if c & 0x80 else (c << 1) & 0xFF
    return c


def parse_header(p: bytes, stream_rate: int, stream_bps: int):
    """One frame header -> dict of its fields and codes (RFC 9639 9.1)."""
    assert p[0] == 0xFF and p[1] == 0xF8, "sync code 0xFFF8 (fixed blocksize)"
    bsc, rc = p[2] >> 4, p[2] & 15
    chc, bpc, reserved = p[3] >> 4, (p[3] >> 1) & 7, p[3] & 1
    assert reserved == 0 and bsc != 0 and rc != 15 and bpc != 3 and chc <= 10
    # coded number: a leading byte with k+1 high ones announces k continuation bytes 10xxxxxx
    lead = p[4]
    k = 0 if lead < 0x80 else next(k for k in range(1, 7) if (lead << k) & 0x80 == 0) - 1
    assert lead < 0x80 or k >= 1
    num = lead & (0x3F >> k) if k else lead
    for q in range(k):
        assert p[5 + q] & 0xC0 == 0x80
        num = (num << 6) | (p[5 + q] & 0x3F)
    i = 5 + k
    if bsc == 1:
        bs = 192
    elif 2 <= bsc <= 5:
        bs = 144 << bsc
    elif bsc == 6:
        bs, i = p[i] + 1, i + 1
    elif bsc == 7:
        bs, i = (p[i] << 8 | p[i + 1]) + 1, i + 2
    else:
        bs = 1 << bsc
    table = {v: k_ for k_, v in RATE_CODE.items()}
    if rc == 0:
        rate = stream_rate
    elif rc <= 11:
        rate = table[rc]
    elif rc == 12:
        rate, i = p[i] * 1000, i + 1
    elif rc == 13:
        rate, i = p[i] << 8 | p[i + 1], i + 2
    else:
        rate, i = (p[i] << 8 | p[i + 1]) * 10, i + 2
    bps = stream_bps if bpc == 0 else {v: k_ for k_, v in BPS_CODE.items()}[bpc]
    assert crc8(p[:i]) == p[i], "CRC-8 of the frame header"
    return dict(bs_code=bsc, rate_code=rc, ch_code=chc, bps_code=bpc, number=num, number_bytes=k + 1, blocksize=bs, rate=rate,
                bps=bps, header_bytes=i + 1)


def expected_codes(n, rate):
    """The code a frame of n samples at `rate` must carry: the table's own code where it has one, else the smallest hint."""
    bsc = BS_CODE.get(n, 6 if n <= 256 else 7)
    if rate in RATE_CODE:
        rc = RATE_CODE[rate]
    elif rate % 1000 == 0 and rate <= 255000:
        rc = 12
    elif rate % 10 == 0 and rate <= 655350:
        rc = 14
    elif rate <= 65535:
        rc = 13
    else:
        rc = 0
    return bsc, rc


def check_stream(enc, fs, x, B, rate, bps):
    n, ch = x.shape
    body = enc[len(enc) - int(fs.sum()):]
    pos, total, nf = 0, 0, len(fs)
    seen = set()
    for k, size in enumerate(fs):
        want_n = B if k + 1 < nf else n - k * B
        h = parse_header(body[pos:pos + 32], rate, bps)
        bsc, rc = expected_codes(want_n, rate)
        assert (h["bs_code"], h["rate_code"], h["number"], h["blocksize"], h["rate"], h["bps"]) == (bsc, rc, k, want_n, rate, bps), (k, h)
        assert h["bps_code"] == BPS_CODE.get(bps, 0)
        assert h["ch_code"] == ch - 1 or (ch == 2 and h["ch_code"] in (8, 9, 10)), h
        utf8 = 1 if k < 0x80 else 2 if k < 0x800 else 3 if k < 0x10000 else 4
        hint = (1 if bsc == 6 else 2 if bsc == 7 else 0) + (1 if rc == 12 else 2 if rc in (13, 14) else 0)
        assert h["number_bytes"] == utf8 and h["header_bytes"] == 4 + utf8 + hint + 1, (k, h)
        seen.add((h["bs_code"], h["rate_code"], utf8))
        pos += int(size)
        total += h["blocksize"]
    assert pos == len(body) and total == n
    return seen


def test_frame_headers_at_every_encoder_blocksize_and_rate(oracle):
    """Every blocksize of the encoder grid, at every rate code (the kHz, Hz and tens-of-Hz hints and code 0): blocksize code
    and hint, rate code and hint, bit-depth code, channel code, frame number and CRC-8 are what RFC 9639 prescribes."""
    codes = set()
    for j, B in enumerate(BLOCKSIZES + DEC_BLOCKSIZES + [512, 1024, 2048, 4096]):
        for q, rate in enumerate(RATES):
            if (j + q) % 3:
                continue
            bps = [16, 32, 8, 12, 20, 24][(j + q) % 6]
            ch = 1 + (j + q) % 3
            n = 2 * B + B // 2 + 1
            x = full_range(n, ch, 24 if bps == 32 else bps, seed=j * 17 + q)
            enc, fs = oracle.encode(x, bps, rate, 5 if B <= 4608 else 0, blocksize=B)
            codes |= check_stream(enc, fs, x, B, rate, bps)
    bs_codes, rate_codes = {c[0] for c in codes}, {c[1] for c in codes}
    assert bs_codes == set(range(1, 16)), bs_codes
    assert rate_codes >= {0, 1, 2, 4, 6, 9, 12, 13, 14}, rate_codes


@pytest.mark.parametrize("bits", [10, 18])
def test_frame_headers_of_bit_depths_without_a_code(oracle, bits):
    """10- and 18-bit streams: the frame header says "see STREAMINFO" (code 0) and the stream still round-trips."""
    x = full_range(3000, 2, bits, seed=bits)
    enc, fs = oracle.encode(x, bits, 44100, 5, blocksize=1000)
    check_stream(enc, fs, x, 1000, 44100, bits)
    dec, info = oracle.decode(enc)
    assert np.array_equal(dec, x) and info.bps == bits


def test_frame_numbers_up_to_four_utf8_bytes(oracle):
    """Blocksize 16 over 70 000 frames: the coded frame number takes 1, 2, 3 and 4 bytes."""
    x = tone_noise(16 * 70000 + 3, 1, seed=2)
    enc, fs = oracle.encode(x, 16, 44100, 0, blocksize=16)
    seen = check_stream(enc, fs, x, 16, 44100, 16)
    assert {c[2] for c in seen} == {1, 2, 3, 4}


def test_stream_encoder_blocksize_zero_follows_libflac():
    """pyflac's default blocksize 0: libFLAC's init_stream takes 1152 for levels 0-2 (no LPC) and 4096 above; the STREAMINFO
    that StreamEncoder writes before any frame says so."""
    from flac_raster_b200 import codec, flacfmt
    for level in range(9):
        chunks = []
        enc = codec.StreamEncoder(44100, lambda b, n, s, f: chunks.append(bytes(b)), compression_level=level)
        enc.process(np.zeros((10, 2), dtype=np.int16))           # header written on the first process(), frames in finish()
        si = flacfmt.parse_header(b"".join(chunks)).streaminfo
        assert si.min_blocksize == si.max_blocksize == (1152 if level <= 2 else 4096), level
    chunks = []
    enc = codec.StreamEncoder(44100, lambda b, n, s, f: chunks.append(bytes(b)), compression_level=1, blocksize=576)
    enc.process(np.zeros((10, 1), dtype=np.int16))
    assert flacfmt.parse_header(b"".join(chunks)).streaminfo.max_blocksize == 576


def test_oracle_stream_params_accepted_by_ffmpeg(oracle):
    """FFmpeg libavcodec decodes oracle streams at other blocksizes, rates and bit depths to their input: every stream is
    byte for byte one FFmpeg decoded (tests/golden/ffmpeg_decoded.json, "oracle_stream_params", made by
    make_ffmpeg_golden.py), and where the bundled FFmpeg libraries are installed they decode it again."""
    import importlib.util
    from oracle import ffmpeg_flac as ff
    spec = importlib.util.spec_from_file_location("make_ffmpeg_golden", GOLDEN / "make_ffmpeg_golden.py")
    mk = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mk)
    golden = json.loads((GOLDEN / "ffmpeg_decoded.json").read_text())["oracle_stream_params"]
    live = ff.available()
    cases = dict(mk.stream_param_cases())
    assert set(golden) <= set(cases) and len(golden) >= 20
    for name, rec in golden.items():
        x, bits, rate, level, B = cases[name]
        enc, _ = oracle.encode(x, bits, rate, level, blocksize=B, finalize=True)
        assert hashlib.md5(enc).hexdigest() == rec["stream_md5"], name
        assert hashlib.md5(np.ascontiguousarray(x, dtype="<i4").tobytes()).hexdigest() == rec["decoded_md5"], name
        if live:
            assert np.array_equal(mk.ffmpeg_samples(enc, x.shape[1], bits), x), name
