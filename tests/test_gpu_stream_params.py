"""GPU suite (-m gpu): the codec at the stream parameters the raster path never uses.

The tile path always codes blocksize 4096 at 44.1/48/96/192 kHz with 16- or 32-bps frames; the public encoder and decoder take
much more (encoder: blocksize 16-4096, any rate up to 1048575 Hz; decoder: blocksize 16-65535, 4-32 bps), and every other
blocksize goes through the one-kernel encoder for every frame.  Each case here is checked against the in-tree C oracle: the
GPU frames are the oracle's bytes, the oracle decodes them back, the GPU decodes them back, and the GPU decodes the oracle's
streams (other encoders' blocksizes and bit depths) to the oracle's samples.
"""
import ctypes as C
import functools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

BLOCKSIZES = [16, 17, 64, 96, 192, 255, 256, 257, 576, 1000, 1001, 1152, 2304, 4095]
CHANNELS = [1, 2, 3, 8]
GRID_RATES = [44100, 48000, 32000, 96000, 11025]
# levels 1 and 4 ("loose" mid/side) decide every int(rate * 0.4 / blocksize + 0.5) frames; these give groups of 17, 23, 17 and
# 6 frames, each one frame longer than without the + 0.5
LOOSE = [(192, 8000), (192, 11025), (1152, 48000), (576, 8000)]


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


# ------------------------------------------------------------------ signals
def tone_noise(n, ch, seed, scale=1):
    """9000 sin(t/40) + 3000 sin(t/7.3) + U(-40, 40) per channel (slightly detuned per channel): LPC wins at every blocksize,
    where a random walk or a pure sine gives FIXED subframes at small blocksizes.  scale=256 keeps it inside 24 bits."""
    rng = np.random.default_rng(seed)
    t = np.arange(n, dtype=np.float64)
    cols = [np.round((9000 * np.sin(t / (40.0 + 3 * c) + c) + 3000 * np.sin(t / (7.3 + 0.4 * c)) + rng.uniform(-40, 40, n)) * scale)
            for c in range(ch)]
    return np.stack(cols, axis=1).astype(np.int32)


def stereo_segments(n, seed):
    """Two channels whose best stereo decorrelation changes every ~1.3 loose groups: left smooth and right = left + noise
    (left/side), the mirror (right/side), anti-correlated (mid/side) and unrelated channels (independent)."""
    rng = np.random.default_rng(seed)
    t = np.arange(n, dtype=np.float64)
    smooth = 7000 * np.sin(t / 53.0) + 2500 * np.sin(t / 9.1)
    other = 6000 * np.sin(t / 31.0 + 1.0) + rng.uniform(-300, 300, n)
    L, R = np.empty(n), np.empty(n)
    pos, kind = 0, 0
    while pos < n:
        end = min(n, pos + int(rng.integers(n // 6, n // 4)))
        s = slice(pos, end)
        m = end - pos
        if kind == 0:
            L[s] = smooth[s]; R[s] = smooth[s] + rng.integers(-6, 7, m)
        elif kind == 1:
            R[s] = smooth[s]; L[s] = smooth[s] + rng.integers(-6, 7, m)
        elif kind == 2:
            L[s] = smooth[s] + rng.integers(-20, 21, m); R[s] = -L[s] + rng.integers(-4, 5, m)
        else:
            L[s] = smooth[s]; R[s] = other[s]
        pos, kind = end, (kind + 1) % 4
    return np.clip(np.stack([L, R], axis=1), -32767, 32767).astype(np.int32)


def full_range(n, ch, bits, seed):
    """Tone + noise at 70 % of full scale for `bits`-bit audio, with runs of the extreme values (both signs) and, for two
    channels, runs of left = max / right = min: the side channel L - R then needs bits + 1 bits."""
    lo, hi = -(1 << (bits - 1)), (1 << (bits - 1)) - 1
    x = tone_noise(n, ch, seed).astype(np.float64) / 12100.0 * 0.7 * hi
    x = np.round(x).astype(np.int64)
    rng = np.random.default_rng(seed + 1)
    for c in range(ch):
        a = int(rng.integers(0, max(1, n - 40)))
        x[a:a + 20, c] = hi
        x[a + 20:a + 40, c] = lo
    if ch == 2:
        x[:, 1] = x[:, 0] + rng.integers(-3, 4, n)                 # correlated: the side forms win
        a = int(rng.integers(0, max(1, n - 30)))
        x[a:a + 30, 0], x[a:a + 30, 1] = hi, lo
    return np.clip(x, lo, hi).astype(np.int32)


# ------------------------------------------------------------------ helpers
def _header(B, rate, ch, bps, n):
    from flac_raster_b200 import flacfmt
    return flacfmt.build_header(flacfmt.StreamInfo(B, B, 0, 0, rate, ch, bps, n))


def _frames(enc, fs):
    return enc[len(enc) - int(fs.sum()):]


@functools.lru_cache(maxsize=None)
def _grid_case(B, i):
    """Case i of blocksize B's row of the grid: (x, bps, rate, level, loose group length or 0).  Cases 0-8 are levels 0-8 with the
    channel count, stream length, sample format and rate rotating; the loose-group streams follow for the blocksizes in LOOSE."""
    b = BLOCKSIZES.index(B)
    k = max(3, 3000 // B)
    if i < 9:
        level = i
        ch = CHANNELS[(i + b) % 4]
        n = [k * B, k * B + 1, k * B + B - 1, (2 * B) // 3][(i // 2 + b) % 4]
        bps = 32 if (i + b) % 3 == 2 else 16
        x = tone_noise(n, ch, seed=100 * b + i, scale=256 if bps == 32 else 1)
        return x, bps, GRID_RATES[(i + 2 * b) % len(GRID_RATES)], level, 0
    loose = [r for bb, r in LOOSE if bb == B]
    rate = loose[(i - 9) // 2]
    level = 1 if i % 2 else 4
    lf = int(rate * 0.4 / B + 0.5)
    return stereo_segments(lf * B * 4 + B // 3, seed=7 * b + i), 16, rate, level, lf


def _grid_ids(B):
    return list(range(9 + 2 * sum(1 for bb, _ in LOOSE if bb == B)))


@functools.lru_cache(maxsize=None)
def _oracle_encode(B, i):
    from oracle import flac_oracle
    x, bps, rate, level, _ = _grid_case(B, i)
    return flac_oracle.encode(x, bps, rate, level, blocksize=B, mid_side=(bps == 16), want_descs=True)


def _check_encode(nat, oracle, x, bps, rate, level, B, oracle_out=None, what=""):
    """GPU frames vs the oracle's: same bytes and frame sizes, decoded back by the oracle and by the GPU.  The one tolerated
    difference is the documented 32-bps tone class (DESIGN.md section 4, "Encoder exactness"): the LPC coefficients of a nearly
    pure 24-bit tone may move by a step; everything else (subframe types, precision, all other subframes) must agree."""
    n, ch = x.shape
    payload, fs = nat.host_encode(x, bps, rate, level, B)
    oenc, ofs, od = oracle_out if oracle_out is not None else oracle.encode(x, bps, rate, level, blocksize=B, mid_side=(bps == 16),
                                                                            want_descs=True)
    assert int(fs.sum()) == len(payload) and len(fs) == (n + B - 1) // B, what
    dec, _, gd = oracle.decode(_header(B, rate, ch, bps, n) + bytes(payload), want_descs=True)
    assert np.array_equal(dec, x), what
    back = nat.host_decode(payload, ch, bps, B, rate, n)
    assert np.array_equal(back, x), what
    if bytes(payload) == _frames(oenc, ofs):
        assert list(fs) == list(ofs), what
        return od
    assert bps == 32, what
    assert len(gd) == len(od) and len(payload) <= 1.01 * int(ofs.sum()) + 16, what
    for a, b in zip(gd, od):
        if any(a[k] != b[k] for k in ("type", "order", "coefs", "partition_order", "params", "shift", "precision", "ch_assign")):
            assert a["type"] == 3 and b["type"] == 3 and a["precision"] == b["precision"], (what, a["frame"], a["channel"])
    return od


# ------------------------------------------------------------------ a. encoder parity over the grid
@pytest.mark.parametrize("B", BLOCKSIZES)
def test_encode_grid_matches_oracle(nat, oracle, B):
    """Levels 0-8 at blocksize B with 1, 2, 3 and 8 channels, lengths k*B, k*B+1, k*B+B-1 and below B, 16-bit and 24-bit-in-32
    audio, plus two-channel loose-mid/side streams of four groups: byte parity with the oracle and both decoders."""
    for i in _grid_ids(B):
        x, bps, rate, level, lf = _grid_case(B, i)
        _check_encode(nat, oracle, x, bps, rate, level, B, _oracle_encode(B, i), what=(B, i, x.shape, bps, rate, level))


def test_encode_grid_covers_the_blocksize_dependent_decisions(oracle):
    """What the grid above holds, read from the oracle's subframe descriptions, so that it cannot shrink to FIXED-only
    subframes unnoticed: LPC at every 16-bit coefficient precision of libFLAC's blocksize table (7-11) and at the 32-bit ones
    (13, 14), partition orders above 0, and left/side, right/side and mid/side chosen at the start of loose groups longer
    than 5 frames."""
    prec = {16: set(), 32: set()}
    orders, loose_assign = set(), set()
    for B in BLOCKSIZES:
        for i in _grid_ids(B):
            x, bps, rate, level, lf = _grid_case(B, i)
            _, _, descs = _oracle_encode(B, i)
            for d in descs:
                if d["type"] == 3:
                    prec[bps].add(d["precision"])
                orders.add(d["partition_order"])
                if lf > 5 and d["frame"] % lf == 0:
                    loose_assign.add(d["ch_assign"])
                if lf and d["frame"] % lf:
                    first = descs[(d["frame"] - d["frame"] % lf) * 2]["ch_assign"]
                    assert d["ch_assign"] == (1 if first == 1 else 10), (B, i, d["frame"])
    assert {7, 8, 9, 10, 11} <= prec[16], prec
    assert {13, 14} <= prec[32], prec
    assert max(orders) >= 3, orders
    assert {8, 9, 10} <= loose_assign, loose_assign


# ------------------------------------------------------------------ b. every sample-rate code
RATES = [8000, 11025, 22050, 37800, 44100, 88200, 176400, 1000, 255000, 65535, 655350, 700001, 1048575]


@pytest.mark.parametrize("B", [1000, 1152])
def test_every_sample_rate_code(nat, oracle, B):
    """Rates with their own code (1-11), kHz (12), Hz (13), tens of Hz (14) and none (0: taken from STREAMINFO), at a blocksize
    with a 16-bit header hint (1000) and one with a code of its own (1152): parity, both decoders, and the probe path."""
    for j, rate in enumerate(RATES):
        x = tone_noise(3 * B + 100 + j, 1 + j % 2, seed=j)
        _check_encode(nat, oracle, x, 16, rate, 5, B, what=(B, rate))
        payload, _ = nat.host_encode(x, 16, rate, 5, B)
        assert np.array_equal(nat.host_decode(payload, x.shape[1], 16, B, rate, 0), x), (B, rate)


def test_three_byte_frame_numbers(nat, oracle):
    """Blocksize 16 with 2100 frames: frame numbers 2048 and up take a 3-byte UTF-8 code (frame header 8 bytes + hint)."""
    x = tone_noise(16 * 2100 - 3, 1, seed=5)
    for level in (0, 5):
        _check_encode(nat, oracle, x, 16, 44100, level, 16, what=level)
        payload, _ = nat.host_encode(x, 16, 44100, level, 16)
        assert np.array_equal(nat.host_decode(payload, 1, 16, 16, 44100, 0), x)


# ------------------------------------------------------------------ c. tiny frames
def test_tiny_frames_many_per_chunk(nat, oracle):
    """Blocksize 16, constant and near-constant mono and stereo: frames of 12-20 bytes, several frame starts in every 16-byte
    chunk of the payload (frame assembly, sync scan, probe).  A damaged byte anywhere is reported, never decoded."""
    rng = np.random.default_rng(3)
    n = 16 * 3000 + 5
    cases = {
        "const1": np.full((n, 1), -1234, dtype=np.int32),
        "near1": (500 + (rng.random((n, 1)) < 0.01) * rng.integers(-3, 4, (n, 1))).astype(np.int32),
        "const2": np.tile(np.array([[77, -32767]], dtype=np.int32), (n, 1)),
        "near2": (np.array([[3000, 2990]]) + (rng.random((n, 2)) < 0.02) * rng.integers(-2, 3, (n, 2))).astype(np.int32),
    }
    for name, x in cases.items():
        ch = x.shape[1]
        for level in (0, 1, 5, 8):
            _check_encode(nat, oracle, x, 16, 48000, level, 16, what=(name, level))
        payload, fs = nat.host_encode(x, 16, 48000, 5, 16)
        assert np.median(fs) <= (13 if ch == 1 else 17) and len(fs) == 3001, (name, np.median(fs))
        assert np.array_equal(nat.host_decode(payload, ch, 16, 16, 48000, 0), x), name
        starts = np.concatenate([[0], np.cumsum(fs)[:-1]]).astype(np.int64)
        for pos in (int(starts[1500]) + 2, int(starts[2222]) + 9, int(starts[2900] + fs[2900]) - 1, len(payload) // 2):
            bad = payload.copy()
            bad[pos] ^= 0x21
            with pytest.raises(nat.NativeError) as ei:
                nat.host_decode(bad, ch, 16, 16, 48000, n)
            assert ei.value.status in (nat.ERR_CRC, nat.ERR_BAD_STREAM), (name, pos, ei.value.status)


# ------------------------------------------------------------------ d. engine batches at other blocksizes
@pytest.mark.parametrize("B", [1001, 1152, 4095])
def test_engine_encode_audio_batches(nat, oracle, torch_cuda, B):
    """encode_audio on streams of different lengths in one batch: int16 audio (two channels, mid/side), int32 audio at 16 bps
    (three channels) and at 32 bps (one channel, 24-bit samples): every stream's bytes are the oracle's."""
    torch = torch_cuda
    from flac_raster_b200.engine import Engine
    eng = Engine()
    lengths = [3 * B + 7, B - 1, 5 * B, 2, B + 1]
    rng = np.random.default_rng(B)
    for ch, bps, dt in ((2, 16, torch.int16), (3, 16, torch.int32), (1, 32, torch.int32)):
        xs = []
        for s, n in enumerate(lengths):
            if ch == 2:
                xs.append(stereo_segments(n, seed=s) if n > 50 else tone_noise(n, 2, seed=s))
            elif bps == 16:
                xs.append(tone_noise(n, ch, seed=s))
            else:
                xs.append((np.cumsum(rng.integers(-3000, 3001, (n, ch)), axis=0) + rng.integers(-50, 51, (n, ch))).clip(-8388607, 8388607)
                          .astype(np.int32))
        planar = np.concatenate([x.T.reshape(-1) for x in xs])
        base = np.concatenate([[0], np.cumsum([x.size for x in xs])[:-1]]).astype(np.int64)
        rates = np.array([44100, 8000, 96000, 37800, 48000], dtype=np.uint32)
        audio = torch.from_numpy(planar.astype(np.int16 if dt == torch.int16 else np.int32)).cuda()
        for level in (1, 5):
            payload, offsets, sizes, fb, sb = eng.encode_audio(audio, np.array(lengths, dtype=np.int64), base, rates, ch, bps, level, B)
            host = payload.cpu().numpy()
            for s, x in enumerate(xs):
                got = host[offsets[s]:offsets[s] + sizes[s]].tobytes()
                oenc, ofs = oracle.encode(x, bps, int(rates[s]), level, blocksize=B, mid_side=(bps == 16))
                if got != _frames(oenc, ofs):
                    # only the documented 32-bps LPC rounding class may differ: decodes exactly, LPC subframes only
                    assert bps == 32, (B, ch, level, s)
                    _check_encode(nat, oracle, x, bps, int(rates[s]), level, B, what=(B, ch, level, s))
                fpt = (lengths[s] + B - 1) // B
                assert int(fb[int(sum((l + B - 1) // B for l in lengths[:s])):][:fpt].sum()) == sizes[s]


@pytest.mark.parametrize("B", [1001, 1152, 4095])
@pytest.mark.parametrize("bands", [1, 2, 3])
def test_engine_tiles_at_blocksize(nat, oracle, torch_cuda, B, bands):
    """encode_tiles(..., blocksize=B) on a ragged grid (frames start at pixel k*B: rarely a multiple of 8 inside a row):
    frames equal the oracle's; decode_tiles fused and two-step, with the seek index and by scanning, give back the raster;
    decode_streams gives back the normalised samples."""
    torch = torch_cuda
    from flac_raster_b200.engine import Engine, tile_grid
    from oracle import normalization_oracle as no
    rng = np.random.default_rng(bands * 7 + B)
    H, W = 211, 333
    yy, xx = np.mgrid[0:H, 0:W]
    planes = [3000 + 1200 * np.sin(xx / 23.0 + b) * np.cos(yy / 17.0) + rng.integers(-25, 26, (H, W)) for b in range(bands)]
    if bands == 2:
        planes[1] = planes[0] + 40 + rng.integers(-5, 6, (H, W))      # correlated bands: the stereo search picks the side forms
    x = np.stack(planes).astype(np.uint16)
    raster = torch.from_numpy(x.view(np.int16)).cuda().view(torch.uint16)
    eng = Engine()
    tiles = tile_grid(H, W, 96)                                          # 3 x 4 tiles, 19-row and 45-column edges
    for level in (1, 5):
        enc = eng.encode_tiles(raster, tiles, level, blocksize=B)
        assert enc.blocksize == B
        payload = enc.payload.cpu().numpy()
        wants = []
        for i, t in enumerate(tiles):
            r, c, h, w = (int(t[k]) for k in ("row_off", "col_off", "h", "w"))
            want, _ = no.normalize_to_audio(x[:, r:r + h, c:c + w].transpose(1, 2, 0).reshape(-1, bands), 16)
            wants.append(want.astype(np.int32))
            oenc, ofs = oracle.encode(want, 16, int(enc.sample_rates[i]), level, blocksize=B)
            assert payload[enc.offsets[i]:enc.offsets[i] + enc.sizes[i]].tobytes() == _frames(oenc, ofs), (level, i)
        dev = torch.cat([enc.payload, torch.zeros(64, dtype=torch.uint8, device="cuda")])
        n_frames = int(enc.frames_per_tile().sum())
        for fused in (True, False):
            for index in (enc.index(), None):
                out = torch.zeros_like(raster)
                st = eng.decode_tiles(dev, enc.offsets, enc.sizes, tiles, enc.sample_rates, enc.minmax, 32767.0, out, 16, B,
                                      fused=fused, index=index)
                assert list(st[:3]) == [0, 0, 0] and st[3] == n_frames and st[5] == 0, (level, fused, index is None, st)
                assert torch.equal(out.view(torch.int16), raster.view(torch.int16)), (level, fused, index is None)
        audio, base, st = eng.decode_streams(dev, enc.offsets, enc.sizes, enc.n_samples, enc.sample_rates, bands, 16, B)
        assert list(st[:3]) == [0, 0, 0], st
        a = audio[: int(enc.n_samples.sum()) * bands * 4].view(torch.int32).cpu().numpy()
        for i, want in enumerate(wants):
            got = a[base[i]: base[i] + want.size].reshape(bands, -1).T
            assert np.array_equal(got, want), (level, i)


# ------------------------------------------------------------------ e. streams from other encoders
DEC_BLOCKSIZES = [192, 255, 256, 257, 576, 1000, 1152, 2304, 4608, 8192, 16384, 32768, 65535]
DEC_BITS = [8, 10, 12, 16, 18, 20, 24]


def _handle_decode(nat, data):
    """The libFLAC-shaped decoder handle fed from memory: (frames [(blocksize, number, samples)], info, errors, ok)."""
    L = nat.lib()
    frames, errors = [], []
    pos = [0]

    def wcb(dec, frame, buffer, client):
        h = frame.contents.header
        frames.append((h.blocksize, h.number.frame_number,
                       np.column_stack([np.ctypeslib.as_array(buffer[c], shape=(h.blocksize,)).copy() for c in range(h.channels)])))
        return 0

    def rcb(dec, buf, pbytes, client):
        n = min(pbytes[0], len(data) - pos[0])
        C.memmove(buf, data[pos[0]:pos[0] + n], n)
        pos[0] += n
        pbytes[0] = n
        return 1 if pos[0] >= len(data) else 0

    w, m, er, r = nat.DEC_WRITE_CB(wcb), nat.DEC_METADATA_CB(lambda *a: None), nat.DEC_ERROR_CB(lambda d, s, c: errors.append(s)), nat.DEC_READ_CB(rcb)
    d = L.frb_stream_decoder_new()
    try:
        assert L.frb_stream_decoder_init_stream(d, nat.cb_ptr(r), None, None, None, None, nat.cb_ptr(w), nat.cb_ptr(m), nat.cb_ptr(er), None) == 0
        ok = L.frb_stream_decoder_process_until_end_of_stream(d)
        info = (L.frb_stream_decoder_get_channels(d), L.frb_stream_decoder_get_bits_per_sample(d),
                L.frb_stream_decoder_get_sample_rate(d), L.frb_stream_decoder_get_blocksize(d))
        L.frb_stream_decoder_finish(d)
        return frames, info, errors, ok
    finally:
        L.frb_stream_decoder_delete(d)


@pytest.mark.parametrize("B", DEC_BLOCKSIZES)
def test_decode_foreign_blocksizes_and_bit_depths(nat, oracle, tmp_path, B):
    """Oracle streams at blocksize B (flac -0..-2 writes 1152, FFmpeg 4608) and full-range 8- to 24-bit audio, 1, 2 (mid/side:
    the side channel needs one bit more, 25 at 24-bit) and 8 channels, levels 0, 5 and 8: the host decoder (with and without
    the sample count), FileDecoder and the decoder handle give back the samples and the frame layout."""
    from flac_raster_b200 import codec
    b = DEC_BLOCKSIZES.index(B)
    for j, bits in enumerate(DEC_BITS):
        ch = [1, 2, 8][(j + b) % 3]
        level = [0, 5, 8][(j + 2 * b) % 3]
        n = 2 * B + B // 3 + 1 if ch < 8 or B <= 8192 else B + 17
        rate = [44100, 48000, 96000][j % 3]
        x = full_range(n, ch, bits, seed=31 * b + j)
        enc, fs, descs = oracle.encode(x, bits, rate, level, blocksize=B, finalize=bool(j % 2), want_descs=True)
        what = (B, bits, ch, level)
        if ch == 2 and level:
            assert {d["ch_assign"] for d in descs} & {8, 9, 10}, what
        ref, _ = oracle.decode(enc)
        assert np.array_equal(ref, x), what
        frames = _frames(enc, fs)
        for hint in (n, 0):
            assert np.array_equal(nat.host_decode(frames, ch, bits, B, rate, hint), x), (what, hint)
        if bits in (8, 12, 16, 20, 24):                     # the bit depths decode_bytes (FileDecoder) accepts
            p = tmp_path / f"s{B}_{bits}.flac"
            p.write_bytes(enc)
            audio, r = codec.FileDecoder(str(p)).process()
            assert r == rate and audio.dtype == (np.int16 if bits == 16 else np.int32) and np.array_equal(audio, x), what
        got, info, errors, ok = _handle_decode(nat, enc)
        assert ok == 1 and errors == [] and info == (ch, bits, rate, B), (what, info, errors)
        nf = (n + B - 1) // B
        assert [(f[0], f[1]) for f in got] == [(B if k + 1 < nf else n - k * B, k) for k in range(nf)], what
        assert np.array_equal(np.concatenate([f[2] for f in got]), x), what


# ------------------------------------------------------------------ f. fused raster sink, foreign frames
@pytest.mark.parametrize("B", [4608, 8192])
@pytest.mark.parametrize("bands", [1, 3])
def test_fused_raster_sink_with_long_foreign_frames(nat, oracle, torch_cuda, B, bands):
    """Oracle 16-bit frames longer than 4096 samples decoded straight into an int16 raster of odd width by the fused launch:
    frame k starts at pixel k*B, which is neither a row start nor a multiple of 8."""
    torch = torch_cuda
    from flac_raster_b200 import _native as natmod
    from flac_raster_b200.engine import default_engine
    from oracle import normalization_oracle as no
    h, w = 23, 1151
    x = tone_noise(h * w, bands, seed=B + bands)
    enc, fs = oracle.encode(x, 16, 44100, 5, blocksize=B)
    frames = _frames(enc, fs)
    eng = default_engine()
    data = torch.cat([torch.from_numpy(np.frombuffer(frames, dtype=np.uint8).copy()), torch.zeros(64, dtype=torch.uint8)]).cuda()
    tiles = np.zeros(1, dtype=natmod.TILE_DTYPE)
    tiles[0] = (0, 0, h, w)
    mn, mx = -12345.0, 20000.0
    out = torch.zeros(bands, h, w, dtype=torch.int16, device="cuda")
    st = eng.decode_tiles(data, np.array([0]), np.array([len(frames)]), tiles, np.array([44100], dtype=np.uint32),
                          np.array([[mn, mx]]), 32767.0, out, 16, B, fused=True)
    assert list(st[:3]) == [0, 0, 0] and st[3] == len(fs) and st[5] == 0, st
    want = no.denormalize_from_audio(x.astype(np.int16), mn, mx, "int16", 32767.0)
    assert np.array_equal(out.cpu().numpy(), want.T.reshape(bands, h, w))


# ------------------------------------------------------------------ g. handle encoder and StreamEncoder
def _handle_encode(nat, x, bps, rate, level, blocksize, seekable=True, verify=True):
    """Encode through the frb_stream_encoder_* handle: (file bytes, [(bytes, samples, frame)], finish rc)."""
    L = nat.lib()
    out = bytearray()
    pos = [0]
    calls = []

    def wcb(enc, buf, nbytes, samples, cur, client):
        data = C.string_at(buf, nbytes)
        calls.append((data, samples, cur))
        end = pos[0] + nbytes
        if end > len(out):
            out.extend(bytes(end - len(out)))
        out[pos[0]:end] = data
        pos[0] = end
        return 0

    def scb(enc, off, client):
        pos[0] = off
        return 0

    def tcb(enc, poff, client):
        poff[0] = pos[0]
        return 0

    w, s_, t_ = nat.WRITE_CB(wcb), nat.ENC_SEEK_CB(scb), nat.ENC_TELL_CB(tcb)
    e = L.frb_stream_encoder_new()
    try:
        for name, v in (("channels", x.shape[1]), ("bits_per_sample", bps), ("sample_rate", rate), ("compression_level", level),
                        ("blocksize", blocksize), ("verify", int(verify))):
            assert getattr(L, f"frb_stream_encoder_set_{name}")(e, v) == 1
        P = nat.cb_ptr
        assert L.frb_stream_encoder_init_stream(e, P(w), P(s_) if seekable else None, P(t_) if seekable else None, None, None) == 0
        a = np.ascontiguousarray(x, dtype=np.int32)
        assert L.frb_stream_encoder_process_interleaved(e, a.ctypes.data, a.shape[0]) == 1
        ok = L.frb_stream_encoder_finish(e)
        return bytes(out), calls, ok
    finally:
        L.frb_stream_encoder_delete(e)


@pytest.mark.parametrize("B", [1152, 192])
def test_handle_encoder_and_stream_encoder_at_blocksize(nat, oracle, B):
    """The handle (seekable, verify on) and the pyflac-shaped StreamEncoder at blocksize B: one callback per frame with
    samples == B (the last one shorter), the oracle's frame bytes, STREAMINFO min = max blocksize = B."""
    from flac_raster_b200 import codec, flacfmt
    for ch, level in ((1, 0), (2, 4), (3, 8)):
        x = stereo_segments(7 * B + 11, seed=ch) if ch == 2 else tone_noise(7 * B + 11, ch, seed=ch)
        n = x.shape[0]
        oenc, ofs = oracle.encode(x, 16, 22050, level, blocksize=B)
        want = _frames(oenc, ofs)
        blob, calls, ok = _handle_encode(nat, x, 16, 22050, level, B)
        assert ok == 1, (B, ch, level)
        fr = [c for c in calls if c[1] != 0]
        assert [(c[1], c[2]) for c in fr] == [(B, k) for k in range(7)] + [(11, 7)]
        assert b"".join(c[0] for c in fr) == want
        si = flacfmt.parse_header(blob).streaminfo
        assert (si.min_blocksize, si.max_blocksize, si.total_samples) == (B, B, n)
        assert (si.min_framesize, si.max_framesize) == (int(ofs.min()), int(ofs.max()))
        dec, _ = oracle.decode(blob)
        assert np.array_equal(dec, x)
        chunks = []
        se = codec.StreamEncoder(22050, lambda b_, nb, s, f: chunks.append((bytes(b_), s, f)), compression_level=level, blocksize=B,
                                 verify=True)
        se.process(x.astype(np.int16))
        assert se.finish() is True
        hdr = [c for c in chunks if c[1] == 0]
        assert flacfmt.parse_header(b"".join(c[0] for c in hdr)).streaminfo.max_blocksize == B
        assert [(c[1], c[2]) for c in chunks[len(hdr):]] == [(B, k) for k in range(7)] + [(11, 7)]
        assert b"".join(c[0] for c in chunks[len(hdr):]) == want


def test_blocksize_zero_follows_libflac(nat, oracle):
    """Blocksize 0 (pyflac's default): libFLAC's init_stream uses 1152 for the presets without LPC (levels 0-2) and 4096 for
    the others; the frames are the oracle's at that blocksize, through the handle and through StreamEncoder."""
    from flac_raster_b200 import codec, flacfmt
    x = tone_noise(10000, 2, seed=9)
    for level in range(9):
        B = 1152 if level <= 2 else 4096
        oenc, ofs = oracle.encode(x, 16, 44100, level, blocksize=B)
        blob, calls, ok = _handle_encode(nat, x, 16, 44100, level, 0, seekable=False, verify=False)
        assert ok == 1
        fr = [c for c in calls if c[1] != 0]
        assert flacfmt.parse_header(blob).streaminfo.max_blocksize == B, level
        assert [c[1] for c in fr[:-1]] == [B] * (len(ofs) - 1) and b"".join(c[0] for c in fr) == _frames(oenc, ofs), level
        chunks = []
        se = codec.StreamEncoder(44100, lambda b_, nb, s, f: chunks.append((bytes(b_), s)), compression_level=level)
        se.process(x.astype(np.int16))
        assert se.finish() is True
        assert b"".join(c[0] for c in chunks if c[1] != 0) == _frames(oenc, ofs), level
        assert [c[1] for c in chunks if c[1] != 0][0] == B
