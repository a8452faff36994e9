// frb_decode.cuh -- FLAC frame discovery + Rice decode + predictor restore (sm_100a).
//
// Replaces pyflac.FileDecoder.process (reference converter.py:181-182), i.e.
// libFLAC's frame_sync_/read_frame_/read_residual_partitioned_rice_/
// FLAC__lpc_restore_signal, for batches of independent fixed-blocksize streams.
//
// Kernels
//   k_sync_scan     every byte position tested for 0xFFF8 + valid header + CRC-8;
//                   hits are scattered by their coded frame number (no sort needed)
//   k_decode_frames one thread per frame, warp = 32 frames in lock-step over the
//                   sample index; decoded samples staged in a 32x33 smem tile
//                   (doubles as the LPC history) and flushed as 128-byte rows
//   k_crc16_frames  one warp per frame, lane-parallel CRC-16 with GF(2) combine
//   k_stereo_fix    undo left/side, side/right, mid/side (2-channel streams only)
#pragma once
#include "frb_common.cuh"

namespace frb {

constexpr unsigned long long kNoPos = 0xFFFFFFFFFFFFFFFFull;

// n_samples / n_frames: what is decoded of the stream.  A window read decodes a run of frames [first_frame, first_frame +
// n_frames) of a stream of total_samples samples (total_frames frames); every other call decodes whole streams
// (first_frame 0, the totals equal to the counts).
struct DecStreamDev {
    uint64_t byte_offset, byte_length, n_samples;
    int64_t audio_base;
    uint32_t sample_rate, frame_base, n_frames, first_frame;
    uint64_t total_samples;
    uint32_t total_frames, pad;
};

struct FrameHdr {
    uint32_t blocksize, sample_rate, ch_assign, bps, header_bytes;
    uint64_t number;
};

__device__ __forceinline__ uint32_t rate_from_code(uint32_t c) {
    switch (c) {
        case 1: return 88200; case 2: return 176400; case 3: return 192000; case 4: return 8000;
        case 5: return 16000; case 6: return 22050; case 7: return 24000; case 8: return 32000;
        case 9: return 44100; case 10: return 48000; case 11: return 96000;
    }
    return 0;
}

// Parse + CRC-8-check a candidate frame header at p (avail bytes readable). Fixed blocksize only.
__device__ inline bool parse_frame_header(const uint8_t *p, uint64_t avail, uint32_t stream_rate,
                                          uint32_t stream_bps, FrameHdr *h) {
    if (avail < 6) return false;
    if (p[0] != 0xFF || p[1] != 0xF8) return false;
    uint32_t b2 = p[2], b3 = p[3];
    uint32_t bsc = b2 >> 4, src = b2 & 15, chc = b3 >> 4, bpc = (b3 >> 1) & 7;
    if ((b3 & 1) || bsc == 0 || src == 15 || bpc == 3 || chc > 10) return false;
    uint32_t i = 4;
    uint32_t b0 = p[i++];
    uint64_t num; int extra;
    if (b0 < 0x80) { num = b0; extra = 0; }
    else if ((b0 & 0xE0) == 0xC0) { num = b0 & 0x1F; extra = 1; }
    else if ((b0 & 0xF0) == 0xE0) { num = b0 & 0x0F; extra = 2; }
    else if ((b0 & 0xF8) == 0xF0) { num = b0 & 0x07; extra = 3; }
    else if ((b0 & 0xFC) == 0xF8) { num = b0 & 0x03; extra = 4; }
    else if ((b0 & 0xFE) == 0xFC) { num = b0 & 0x01; extra = 5; }
    else return false;
    if (avail < (uint64_t)(i + extra + 5)) return false;
    for (int k = 0; k < extra; k++) {
        uint32_t b = p[i++];
        if ((b & 0xC0) != 0x80) return false;
        num = (num << 6) | (b & 0x3F);
    }
    h->number = num;
    if (bsc == 1) h->blocksize = 192;
    else if (bsc <= 5) h->blocksize = 576u << (bsc - 2);
    else if (bsc == 6) h->blocksize = (uint32_t)p[i++] + 1;
    else if (bsc == 7) { h->blocksize = (((uint32_t)p[i] << 8) | p[i + 1]) + 1; i += 2; }
    else h->blocksize = 256u << (bsc - 8);
    if (src == 0) h->sample_rate = stream_rate;
    else if (src <= 11) h->sample_rate = rate_from_code(src);
    else if (src == 12) h->sample_rate = (uint32_t)p[i++] * 1000u;
    else if (src == 13) { h->sample_rate = ((uint32_t)p[i] << 8) | p[i + 1]; i += 2; }
    else { h->sample_rate = (((uint32_t)p[i] << 8) | p[i + 1]) * 10u; i += 2; }
    h->ch_assign = chc;
    const uint32_t bt[8] = {0, 8, 12, 0, 16, 20, 24, 32};
    h->bps = bpc == 0 ? stream_bps : bt[bpc];
    uint8_t crc = 0;
    for (uint32_t k = 0; k < i; k++) crc = c_crc8[crc ^ p[k]];
    if (crc != p[i]) return false;
    h->header_bytes = i + 1;
    return true;
}

__global__ void k_fill_u64(unsigned long long *p, uint64_t n, unsigned long long v) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) p[i] = v;
}

// flattened grid of `parts` CTAs per stream; every thread tests the 16 byte positions of one aligned 16-byte chunk per step
// (the sync code may straddle into the next chunk: one extra word).  SIMD byte compares reject a word without a
// 0xFF 0xF8 pair in ~6 instructions; v1 tested 4 positions per two 4-byte loads (0.85 ms on C3).
__device__ __forceinline__ void sync_candidate(const uint8_t *__restrict__ bytes, const DecStreamDev &st, uint64_t pos, uint64_t start,
                                               uint64_t end, uint32_t channels, uint32_t bps, uint32_t blocksize,
                                               unsigned long long *__restrict__ frame_pos, unsigned long long *__restrict__ frame_pos2,
                                               unsigned long long *__restrict__ probe, unsigned long long *__restrict__ end_cand) {
    if (pos < start || pos + 8 > end) return;
    FrameHdr h;
    if (!parse_frame_header(bytes + pos, end - pos, st.sample_rate, bps, &h)) return;
    if (h.bps != bps || h.sample_rate != st.sample_rate) return;
    const uint32_t nch = h.ch_assign < 8 ? h.ch_assign + 1 : 2;
    if (nch != channels || h.blocksize > blocksize) return;
    if (probe) {
        atomicMax(&probe[0], (h.number << 20) | h.blocksize);
        atomicAdd(&probe[1], 1ull);
    }
    if (!frame_pos) return;
    // frame numbers are absolute: a run keeps [first_frame, first_frame + n_frames] (the last one marks where the run ends)
    if (h.number < st.first_frame || h.number >= st.total_frames || h.number > (uint64_t)st.first_frame + st.n_frames) return;
    const uint64_t expect = (h.number + 1 < st.total_frames) ? blocksize : (st.total_samples - h.number * blocksize);
    if (h.blocksize != expect) return;
    // the two smallest candidate positions per frame number: cand[f] and cand2[f] (k_sync_resolve picks between them).
    // Every position other than the final minimum is at some point the larger side of an atomicMin exchange, so the
    // minimum of those larger sides is the second smallest.
    const uint64_t k = h.number - st.first_frame;
    unsigned long long *c1 = k < st.n_frames ? &frame_pos[st.frame_base + k] : end_cand;
    unsigned long long *c2 = k < st.n_frames ? (frame_pos2 ? &frame_pos2[st.frame_base + k] : nullptr) : end_cand + 1;
    if (!c1) return;
    const unsigned long long old = atomicMin(c1, (unsigned long long)pos);
    if (c2 && old != kNoPos && old != pos) atomicMin(c2, old > pos ? old : (unsigned long long)pos);
}

// Scan path of a window read: the frame behind a run's last frame gives the run's end (candidates picked as in
// k_sync_resolve).  Written into the stream's byte_length, so that every later kernel sees a stream that ends there; a run
// whose end was not found gets length 0 and its last frame is reported missing.
__global__ void k_run_end(DecStreamDev *__restrict__ streams, uint32_t n_streams, const unsigned long long *__restrict__ cand,
                          const unsigned long long *__restrict__ end_cand) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_streams) return;
    DecStreamDev &st = streams[i];
    if ((uint64_t)st.first_frame + st.n_frames >= st.total_frames) return;      // the run reaches the end of the stream
    unsigned long long c = end_cand[2 * i];
    const unsigned long long prev = cand[st.frame_base + st.n_frames - 1], c2 = end_cand[2 * i + 1];
    if (c != kNoPos && prev != kNoPos && c <= prev && c2 != kNoPos) c = c2;
    st.byte_length = (c == kNoPos || c < st.byte_offset) ? 0 : c - st.byte_offset;
}

// A byte sequence inside some frame's payload can look like a frame header (sync code, plausible fields, CRC-8: about
// 2^-39 per byte position, ~1e-3 per 1.5 GB container).  libFLAC decodes sequentially and never looks there; a parallel
// scan that keeps the FIRST candidate per frame number is shadowed by it whenever it lies before the real frame.  Frame
// starts grow with the frame number, so a first candidate at or before the previous frame's first candidate cannot be
// the frame: the second candidate takes its place.  (A false header inside the immediately preceding frame is still
// not told apart -- 1/n_frames of the cases; the decode then reports a parse / CRC-16 error, never wrong samples.)
__global__ void __launch_bounds__(256)
k_sync_resolve(const DecStreamDev *__restrict__ streams, uint32_t n_streams, uint32_t total_frames,
               const unsigned long long *__restrict__ cand, const unsigned long long *__restrict__ cand2,
               unsigned long long *__restrict__ frame_pos) {
    const uint32_t f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= total_frames) return;
    uint32_t lo = 0, hi = n_streams - 1;
    while (lo < hi) {
        const uint32_t mid = (lo + hi + 1) >> 1;
        if (streams[mid].frame_base <= f) lo = mid; else hi = mid - 1;
    }
    unsigned long long c = cand[f];
    if (f > streams[lo].frame_base && c != kNoPos) {
        const unsigned long long prev = cand[f - 1], c2 = cand2[f];
        if (prev != kNoPos && c <= prev && c2 != kNoPos) c = c2;
    }
    frame_pos[f] = c;
}

__global__ void __launch_bounds__(256)
k_sync_scan(const uint8_t *__restrict__ bytes, const DecStreamDev *__restrict__ streams, uint32_t channels,
            uint32_t bps, uint32_t blocksize, unsigned long long *__restrict__ frame_pos,
            unsigned long long *__restrict__ frame_pos2 /* optional: second smallest candidate per frame */,
            unsigned long long *__restrict__ probe /* optional: [0]=max key, [1]=count */, uint32_t parts,
            unsigned long long *__restrict__ run_end = nullptr /* window reads: 2 candidates per stream for the frame behind the run */) {
    // flattened grid, `parts` CTAs per stream (gridDim.y stops at 65535 streams)
    const uint32_t si = blockIdx.x / parts, part = blockIdx.x - si * parts;
    const DecStreamDev st = streams[si];
    const uint64_t start = st.byte_offset, end = st.byte_offset + st.byte_length;
    const uint64_t q0 = start >> 4, q1 = (end + 15) >> 4;            // 16-byte chunks touching the stream
    const uint4 *chunks = (const uint4 *)bytes;                      // 16-byte aligned base, 16 readable bytes past the end
    const uint32_t *words = (const uint32_t *)bytes;
    for (uint64_t q = q0 + (uint64_t)part * blockDim.x + threadIdx.x; q < q1; q += (uint64_t)parts * blockDim.x) {
        const uint4 c = __ldg(chunks + q);
        // first word of the next chunk (little-endian bytes); a sync code straddling out of the stream's last chunk
        // would fail the length check anyway, so nothing is read past the 16-byte slack
        const uint32_t nxt = (q + 1 < q1) ? __ldg(words + 4 * q + 4) : 0u;
        const uint32_t w[5] = {c.x, c.y, c.z, c.w, nxt};
#pragma unroll
        for (int j = 0; j < 4; j++) {
            // byte k of word j is 0xFF and the following byte is 0xF8
            const uint32_t follow = __funnelshift_r(w[j], w[j + 1], 8);          // bytes 1,2,3 of w[j] and byte 0 of w[j+1]
            const uint32_t hit = __vcmpeq4(w[j], 0xFFFFFFFFu) & __vcmpeq4(follow, 0xF8F8F8F8u);
            if (hit == 0) continue;
#pragma unroll
            for (int k = 0; k < 4; k++)
                if (hit & (0xFFu << (8 * k)))
                    sync_candidate(bytes, st, 16 * q + 4 * j + k, start, end, channels, bps, blocksize, frame_pos, frame_pos2, probe,
                                   run_end ? run_end + 2 * si : nullptr);
        }
    }
}


#include "frb_decode_kernels.cuh"   // bit reader, skim, subframe decode, CRC-16 (inside namespace frb)


// Indexed streams: frame positions from the frame sizes of the seek index.  One CTA per stream, chunked block scan.  A
// stream whose sizes do not add up to its byte length is reported as "frames missing" (status[0]) and left unlocated.
__global__ void __launch_bounds__(256)
k_index_frame_pos(const DecStreamDev *__restrict__ streams, const uint32_t *__restrict__ frame_bytes,
                  unsigned long long *__restrict__ frame_pos, uint32_t *__restrict__ status) {
    __shared__ unsigned long long s_warp[8];
    __shared__ unsigned long long s_carry;
    const DecStreamDev st = streams[blockIdx.x];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < st.n_frames; base += blockDim.x) {
        const uint32_t i = base + threadIdx.x;
        const unsigned long long v = i < st.n_frames ? frame_bytes[st.frame_base + i] : 0ull;
        unsigned long long inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const unsigned long long t = __shfl_up_sync(0xFFFFFFFFu, inc, o); if (lane >= o) inc += t; }
        if (lane == 31) s_warp[warp] = inc;
        __syncthreads();
        unsigned long long wbase = 0, tot = 0;
#pragma unroll
        for (int w = 0; w < 8; w++) { const unsigned long long x = s_warp[w]; if (w < warp) wbase += x; tot += x; }
        const unsigned long long carry = s_carry;
        if (i < st.n_frames) frame_pos[st.frame_base + i] = st.byte_offset + carry + wbase + inc - v;
        __syncthreads();
        if (threadIdx.x == 0) s_carry = carry + tot;
        __syncthreads();
    }
    if (threadIdx.x == 0 && s_carry != st.byte_length) {
        atomicAdd(&status[0], st.n_frames);
        for (uint32_t i = 0; i < st.n_frames; i++) frame_pos[st.frame_base + i] = kNoPos;
    }
}

// one CTA per frame; only frames with ch_assign 8/9/10 do work
__global__ void __launch_bounds__(128)
k_stereo_fix(const DecStreamDev *__restrict__ streams, uint32_t n_streams, uint32_t blocksize, uint32_t total_frames,
             const uint8_t *__restrict__ frame_chassign, const unsigned long long *__restrict__ frame_pos,
             int32_t *__restrict__ audio) {
    const uint32_t f = blockIdx.x;
    if (f >= total_frames || frame_pos[f] == kNoPos) return;
    const uint32_t ca = frame_chassign[f];
    if (ca < 8 || ca > 10) return;
    uint32_t lo = 0, hi = n_streams - 1;
    while (lo < hi) {
        uint32_t mid = (lo + hi + 1) >> 1;
        if (streams[mid].frame_base <= f) lo = mid; else hi = mid - 1;
    }
    const DecStreamDev st = streams[lo];
    uint32_t k = f - st.frame_base;
    uint32_t n = (k + 1 < st.n_frames) ? blocksize : (uint32_t)(st.n_samples - (uint64_t)k * blocksize);
    int32_t *c0 = audio + st.audio_base + (int64_t)k * blocksize;
    int32_t *c1 = c0 + st.n_samples;
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
        int64_t a = c0[i], b = c1[i];
        if (ca == 8) c1[i] = (int32_t)(a - b);
        else if (ca == 9) c0[i] = (int32_t)(a + b);
        else {
            int64_t m = (a << 1) | (b & 1);
            c0[i] = (int32_t)((m + b) >> 1);
            c1[i] = (int32_t)((m - b) >> 1);
        }
    }
}

struct DecWorkspace {
    DecStreamDev *streams;
    unsigned long long *frame_pos;
    unsigned long long *frame_cand;     // scan path: smallest and second smallest candidate per frame, 2 x (total_frames + 1)
    uint8_t *chassign;
    uint32_t *sub_bitoff;      // only used when channels > 1
    unsigned long long *run_end;        // scan path of a window read: 2 candidates per stream for the frame behind its run
};
static inline size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }
static inline size_t dec_ws_layout(uint32_t n_streams, uint32_t channels, uint64_t total_frames, void *base, DecWorkspace *w) {
    size_t off = 0;
    uint8_t *b = (uint8_t *)base;
    if (w) w->streams = (DecStreamDev *)(b + off);
    off += align256(sizeof(DecStreamDev) * (size_t)n_streams);
    if (w) w->frame_pos = (unsigned long long *)(b + off);
    off += align256(8 * (size_t)(total_frames + 1));
    if (w) w->frame_cand = (unsigned long long *)(b + off);
    off += align256(16 * (size_t)(total_frames + 1));
    if (w) w->chassign = b + off;
    off += align256((size_t)total_frames + 1);
    if (w) w->sub_bitoff = (uint32_t *)(b + off);
    off += align256(4 * (size_t)(total_frames * channels + 1));
    if (w) w->run_end = (unsigned long long *)(b + off);
    off += align256(16 * (size_t)n_streams);
    return off;
}

}  // namespace frb

extern "C" int frb_decode_workspace_size(const frb_decode_params *p, uint64_t total_frames, size_t *bytes) {
    if (!p || !bytes) return FRB_ERR_INVALID_ARG;
    *bytes = frb::dec_ws_layout(p->n_streams, p->channels, total_frames, nullptr, nullptr);
    return FRB_OK;
}

namespace frb {
static int decode_streams_impl(const frb_decode_params *p, const std::vector<DecStreamDev> &hs,
                               const uint8_t *d_bytes, uint64_t total_frames, int32_t *d_audio,
                               void *d_workspace, size_t workspace_bytes, uint32_t *d_status, void *stream, const SinkCfg &sink,
                               const uint32_t *d_frame_bytes, const uint32_t *d_index_bitoff);

static int check_decode_args(const frb_decode_params *p, const void *h_streams, const uint8_t *d_bytes, uint64_t total_frames,
                             const int32_t *d_audio, const void *d_workspace, const uint32_t *d_status, const SinkCfg &sink,
                             const uint32_t *d_frame_bytes, const uint32_t *d_index_bitoff) {
    if ((d_frame_bytes == nullptr) != (d_index_bitoff == nullptr) && p && p->channels > 1) return FRB_ERR_INVALID_ARG;
    if (!p || !h_streams || !d_bytes || (!d_audio && sink.dtype < 0) || !d_workspace || !d_status) return FRB_ERR_INVALID_ARG;
    if (p->n_streams == 0 || p->channels < 1 || p->channels > FRB_MAX_CHANNELS || p->blocksize < 16 ||
        p->blocksize > 65535 || p->bps < 4 || p->bps > 32) return FRB_ERR_INVALID_ARG;
    if (total_frames == 0 || total_frames > 0x7FFFFFFFull) return FRB_ERR_INVALID_ARG;
    return FRB_OK;
}

// The sink of a decode to planar int32 audio.
static SinkCfg audio_sink() { SinkCfg sink; memset(&sink, 0, sizeof sink); sink.dtype = -1; return sink; }

// The sink of a decode straight into a (bands, H, W) raster of `dtype` at `out`.  frb_decode_tiles and frb_decode_window
// both take it from here, which is what keeps a window's pixels bit-identical to those of a whole decode.
static SinkCfg raster_sink(int dtype, double scale, const frb_tile *d_tiles, const double *d_minmax, void *out, uint32_t H, uint32_t W) {
    static const uint32_t esz[8] = {1, 1, 2, 2, 4, 4, 4, 8};
    SinkCfg sink = audio_sink();
    sink.dtype = dtype; sink.esize = esz[dtype]; sink.H = H; sink.W = W; sink.tiles = d_tiles; sink.minmax = d_minmax;
    sink.raster = (uint8_t *)out; sink.scale = scale; sink.rcp = 1.0 / scale;
    sink.fast = (scale == 32767.0 || scale == 8388607.0 || scale == 2147483647.0) ? 1 : 0;
    sink.intpath = (dtype <= FRB_I16 && scale == 32767.0) ? 1 : 0;      // integer min/max, range < 2^16, |audio| <= 32767
    return sink;
}

// One entry of the device stream table: frames [first_frame, first_frame + n_frames) of a stream of total_samples samples,
// which must lie inside the stream.  `frames`: the frames of the entries before it, which frame_base must equal.
static int dec_stream(const frb_decode_params *p, uint64_t byte_offset, uint64_t byte_length, uint64_t total_samples,
                      int64_t audio_base, uint32_t sample_rate, uint32_t frame_base, uint32_t first_frame, uint64_t n_frames,
                      uint64_t &frames, DecStreamDev &d) {
    const uint64_t all = (total_samples + p->blocksize - 1) / p->blocksize;
    if (all > 0xFFFFFFFFull || first_frame + n_frames > all || frame_base != frames) return FRB_ERR_INVALID_ARG;
    const uint64_t s0 = (uint64_t)first_frame * p->blocksize, s1 = (first_frame + n_frames) * p->blocksize;
    d.byte_offset = byte_offset; d.byte_length = byte_length; d.n_samples = (s1 < total_samples ? s1 : total_samples) - s0;
    d.audio_base = audio_base; d.sample_rate = sample_rate; d.frame_base = frame_base; d.n_frames = (uint32_t)n_frames;
    d.first_frame = first_frame; d.total_samples = total_samples; d.total_frames = (uint32_t)all; d.pad = 0;
    frames += n_frames;
    return FRB_OK;
}

static int decode_batch_impl(const frb_decode_params *p, const frb_decode_stream *h_streams,
                             const uint8_t *d_bytes, uint64_t total_frames, int32_t *d_audio,
                             void *d_workspace, size_t workspace_bytes, uint32_t *d_status, void *stream, const SinkCfg &sink,
                             const uint32_t *d_frame_bytes = nullptr, const uint32_t *d_index_bitoff = nullptr) {
    FRB_TRY(check_decode_args(p, h_streams, d_bytes, total_frames, d_audio, d_workspace, d_status, sink, d_frame_bytes, d_index_bitoff));
    // stream table (host -> device), every stream whole. Pageable source: staged by the runtime before return.
    std::vector<DecStreamDev> hs(p->n_streams);
    uint64_t frames = 0;
    for (uint32_t i = 0; i < p->n_streams; i++) {
        const frb_decode_stream &a = h_streams[i];
        FRB_TRY(dec_stream(p, a.byte_offset, a.byte_length, a.n_samples, a.audio_base, a.sample_rate, a.frame_base, 0,
                           (a.n_samples + p->blocksize - 1) / p->blocksize, frames, hs[i]));
    }
    if (frames != total_frames) return FRB_ERR_INVALID_ARG;
    return decode_streams_impl(p, hs, d_bytes, total_frames, d_audio, d_workspace, workspace_bytes, d_status, stream, sink,
                               d_frame_bytes, d_index_bitoff);
}

// the work of every decode call, on a stream table that holds whole streams or frame runs (DecStreamDev)
static int decode_streams_impl(const frb_decode_params *p, const std::vector<DecStreamDev> &hs,
                               const uint8_t *d_bytes, uint64_t total_frames, int32_t *d_audio,
                               void *d_workspace, size_t workspace_bytes, uint32_t *d_status, void *stream, const SinkCfg &sink,
                               const uint32_t *d_frame_bytes, const uint32_t *d_index_bitoff) {
    int rc = ensure_tables_impl();
    if (rc) return rc;
    DecWorkspace w;
    if (dec_ws_layout(p->n_streams, p->channels, total_frames, d_workspace, &w) > workspace_bytes) return FRB_ERR_OVERFLOW;
    if (reinterpret_cast<uintptr_t>(d_bytes) & 15u) return FRB_ERR_INVALID_ARG;   // vector loads need a 16-byte aligned base
    cudaStream_t s = (cudaStream_t)stream;
    uint64_t max_len = 0;
    bool open_runs = false;                  // a run that ends before its stream does (scan path: k_run_end finds its end)
    for (const DecStreamDev &d : hs) {
        if (d.byte_length > max_len) max_len = d.byte_length;
        if ((uint64_t)d.first_frame + d.n_frames < d.total_frames) open_runs = true;
    }
    FRB_TRY(small_upload(w.streams, hs.data(), sizeof(DecStreamDev) * hs.size(), s));   // staged in pinned memory before returning
    FRB_TRY(small_fill(d_status, 0u, 8 * sizeof(uint32_t), s));
    FRB_TRY(small_fill(w.chassign, 0u, ((size_t)total_frames + 1 + 3) & ~(size_t)3, s));
    const bool indexed = d_frame_bytes != nullptr;
    if (indexed) {
        // seek index supplied (frb_encode_index / the container's index block): frame positions are a scan of the frame sizes,
        // no byte of the streams is inspected to find them
        k_index_frame_pos<<<p->n_streams, 256, 0, s>>>(w.streams, d_frame_bytes, w.frame_pos, d_status);
        FRB_LAUNCH_CHECK("k_index_frame_pos");
    } else {
        k_fill_u64<<<grid_for(2 * (total_frames + 1), 256 * 4, kNumSMs * 4), 256, 0, s>>>(w.frame_cand, 2 * (total_frames + 1), kNoPos);
        FRB_LAUNCH_CHECK("k_fill_u64");
        if (open_runs) {
            k_fill_u64<<<1, 256, 0, s>>>(w.run_end, 2 * (uint64_t)p->n_streams, kNoPos);
            FRB_LAUNCH_CHECK("k_fill_u64");
        }
        uint64_t chunks = max_len / 16 + 2;
        uint32_t gx = (uint32_t)((chunks + 256 * 4 - 1) / (256 * 4));
        uint32_t cap = (kNumSMs * 16 + p->n_streams - 1) / p->n_streams;
        if (gx > cap) gx = cap;
        if (gx < 1) gx = 1;
        prof_begin(3, s);
        k_sync_scan<<<gx * p->n_streams, 256, 0, s>>>(d_bytes, w.streams, p->channels, p->bps, p->blocksize, w.frame_cand,
                                                      w.frame_cand + total_frames + 1, nullptr, gx, open_runs ? w.run_end : nullptr);
        prof_end(3, s);
        FRB_LAUNCH_CHECK("k_sync_scan");
        k_sync_resolve<<<(uint32_t)((total_frames + 255) / 256), 256, 0, s>>>(w.streams, p->n_streams, (uint32_t)total_frames, w.frame_cand,
                                                                            w.frame_cand + total_frames + 1, w.frame_pos);
        FRB_LAUNCH_CHECK("k_sync_resolve");
        if (open_runs) {
            k_run_end<<<(p->n_streams + 255) / 256, 256, 0, s>>>(w.streams, p->n_streams, w.frame_cand, w.run_end);
            FRB_LAUNCH_CHECK("k_run_end");
        }
    }
    // CRC-16 only needs the frame positions: it runs on a side stream and joins the caller's stream at the end.  It is launched
    // AFTER the decode kernel: CTAs of the earlier launch are placed first, so the CRC's CTAs fill the SMs only as the decode grid
    // drains -- a thread per subframe leaves a tail of ~0.4 ms in which most decode threads are done and the last ones run at the
    // speed of their dependent chains.  Launched first (as it was), the CRC's persistent CTAs took most of every SM's registers
    // and the decode CTAs queued behind them.  FRB_CRC_FIRST=1 restores the old order (A/B runs).
    static cudaStream_t side_of[64] = {nullptr};
    static cudaEvent_t fork_of[64] = {nullptr}, join_of[64] = {nullptr};
    static int crc_first = -1;
    if (crc_first < 0) { const char *e = getenv("FRB_CRC_FIRST"); crc_first = e ? atoi(e) : 0; }
    int dev = 0;
    FRB_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64) return FRB_ERR_UNSUPPORTED;
    cudaStream_t &side = side_of[dev];
    cudaEvent_t &ev_fork = fork_of[dev], &ev_join = join_of[dev];
    auto launch_crc = [&]() -> int {
        FRB_CUDA(cudaStreamWaitEvent(side, ev_fork, 0));
        const uint64_t threads = total_frames * 32;
        uint32_t crc_grid = (uint32_t)((threads + 255) / 256);
        if (crc_grid > (uint32_t)kNumSMs * 8) crc_grid = kNumSMs * 8;         // persistent: the tables are staged once per CTA
        k_crc16_frames<<<crc_grid, 256, 0, side>>>(d_bytes, w.streams, p->n_streams, p->blocksize,
                                                  (uint32_t)total_frames, w.frame_pos, d_status);
        FRB_LAUNCH_CHECK("k_crc16_frames");
        FRB_CUDA(cudaEventRecord(ev_join, side));
        return FRB_OK;
    };
    if (p->verify_crc16 & 1u) {
        if (!side) {
            FRB_CUDA(cudaStreamCreateWithFlags(&side, cudaStreamNonBlocking));
            FRB_CUDA(cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming));
            FRB_CUDA(cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming));
        }
        FRB_CUDA(cudaEventRecord(ev_fork, s));               // frame positions are ready here
        if (crc_first) FRB_TRY(launch_crc());
    }
    {
        uint32_t *sub_bitoff = nullptr;
        uint32_t n_skim_ctas = 0, skim_lanes = 32;
        if (p->channels > 1) {
            // subframes of a frame are bit-packed back to back: their starts are found by the skim CTAs of the SAME
            // launch and handed to the decode threads through sub_bitoff (kNotReady until published)
            static uint32_t skim_lanes_cfg = 0;
            if (!skim_lanes_cfg) { const char *e = getenv("FRB_SKIM_LANES"); skim_lanes_cfg = e ? (uint32_t)atoi(e) : 32u; if (skim_lanes_cfg < 1 || skim_lanes_cfg > 32) skim_lanes_cfg = 32; }
            skim_lanes = skim_lanes_cfg;
            const uint32_t frames_per_cta = (kDecThreads / 32) * skim_lanes;
            n_skim_ctas = (uint32_t)((total_frames + frames_per_cta - 1) / frames_per_cta);
            sub_bitoff = w.sub_bitoff;
            if (indexed) { n_skim_ctas = 0; sub_bitoff = const_cast<uint32_t *>(d_index_bitoff); }
            else FRB_TRY(small_fill(sub_bitoff, 0xFFFFFFFFu, 4 * (size_t)(total_frames * p->channels), s));
        }
        const uint64_t total_sub = total_frames * p->channels;
        const uint32_t dec_ctas = (uint32_t)((total_sub + kDecThreads - 1) / kDecThreads);
        const bool big = p->reserved > 12;
        // The fused launch relies on in-order dispatch of CTAs (skim CTAs, the lowest block indices, are resident or done
        // before any decode CTA that waits for them).  verify_crc16 bit 1 (or FRB_DECODE_TWO_LAUNCH=1) takes the assumption
        // away: the skim CTAs run as a launch of their own and the decode launch finds every offset already published.
        static int two_env = -1;
        if (two_env < 0) { const char *e = getenv("FRB_DECODE_TWO_LAUNCH"); two_env = e ? atoi(e) : 0; }
        const bool two_launch = n_skim_ctas > 0 && ((p->verify_crc16 & 2u) || two_env);
        prof_begin(1, s);
#define FRB_DECODE(BIG, SINK, GRID, NSKIM) k_decode_subframes<BIG, SINK><<<GRID, kDecThreads, 0, s>>>(d_bytes, w.streams, p->n_streams, p->channels, p->bps, \
            p->blocksize, (uint32_t)total_frames, w.frame_pos, sub_bitoff, d_audio, w.chassign, d_status, NSKIM, skim_lanes, sink, \
            indexed ? 1u : 0u)
#define FRB_DECODE_ANY(GRID, NSKIM) do { \
        if (sink.dtype < 0) { if (big) FRB_DECODE(true, kSinkAudio, GRID, NSKIM); else FRB_DECODE(false, kSinkAudio, GRID, NSKIM); } \
        else if (!sink.window) { if (big) FRB_DECODE(true, kSinkTile, GRID, NSKIM); else FRB_DECODE(false, kSinkTile, GRID, NSKIM); } \
        else { if (big) FRB_DECODE(true, kSinkWindow, GRID, NSKIM); else FRB_DECODE(false, kSinkWindow, GRID, NSKIM); } } while (0)
        if (two_launch) {
            FRB_DECODE_ANY(n_skim_ctas, n_skim_ctas);          // a grid of skim CTAs only
            FRB_LAUNCH_CHECK("k_decode_subframes(skim)");
            FRB_DECODE_ANY(dec_ctas, 0u);                      // decode CTAs: offsets are all there (0 = bad frame)
        } else {
            FRB_DECODE_ANY(n_skim_ctas + dec_ctas, n_skim_ctas);
        }
#undef FRB_DECODE_ANY
#undef FRB_DECODE
        prof_end(1, s);
        FRB_LAUNCH_CHECK("k_decode_subframes");
    }
    if ((p->verify_crc16 & 1u) && !crc_first) FRB_TRY(launch_crc());
    if (p->verify_crc16 & 1u) FRB_CUDA(cudaStreamWaitEvent(s, ev_join, 0));
    if (p->channels == 2 && sink.dtype < 0) {
        k_stereo_fix<<<(uint32_t)total_frames, 128, 0, s>>>(w.streams, p->n_streams, p->blocksize, (uint32_t)total_frames,
                                                           w.chassign, w.frame_pos, d_audio);
        FRB_LAUNCH_CHECK("k_stereo_fix");
    }
    return FRB_OK;
}
}  // namespace frb

extern "C" int frb_decode_batch(const frb_decode_params *p, const frb_decode_stream *h_streams,
                                const uint8_t *d_bytes, uint64_t total_frames, int32_t *d_audio,
                                void *d_workspace, size_t workspace_bytes, uint32_t *d_status, void *stream) {
    return frb::decode_batch_impl(p, h_streams, d_bytes, total_frames, d_audio, d_workspace, workspace_bytes, d_status, stream,
                                  frb::audio_sink());
}

static int frb_decode_tiles_impl(const frb_decode_params *p, const frb_decode_stream *h_streams,
                                 const uint8_t *d_bytes, uint64_t total_frames,
                                 const frb_tile *d_tiles, const double *d_minmax, double scale,
                                 void *d_raster, int dtype, uint32_t bands, uint32_t H, uint32_t W,
                                 void *d_workspace, size_t workspace_bytes, uint32_t *d_status, void *stream,
                                 const uint32_t *d_frame_bytes, const uint32_t *d_sub_bitoff) {
    using namespace frb;
    if (!p || !d_tiles || !d_minmax || !d_raster || dtype < 0 || dtype > FRB_F64 || !(scale > 0.0)) return FRB_ERR_INVALID_ARG;
    if (bands != p->channels) return FRB_ERR_INVALID_ARG;
    // two-channel streams may carry left/side, side/right or mid/side frames, whose samples only exist after both
    // subframes have been decoded: those go through frb_decode_batch + frb_denormalize_tiles
    if (p->channels == 2) return FRB_ERR_UNSUPPORTED;
    return decode_batch_impl(p, h_streams, d_bytes, total_frames, nullptr, d_workspace, workspace_bytes, d_status, stream,
                             raster_sink(dtype, scale, d_tiles, d_minmax, d_raster, H, W), d_frame_bytes, d_sub_bitoff);
}

extern "C" int frb_decode_tiles(const frb_decode_params *p, const frb_decode_stream *h_streams,
                                const uint8_t *d_bytes, uint64_t total_frames,
                                const frb_tile *d_tiles, const double *d_minmax, double scale,
                                void *d_raster, int dtype, uint32_t bands, uint32_t H, uint32_t W,
                                void *d_workspace, size_t workspace_bytes, uint32_t *d_status, void *stream) {
    return frb_decode_tiles_impl(p, h_streams, d_bytes, total_frames, d_tiles, d_minmax, scale, d_raster, dtype, bands, H, W,
                                 d_workspace, workspace_bytes, d_status, stream, nullptr, nullptr);
}

extern "C" int frb_decode_tiles_indexed(const frb_decode_params *p, const frb_decode_stream *h_streams,
                                        const uint8_t *d_bytes, uint64_t total_frames,
                                        const uint32_t *d_frame_bytes, const uint32_t *d_sub_bitoff,
                                        const frb_tile *d_tiles, const double *d_minmax, double scale,
                                        void *d_raster, int dtype, uint32_t bands, uint32_t H, uint32_t W,
                                        void *d_workspace, size_t workspace_bytes, uint32_t *d_status, void *stream) {
    if (!d_frame_bytes || !d_sub_bitoff) return FRB_ERR_INVALID_ARG;
    return frb_decode_tiles_impl(p, h_streams, d_bytes, total_frames, d_tiles, d_minmax, scale, d_raster, dtype, bands, H, W,
                                 d_workspace, workspace_bytes, d_status, stream, d_frame_bytes, d_sub_bitoff);
}

extern "C" int frb_decode_batch_indexed(const frb_decode_params *p, const frb_decode_stream *h_streams,
                                        const uint8_t *d_bytes, uint64_t total_frames,
                                        const uint32_t *d_frame_bytes, const uint32_t *d_sub_bitoff, int32_t *d_audio,
                                        void *d_workspace, size_t workspace_bytes, uint32_t *d_status, void *stream) {
    if (!d_frame_bytes || !d_sub_bitoff) return FRB_ERR_INVALID_ARG;
    return frb::decode_batch_impl(p, h_streams, d_bytes, total_frames, d_audio, d_workspace, workspace_bytes, d_status, stream,
                                  frb::audio_sink(), d_frame_bytes, d_sub_bitoff);
}

extern "C" int frb_decode_window(const frb_decode_params *p, const frb_window_stream *h_streams,
                                 const uint8_t *d_bytes, uint64_t total_frames,
                                 const uint32_t *d_frame_bytes, const uint32_t *d_sub_bitoff,
                                 const frb_tile *d_tiles, const double *d_minmax, double scale, frb_tile window,
                                 void *d_out, int dtype, void *d_workspace, size_t workspace_bytes, uint32_t *d_status, void *stream) {
    using namespace frb;
    if (!p || !d_out || dtype < -1 || dtype > FRB_F64) return FRB_ERR_INVALID_ARG;
    if (dtype >= 0 && (!d_tiles || !d_minmax || !(scale > 0.0) || window.h == 0 || window.w == 0)) return FRB_ERR_INVALID_ARG;
    if (dtype >= 0 && p->channels == 2) return FRB_ERR_UNSUPPORTED;       // mid/side frames: dtype -1 + frb_denormalize_window
    SinkCfg sink = dtype >= 0 ? raster_sink(dtype, scale, d_tiles, d_minmax, d_out, window.h, window.w) : audio_sink();
    if (dtype >= 0) { sink.window = 1; sink.win_row = window.row_off; sink.win_col = window.col_off; }
    int32_t *d_audio = dtype < 0 ? (int32_t *)d_out : nullptr;
    FRB_TRY(check_decode_args(p, h_streams, d_bytes, total_frames, d_audio, d_workspace, d_status, sink, d_frame_bytes, d_sub_bitoff));
    std::vector<DecStreamDev> hs(p->n_streams);
    uint64_t frames = 0;
    for (uint32_t i = 0; i < p->n_streams; i++) {
        const frb_window_stream &a = h_streams[i];
        if (a.n_frames == 0) return FRB_ERR_INVALID_ARG;
        FRB_TRY(dec_stream(p, a.byte_offset, a.byte_length, a.total_samples, a.audio_base, a.sample_rate, a.frame_base,
                           a.first_frame, a.n_frames, frames, hs[i]));
    }
    if (frames != total_frames) return FRB_ERR_INVALID_ARG;
    return decode_streams_impl(p, hs, d_bytes, total_frames, d_audio, d_workspace, workspace_bytes, d_status, stream, sink,
                               d_frame_bytes, d_sub_bitoff);
}

extern "C" int frb_denormalize_window(const int32_t *d_audio, const frb_window_stream *d_streams, uint32_t n_tiles, uint32_t blocksize,
                                      const frb_tile *d_tiles, const double *d_minmax, double scale, frb_tile window,
                                      void *d_out, int dtype, uint32_t bands, void *stream) {
    using namespace frb;
    if (!d_audio || !d_streams || !d_tiles || !d_minmax || !d_out || dtype < 0 || dtype > FRB_F64 || !bands || !n_tiles ||
        !blocksize || !(scale > 0.0) || window.h == 0 || window.w == 0) return FRB_ERR_INVALID_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    const uint32_t parts = tile_grid_parts(n_tiles, bands * window.h), grid = parts * n_tiles;
    FRB_DISPATCH_DTYPE(dtype, (k_denormalize_window<T><<<grid, kMapThreads, 0, s>>>(d_audio, d_streams, blocksize, d_tiles, d_minmax, scale,
                                                                                   window, (T *)d_out, bands, parts)));
    FRB_LAUNCH_CHECK("k_denormalize_window");
    return FRB_OK;
}

#ifdef FRB_DEC_TIMING
extern "C" int frb_debug_decode_timing(unsigned long long *out16, int reset) {
    using namespace frb;
    if (out16) FRB_CUDA(cudaMemcpyFromSymbol(out16, g_dec_dbg, sizeof(unsigned long long) * 16));
    if (reset) {
        unsigned long long z[16];
        for (int i = 0; i < 16; i++) z[i] = 0;
        z[0] = z[11] = ~0ull;
        FRB_CUDA(cudaMemcpyToSymbol(g_dec_dbg, z, sizeof z));
    }
    return FRB_OK;
}
#endif

extern "C" int frb_probe_stream(const uint8_t *d_bytes, uint64_t byte_offset, uint64_t byte_length,
                                uint32_t channels, uint32_t bps, uint32_t blocksize, uint32_t sample_rate,
                                uint64_t *n_frames, uint64_t *n_samples, void *stream) {
    using namespace frb;
    if (!d_bytes || !n_frames || !n_samples || !byte_length) return FRB_ERR_INVALID_ARG;
    int rc = ensure_tables_impl();
    if (rc) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    DecStreamDev hs;
    hs.byte_offset = byte_offset; hs.byte_length = byte_length; hs.n_samples = 0; hs.audio_base = 0;
    hs.sample_rate = sample_rate; hs.frame_base = 0; hs.n_frames = 0; hs.pad = 0;
    uint8_t *d_tmp = nullptr;
    FRB_CUDA(cudaMalloc(&d_tmp, 512));
    DecStreamDev *d_st = (DecStreamDev *)d_tmp;
    unsigned long long *d_probe = (unsigned long long *)(d_tmp + 256);
    cudaError_t e = cudaMemcpyAsync(d_st, &hs, sizeof hs, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_probe, 0, 16, s);
    if (e != cudaSuccess) { cudaFree(d_tmp); return cuda_fail(e, "probe setup"); }
    uint64_t chunks = byte_length / 16 + 2;
    uint32_t gx = (uint32_t)((chunks + 256 * 4 - 1) / (256 * 4));
    if (gx > (uint32_t)kNumSMs * 16) gx = kNumSMs * 16;
    k_sync_scan<<<gx, 256, 0, s>>>(d_bytes, d_st, channels, bps, blocksize, nullptr, nullptr, d_probe, gx);
    g_launches.fetch_add(1);
    unsigned long long h_probe[2] = {0, 0};
    e = cudaMemcpyAsync(h_probe, d_probe, 16, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    cudaFree(d_tmp);
    if (e != cudaSuccess) return cuda_fail(e, "probe");
    if (h_probe[1] == 0) return FRB_ERR_BAD_STREAM;
    uint64_t last_no = h_probe[0] >> 20, last_bs = h_probe[0] & 0xFFFFF;
    if (h_probe[1] != last_no + 1) return FRB_ERR_BAD_STREAM;
    *n_frames = last_no + 1;
    *n_samples = last_no * blocksize + last_bs;
    return FRB_OK;
}
