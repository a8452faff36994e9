// frb_encode.cuh -- FLAC subframe analysis, Rice coding, bit packing and frame assembly (sm_100a).
//
// Replaces pyflac.StreamEncoder.process/finish (reference converter.py:139-154,
// spatial_encoder.py:291-304), i.e. libFLAC 1.4.3's process_subframe_ pipeline,
// for batches of independent streams.  The decision procedure follows libFLAC's
// preset table (docs/sonos-pyflac.txt:6926-6934): wasted bits, CONSTANT/VERBATIM,
// FIXED order by abs-error sums, windowed autocorrelation -> Levinson-Durbin ->
// order estimate -> quantisation, Rice partition order/parameter by the abs-sum
// estimate.  Bit lengths are exact; a subframe that would exceed VERBATIM falls
// back to VERBATIM.
//
// Kernels
//   k_encode_subframes  one 256-thread CTA per (frame, channel): 16 samples per
//                       thread, samples/residuals in shared memory, warp-shuffle
//                       reductions, CTA prefix scan for bit offsets, per-thread
//                       bit assembly, 128-bit coalesced slot stores
//   k_frame_sizes       header + subframe bits -> bytes per frame
//   k_stream_scan       per-stream exclusive scan of frame sizes (CTA scan)
//   k_emit_frames       one CTA per frame: header + CRC-8, funnel-shift
//                       concatenation of subframe slots, padding, parallel CRC-16
#pragma once
#include "frb_common.cuh"

namespace frb {

constexpr int kEncThreads = 256;
constexpr int kSPT = 16;                 // samples per thread at blocksize 4096
constexpr int kMaxBlock = kEncThreads * kSPT;   // 4096
constexpr int kMaxOrd = 12;              // libFLAC presets never exceed 12
constexpr int kMaxPO = 8;
// Shared sample/residual buffers are indexed through PX(): one pad word after every 16 samples, so a
// thread's 16-sample chunk (stride 17 words) is bank-conflict free across the warp.  The linear
// layout gave 16-way conflicts (5.2e9 conflict cycles, profiles/r01_ncu_enc_v1_raw_subset.csv).
#define PX(i) ((i) + ((uint32_t)(i) >> 4))
constexpr int kBufWords = kMaxBlock + kMaxBlock / 16;

// Where the samples come from: planar audio with int32 elements, or -- 16-bps streams of the tile path -- int16 elements
// (round 1 moved every sample as int32: the mapping kernel wrote 4 bytes per sample and both analysis kernels read them
// again, 3.8 GB + 2 x 3.9 GB per C3 scene where 16-bit samples need half).  Sample indices are the same in both cases.
struct EncSrc {
    const void *audio;
    uint32_t a16;            // elements are int16
};
__device__ __forceinline__ const void *audio_at(const EncSrc &S, int64_t idx) {
    return reinterpret_cast<const uint8_t *>(S.audio) + idx * (S.a16 ? 2 : 4);
}
struct TaskLoc {
    uint32_t n, a16;
    const void *src;
};
__device__ __forceinline__ int32_t sample_at(const TaskLoc &L, uint32_t i) {
    return L.a16 ? (int32_t)__ldg(reinterpret_cast<const int16_t *>(L.src) + i) : __ldg(reinterpret_cast<const int32_t *>(L.src) + i);
}
struct EncStreamDev {
    uint64_t n_samples;
    int64_t audio_base;
    uint64_t out_offset;
    uint32_t sample_rate, frame_base, n_frames, pad;
};

struct LevelCfg { int max_lpc_order, max_po, windows, mid_side, loose; };   // mid_side/loose: exactly-two-channel streams only
__host__ __device__ __forceinline__ LevelCfg level_cfg(uint32_t level) {
    // docs/sonos-pyflac.txt:6926-6934
    switch (level) {
        case 0: return {0, 3, 1, 0, 0};
        case 1: return {0, 3, 1, 1, 1};
        case 2: return {0, 3, 1, 1, 0};
        case 3: return {6, 4, 1, 0, 0};
        case 4: return {8, 4, 1, 1, 1};
        case 5: return {8, 5, 1, 1, 0};
        case 6: return {8, 6, 2, 1, 0};
        case 7: return {12, 6, 2, 1, 0};
        default: return {12, 6, 3, 1, 0};
    }
}
__host__ __device__ __forceinline__ uint32_t qlp_precision_for(uint32_t bps, uint32_t blocksize) {
    if (bps < 16) { uint32_t p = 2 + bps / 2; return p < 5 ? 5 : p; }
    if (bps == 16) return blocksize <= 192 ? 7 : blocksize <= 384 ? 8 : blocksize <= 576 ? 9 : blocksize <= 1152 ? 10 : blocksize <= 2304 ? 11 : blocksize <= 4608 ? 12 : 13;
    return blocksize <= 384 ? 13 : blocksize <= 1152 ? 14 : 15;
}
__host__ __device__ __forceinline__ uint32_t slot_words_for(uint32_t blocksize, uint32_t bps) {
    // VERBATIM upper bound: 8 + 32 (wasted unary) + n*bps bits, rounded up to 16 bytes (+1 word for funnel reads)
    uint32_t bits = 8 + 32 + blocksize * bps;
    uint32_t words = (bits + 31) / 32 + 1;
    return (words + 3) & ~3u;
}

struct Choice {
    int type;            // 0 CONSTANT 1 VERBATIM 2 FIXED 3 LPC
    int order, wasted, precision, shift, method, po;
    uint32_t bits;       // estimated bits (decision metric)
    int32_t coefs[kMaxOrd];
    uint8_t params[1 << kMaxPO];
};

struct EncShared {
    // [resA | x | resB]: the bit buffer aliases x plus the non-best residual buffer
    int32_t buf[3][kBufWords];
    unsigned long long psum[1 << (kMaxPO + 1)];
    uint32_t pbits[1 << (kMaxPO + 1)];
    uint8_t pk[1 << (kMaxPO + 1)];
    unsigned long long red_u64[8][8];
    double red_f64[8][kMaxOrd + 1];
    double autoc[kMaxOrd + 1], autoc_root[kMaxOrd + 1];
    double lp_err[kMaxOrd];
    float lp[kMaxOrd][kMaxOrd];
    uint32_t scan[kEncThreads / 32];
    uint32_t order_bits[kMaxPO + 1];
    Choice best, cand;
    int best_buf;          // 0 -> resA holds best residual, 2 -> resB
    int flag, flag2;
    uint32_t misc[8];
    double ord_bits[kMaxOrd], ord_eb2[kMaxOrd];
};

// ---- block reductions -------------------------------------------------------
__device__ __forceinline__ uint32_t block_or(uint32_t v, EncShared &S) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v |= __shfl_xor_sync(0xFFFFFFFFu, v, o);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) S.scan[warp] = v;
    __syncthreads();
    uint32_t r = 0;
#pragma unroll
    for (int w = 0; w < kEncThreads / 32; w++) r |= S.scan[w];
    return r;
}

template <int N>
__device__ __forceinline__ void block_sum_u64(unsigned long long (&v)[N], EncShared &S) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < N; k++)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(0xFFFFFFFFu, v[k], o);
    __syncthreads();
    if (lane == 0)
#pragma unroll
        for (int k = 0; k < N; k++) S.red_u64[warp][k] = v[k];
    __syncthreads();
#pragma unroll
    for (int k = 0; k < N; k++) {
        unsigned long long s = 0;
#pragma unroll
        for (int w = 0; w < kEncThreads / 32; w++) s += S.red_u64[w][k];
        v[k] = s;
    }
}

// exclusive prefix sum over the CTA; returns this thread's offset, total in *total
__device__ __forceinline__ uint32_t block_exscan(uint32_t v, uint32_t *total, EncShared &S) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, o);
        if (lane >= o) inc += t;
    }
    __syncthreads();
    if (lane == 31) S.scan[warp] = inc;
    __syncthreads();
    uint32_t base = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < kEncThreads / 32; w++) {
        uint32_t s = S.scan[w];
        if (w < warp) base += s;
        tot += s;
    }
    *total = tot;
    return base + inc - v;
}

// ---- thread-local bit writer into a zeroed shared word buffer (MSB first) ----
struct SmemBitWriter {
    uint32_t *buf;
    uint32_t pos;      // absolute bit position
    uint32_t cur;      // pending bits of word pos>>5
    __device__ __forceinline__ void init(uint32_t *b, uint32_t bitpos) { buf = b; pos = bitpos; cur = 0; }
    __device__ __forceinline__ void flush_word(uint32_t idx) { if (cur) atomicOr(&buf[idx], cur); cur = 0; }
    __device__ __forceinline__ void put(uint32_t value, uint32_t nbits) {   // nbits 0..32, value < 2^nbits
        if (nbits == 0) return;
        const uint32_t room = 32 - (pos & 31);
        const uint32_t idx = pos >> 5;
        if (nbits < room) { cur |= value << (room - nbits); }
        else {
            cur |= value >> (nbits - room);
            flush_word(idx);
            const uint32_t rest = nbits - room;
            if (rest) cur = value << (32 - rest);
        }
        pos += nbits;
    }
    __device__ __forceinline__ void zeros(uint32_t q) {
        if (q == 0) return;
        const uint32_t idx = pos >> 5;
        pos += q;
        if ((pos >> 5) != idx) flush_word(idx);
    }
    __device__ __forceinline__ void finish() { flush_word(pos >> 5); }
};

__device__ __forceinline__ uint32_t zigzag(int32_t v) { return ((uint32_t)v << 1) ^ (uint32_t)(v >> 31); }
__device__ __forceinline__ int ilog2_u32(uint32_t v) { return 31 - __clz(v); }
__device__ __forceinline__ int ilog2_u64(unsigned long long v) { return 63 - __clzll(v); }

__device__ __forceinline__ uint32_t rice_bits_estimate(uint32_t k, uint32_t n, unsigned long long sum) {
    unsigned long long v = 4ull + (unsigned long long)(1 + k) * n + (k ? (sum >> (k - 1)) : (sum << 1)) - (n >> 1);
    return v > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t)v;
}

__device__ __forceinline__ uint32_t max_po_for(uint32_t limit, uint32_t n, uint32_t order) {
    uint32_t m = n ? (uint32_t)(__ffs((int)n) - 1) : 0;
    if (m > limit) m = limit;
    if (m > (uint32_t)kMaxPO) m = kMaxPO;
    while (m > 0 && (n >> m) <= order) m--;
    return m;
}

// Compute the residual of predictor (coefs, order, shift) into res[i] (indexed by sample), for this
// thread's samples.  Returns false if any residual does not fit in int32 (or is INT32_MIN).
template <bool WIDE>
__device__ __forceinline__ bool compute_residual(const int32_t *x, int32_t *res, uint32_t n, int order, int shift,
                                                 const int32_t *coefs /*smem, kMaxOrd padded*/) {
    const uint32_t i0 = threadIdx.x * kSPT;
    int32_t xv[kSPT + kMaxOrd];
#pragma unroll
    for (int j = 0; j < kSPT + kMaxOrd; j++) {
        int idx = (int)i0 - kMaxOrd + j;
        xv[j] = (idx >= 0 && (uint32_t)idx < n) ? x[PX(idx)] : 0;
    }
    int32_t cf[kMaxOrd];
#pragma unroll
    for (int j = 0; j < kMaxOrd; j++) cf[j] = coefs[j];
    bool ok = true;
#pragma unroll
    for (int s = 0; s < kSPT; s++) {
        const uint32_t i = i0 + s;
        long long r;
        if (WIDE) {
            long long acc = 0;
#pragma unroll
            for (int j = 0; j < kMaxOrd; j++) acc += (long long)cf[j] * (long long)xv[kMaxOrd + s - 1 - j];
            r = (long long)xv[kMaxOrd + s] - (acc >> shift);
        } else {
            // <= 16-bit samples, precision <= 32 - bps - ilog2(order): every partial sum fits int32 (libFLAC's rule)
            int32_t acc = 0;
#pragma unroll
            for (int j = 0; j < kMaxOrd; j++) acc += cf[j] * xv[kMaxOrd + s - 1 - j];
            r = (long long)(xv[kMaxOrd + s] - (acc >> shift));
        }
        if (i < n) {
            if (i >= (uint32_t)order) {
                if (r > 2147483647ll || r <= -2147483648ll) ok = false;
                res[PX(i)] = (int32_t)r;
            } else res[PX(i)] = 0;
        }
    }
    return ok;
}

// Partition sums + libFLAC estimate search.  On return S.cand.{po,method,params,bits(residual bits)} are set.
__device__ __forceinline__ uint32_t search_partitions(const int32_t *res, uint32_t n, int order, uint32_t max_po_cfg,
                                                      uint32_t k_limit, EncShared &S) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t P = max_po_for(max_po_cfg, n, (uint32_t)order);
    const uint32_t parts = 1u << P, psize = n >> P;
    // level 0 (finest) sums at psum[0..parts)
    for (uint32_t p = warp; p < parts; p += kEncThreads / 32) {
        unsigned long long s = 0;
        const uint32_t a = p * psize, b = a + psize;
        for (uint32_t i = a + lane; i < b; i += 32) {
            if (i >= (uint32_t)order) { int32_t v = res[PX(i)]; s += (unsigned long long)(v < 0 ? -(long long)v : (long long)v); }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, o);
        if (lane == 0) S.psum[p] = s;
    }
    __syncthreads();
    // merge upward: level l holds order P-l at offset off_l
    {
        uint32_t off = 0, cnt = parts;
        for (uint32_t l = 0; l < P; l++) {
            for (uint32_t p = threadIdx.x; p < cnt / 2; p += kEncThreads)
                S.psum[off + cnt + p] = S.psum[off + 2 * p] + S.psum[off + 2 * p + 1];
            off += cnt; cnt >>= 1;
            __syncthreads();
        }
    }
    // per (order, partition) parameter + estimated bits
    const uint32_t total_entries = (parts << 1) - 1;
    for (uint32_t e = threadIdx.x; e < total_entries; e += kEncThreads) {
        // find level: entries [off_l, off_l + parts>>l)
        uint32_t l = 0, off = 0, cnt = parts;
        while (e >= off + cnt) { off += cnt; cnt >>= 1; l++; }
        const uint32_t po = P - l, p = e - off;
        uint32_t np = n >> po;
        if (p == 0) np -= (uint32_t)order;
        const uint32_t div = 0x40000u / np;
        const unsigned long long mean = S.psum[e];
        uint32_t k;
        unsigned long long t = mean < 2 ? 0ull : (((mean - 1) * div) >> 18);
        if (t == 0) k = 0; else k = (uint32_t)ilog2_u64(t) + 1;
        if (k >= k_limit) k = k_limit - 1;
        S.pk[e] = (uint8_t)k;
        S.pbits[e] = rice_bits_estimate(k, np, mean);
    }
    __syncthreads();
    // per-order totals: warp w sums order P-w, P-w-8...
    for (uint32_t l = warp; l <= P; l += kEncThreads / 32) {
        uint32_t off = 0, cnt = parts;
        for (uint32_t q = 0; q < l; q++) { off += cnt; cnt >>= 1; }
        unsigned long long s = 0;
        for (uint32_t p = lane; p < cnt; p += 32) s += S.pbits[off + p];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, o);
        s += 6;
        if (lane == 0) S.order_bits[l] = s > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t)s;
    }
    __syncthreads();
    // choose: iterate partition order from max down to 0, strict improvement only
    uint32_t best_l = 0, best_bits = S.order_bits[0];
    for (uint32_t l = 1; l <= P; l++) { uint32_t b = S.order_bits[l]; if (b < best_bits) { best_bits = b; best_l = l; } }
    {
        uint32_t off = 0, cnt = parts;
        for (uint32_t q = 0; q < best_l; q++) { off += cnt; cnt >>= 1; }
        bool rice2 = false;
        for (uint32_t p = threadIdx.x; p < cnt; p += kEncThreads) { uint8_t k = S.pk[off + p]; S.cand.params[p] = k; if (k >= 15) rice2 = true; }
        int any = __syncthreads_or(rice2 ? 1 : 0);
        if (threadIdx.x == 0) { S.cand.po = (int)(P - best_l); S.cand.method = any ? 1 : 0; }
    }
    __syncthreads();
    return best_bits;
}

// If the candidate in S.cand (with residual in buffer cand_buf) beats S.best, adopt it.
__device__ __forceinline__ void consider_candidate(uint32_t cand_bits, int cand_buf, EncShared &S) {
    __syncthreads();
    const bool better = cand_bits < S.best.bits;
    __syncthreads();
    if (better) {
        if (threadIdx.x == 0) { S.cand.bits = cand_bits; S.best_buf = cand_buf; }
        __syncthreads();
        // struct copy by words
        const uint32_t words = sizeof(Choice) / 4;
        uint32_t *d = (uint32_t *)&S.best; const uint32_t *s = (const uint32_t *)&S.cand;
        for (uint32_t i = threadIdx.x; i < words; i += kEncThreads) d[i] = s[i];
    }
    __syncthreads();
}

__global__ void __launch_bounds__(kEncThreads, 3)
k_encode_subframes(const EncStreamDev *__restrict__ streams, uint32_t n_streams, uint32_t channels, uint32_t bps_stream,
                   uint32_t blocksize, uint32_t level, const EncSrc audio,
                   const float *__restrict__ window, uint32_t slot_words, uint32_t *__restrict__ slots,
                   uint32_t *__restrict__ sub_bits, const uint32_t *__restrict__ task_list, uint32_t side_ch,
                   uint32_t *__restrict__ sub_est) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    EncShared &S = *reinterpret_cast<EncShared *>(smem_raw);
    const uint32_t task = task_list ? task_list[blockIdx.x] : blockIdx.x;
    const uint32_t f = task / channels, c = task - f * channels;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    // locate stream
    uint32_t lo = 0, hi = n_streams - 1;
    while (lo < hi) {
        uint32_t mid = (lo + hi + 1) >> 1;
        if (streams[mid].frame_base <= f) lo = mid; else hi = mid - 1;
    }
    const EncStreamDev st = streams[lo];
    const uint32_t kf = f - st.frame_base;
    const uint32_t n = (kf + 1 < st.n_frames) ? blocksize : (uint32_t)(st.n_samples - (uint64_t)kf * blocksize);
    TaskLoc src;
    src.n = n; src.a16 = audio.a16;
    src.src = audio_at(audio, st.audio_base + (int64_t)c * (int64_t)st.n_samples + (int64_t)kf * blocksize);
    int32_t *X = S.buf[1];
    const LevelCfg cfg = level_cfg(level);
    const uint32_t k_limit = bps_stream > 16 ? 31u : 15u;      // by the STREAM's bps, also for a 17-bit side channel
    const uint32_t sbps = bps_stream + (c == side_ch ? 1u : 0u);
    const uint32_t i0 = tid * kSPT;

    // ---- load, wasted bits, constant check -----------------------------------
    uint32_t orv = 0, diff = 0;
    const int32_t x_first = n ? sample_at(src, 0) : 0;
#pragma unroll
    for (int s = 0; s < kSPT; s++) {
        const uint32_t i = i0 + s;
        if (i < n) { int32_t v = sample_at(src, i); X[PX(i)] = v; orv |= (uint32_t)v; diff |= (uint32_t)(v ^ x_first); }
    }
    orv = block_or(orv, S);
    diff = block_or(diff, S);
    uint32_t wasted = orv ? (uint32_t)(__ffs((int)orv) - 1) : 0;
    if (wasted > sbps) wasted = sbps;
    const uint32_t bps = sbps - wasted;
    if (wasted) {
#pragma unroll
        for (int s = 0; s < kSPT; s++) { const uint32_t i = i0 + s; if (i < n) X[PX(i)] >>= wasted; }
    }
    if (tid == 0) {
        S.best.type = 1; S.best.order = 0; S.best.wasted = (int)wasted; S.best.precision = 0; S.best.shift = 0;
        S.best.method = 0; S.best.po = 0; S.best.bits = 8 + wasted + n * bps;
        S.best_buf = 0;
    }
    __syncthreads();
    const uint32_t verbatim_bits = 8 + wasted + n * bps;

    if (n > 4) {
        if (diff == 0) {
            if (tid == 0) { uint32_t b = 8 + wasted + bps; if (b < S.best.bits) { S.best.type = 0; S.best.bits = b; } }
            __syncthreads();
        } else {
            // ---- fixed predictor abs-error sums over i in [4, n) --------------------
            unsigned long long e[5] = {0, 0, 0, 0, 0};
            {
                int32_t xv[kSPT + 4];
#pragma unroll
                for (int j = 0; j < kSPT + 4; j++) { int idx = (int)i0 - 4 + j; xv[j] = (idx >= 0 && (uint32_t)idx < n) ? X[PX(idx)] : 0; }
                if (sbps <= 16) {
                    // successive differences in 32-bit: |4th difference| <= 16 * 2^15, 16 samples per thread
                    uint32_t e32[5] = {0, 0, 0, 0, 0};
                    int32_t d1[kSPT + 3], d2[kSPT + 2], d3[kSPT + 1], d4[kSPT];
#pragma unroll
                    for (int j = 0; j < kSPT + 3; j++) d1[j] = xv[j + 1] - xv[j];
#pragma unroll
                    for (int j = 0; j < kSPT + 2; j++) d2[j] = d1[j + 1] - d1[j];
#pragma unroll
                    for (int j = 0; j < kSPT + 1; j++) d3[j] = d2[j + 1] - d2[j];
#pragma unroll
                    for (int j = 0; j < kSPT; j++) d4[j] = d3[j + 1] - d3[j];
#pragma unroll
                    for (int s = 0; s < kSPT; s++) {
                        const uint32_t i = i0 + s;
                        if (i >= 4 && i < n) {
                            e32[0] += (uint32_t)abs(xv[s + 4]); e32[1] += (uint32_t)abs(d1[s + 3]); e32[2] += (uint32_t)abs(d2[s + 2]);
                            e32[3] += (uint32_t)abs(d3[s + 1]); e32[4] += (uint32_t)abs(d4[s]);
                        }
                    }
#pragma unroll
                    for (int q = 0; q < 5; q++) e[q] = e32[q];
                } else {
#pragma unroll
                    for (int s = 0; s < kSPT; s++) {
                        const uint32_t i = i0 + s;
                        if (i >= 4 && i < n) {
                            long long a = xv[s + 4], b = xv[s + 3], cc = xv[s + 2], d = xv[s + 1], ee = xv[s];
                            long long r0 = a, r1 = a - b, r2 = a - 2 * b + cc, r3 = a - 3 * b + 3 * cc - d, r4 = a - 4 * b + 6 * cc - 4 * d + ee;
                            e[0] += (unsigned long long)(r0 < 0 ? -r0 : r0);
                            e[1] += (unsigned long long)(r1 < 0 ? -r1 : r1);
                            e[2] += (unsigned long long)(r2 < 0 ? -r2 : r2);
                            e[3] += (unsigned long long)(r3 < 0 ? -r3 : r3);
                            e[4] += (unsigned long long)(r4 < 0 ? -r4 : r4);
                        }
                    }
                }
            }
            block_sum_u64<5>(e, S);
            uint32_t guess;
            {
                unsigned long long m1234 = min(min(e[1], e[2]), min(e[3], e[4]));
                unsigned long long m234 = min(e[2], min(e[3], e[4]));
                unsigned long long m34 = min(e[3], e[4]);
                if (e[0] <= m1234) guess = 0; else if (e[1] <= m234) guess = 1; else if (e[2] <= m34) guess = 2; else if (e[3] <= e[4]) guess = 3; else guess = 4;
            }
            const float fbits_guess = (float)(e[guess] > 0 ? log(0.69314718055994530942 * (double)e[guess] / (double)(n - 4)) / 0.69314718055994530942 : 0.0);
            int cand_buf = 0;      // first candidate residual goes to resA (buf[0]); next to the non-best one
            if (!(fbits_guess >= (float)bps)) {
                if (tid == 0) {
                    Choice &C = S.cand;
                    C.type = 2; C.order = (int)guess; C.wasted = (int)wasted; C.precision = 0; C.shift = 0;
                    for (int j = 0; j < kMaxOrd; j++) C.coefs[j] = 0;
                    if (guess == 1) { C.coefs[0] = 1; }
                    else if (guess == 2) { C.coefs[0] = 2; C.coefs[1] = -1; }
                    else if (guess == 3) { C.coefs[0] = 3; C.coefs[1] = -3; C.coefs[2] = 1; }
                    else if (guess == 4) { C.coefs[0] = 4; C.coefs[1] = -6; C.coefs[2] = 4; C.coefs[3] = -1; }
                }
                __syncthreads();
                int32_t *R = S.buf[cand_buf];
                bool ok = sbps <= 16 ? compute_residual<false>(X, R, n, (int)guess, 0, S.cand.coefs)
                                            : compute_residual<true>(X, R, n, (int)guess, 0, S.cand.coefs);
                int bad = __syncthreads_or(ok ? 0 : 1);
                if (!bad) {
                    uint32_t rb = search_partitions(R, n, (int)guess, (uint32_t)cfg.max_po, k_limit, S);
                    uint32_t total = 8 + wasted + guess * bps + rb;
                    consider_candidate(total, cand_buf, S);
                }
            }
            // ---- LPC ---------------------------------------------------------------
            uint32_t max_lpc = (uint32_t)cfg.max_lpc_order;
            if (max_lpc >= n) max_lpc = n - 1;
            if (max_lpc > 0) {
                const uint32_t qprec_cfg = qlp_precision_for(bps_stream, blocksize);
                const int kinds = cfg.windows;
                for (int b = 1; b <= kinds; b++) {
                    const int ncs = (b == 1) ? 1 : (b == 2 ? 2 : 2 * b);
                    for (int ci = 0; ci < ncs; ci++) {
                        const int cidx = (b == 2) ? 2 * ci : ci;
                        bool have_ac = true;
                        if (b > 1 && n / (uint32_t)b <= 32) have_ac = false;
                        if (have_ac && (b == 1 || !(cidx & 1))) {
                            // windowed autocorrelation over [wshift, wshift + wlen)
                            uint32_t wshift = 0, wlen = n, part = 0;
                            if (b > 1) { part = n / (uint32_t)b / 2; wshift = ((uint32_t)(cidx / 2) * n) / (uint32_t)b; wlen = n / (uint32_t)b; }
                            double dd[kSPT + kMaxOrd];
#pragma unroll
                            for (int j = 0; j < kSPT + kMaxOrd; j++) {
                                int idx = (int)i0 - kMaxOrd + j;
                                double v = 0.0;
                                if (idx >= (int)wshift && (uint32_t)idx < wshift + wlen && (uint32_t)idx < n) {
                                    uint32_t local = (uint32_t)idx - wshift;
                                    float wv;
                                    if (b == 1) wv = __ldg(window + idx);
                                    else if (local < part) wv = __ldg(window + local);
                                    else if (local < 2 * part) wv = __ldg(window + (n - 2 * part + local));
                                    else wv = 0.0f;
                                    v = (double)__fmul_rn((float)X[PX(idx)], wv);
                                }
                                dd[j] = v;
                            }
                            double ac[kMaxOrd + 1];
#pragma unroll
                            for (int l = 0; l <= kMaxOrd; l++) ac[l] = 0.0;
#pragma unroll
                            for (int s = 0; s < kSPT; s++)
#pragma unroll
                                for (int l = 0; l <= kMaxOrd; l++) ac[l] = fma(dd[kMaxOrd + s], dd[kMaxOrd + s - l], ac[l]);
#pragma unroll
                            for (int l = 0; l <= kMaxOrd; l++)
#pragma unroll
                                for (int o = 16; o > 0; o >>= 1) ac[l] += __shfl_xor_sync(0xFFFFFFFFu, ac[l], o);
                            __syncthreads();
                            if (lane == 0)
#pragma unroll
                                for (int l = 0; l <= kMaxOrd; l++) S.red_f64[warp][l] = ac[l];
                            __syncthreads();
                            if (tid <= kMaxOrd) {
                                double s = 0.0;
                                for (int w = 0; w < kEncThreads / 32; w++) s += S.red_f64[w][tid];
                                S.autoc[tid] = s;
                                if (b == 1) S.autoc_root[tid] = s;
                            }
                            __syncthreads();
                        } else if (have_ac) {
                            // punch-out window: root minus the previous partial window (lags < max_lpc as libFLAC does)
                            if ((uint32_t)tid < max_lpc) S.autoc[tid] = S.autoc_root[tid] - S.autoc[tid];
                            __syncthreads();
                        }
                        // ---- Levinson-Durbin (lane 0), expected bits per order (one lane per order, the
                        // logarithms dominated the serial section), order pick + quantisation (lane 0) ----
                        if (warp == 0) {
                            if (lane == 0) {
                                S.flag = 0; S.misc[0] = 0;
                                if (have_ac && S.autoc[0] != 0.0) {
                                    double lpc[kMaxOrd];
                                    double err = S.autoc[0];
                                    uint32_t mo = max_lpc;
                                    for (uint32_t i = 0; i < max_lpc; i++) {
                                        double r = -S.autoc[i + 1];
                                        for (uint32_t j = 0; j < i; j++) r = __dsub_rn(r, __dmul_rn(lpc[j], S.autoc[i - j]));
                                        r = __ddiv_rn(r, err);
                                        lpc[i] = r;
                                        uint32_t j;
                                        for (j = 0; j < (i >> 1); j++) {
                                            double tmp = lpc[j];
                                            lpc[j] = __dadd_rn(lpc[j], __dmul_rn(r, lpc[i - 1 - j]));
                                            lpc[i - 1 - j] = __dadd_rn(lpc[i - 1 - j], __dmul_rn(r, tmp));
                                        }
                                        if (i & 1) lpc[j] = __dadd_rn(lpc[j], __dmul_rn(lpc[j], r));
                                        err = __dmul_rn(err, __dsub_rn(1.0, __dmul_rn(r, r)));
                                        for (j = 0; j <= i; j++) S.lp[i][j] = (float)(-lpc[j]);
                                        S.lp_err[i] = err;
                                        if (err == 0.0) { mo = i + 1; break; }
                                    }
                                    S.misc[0] = mo;
                                }
                            }
                            __syncwarp();
                            const uint32_t mo = S.misc[0];
                            if ((uint32_t)lane < mo) {
                                // FLAC__lpc_compute_best_order term and the "don't even try" estimate for this order
                                const double le = S.lp_err[lane];
                                const uint32_t ord = (uint32_t)lane + 1;
                                const double scale = 0.5 / (double)n, scale2 = 0.5 / (double)(n - ord);
                                double eb, eb2;
                                if (le > 0.0) {
                                    eb = 0.5 * log(scale * le) / 0.69314718055994530942; if (eb < 0.0) eb = 0.0;
                                    eb2 = 0.5 * log(scale2 * le) / 0.69314718055994530942; if (eb2 < 0.0) eb2 = 0.0;
                                } else if (le < 0.0) { eb = 1e32; eb2 = 1e32; } else { eb = 0.0; eb2 = 0.0; }
                                S.ord_bits[lane] = eb * (double)(n - ord) + (double)(ord * (bps + qprec_cfg));
                                S.ord_eb2[lane] = eb2;
                            }
                            __syncwarp();
                            if (lane == 0 && mo > 0) {
                                uint32_t best_i = 0; double best_b = 4294967295.0;
                                for (uint32_t i = 0; i < mo; i++) { const double bits = S.ord_bits[i]; if (bits < best_b) { best_b = bits; best_i = i; } }
                                const uint32_t order = best_i + 1;
                                const double eb = S.ord_eb2[order - 1];
                                if (!(eb >= (double)bps)) {
                                    uint32_t prec = qprec_cfg;
                                    if (bps <= 17) { uint32_t lim = 32 - bps - (uint32_t)ilog2_u32(order); if (lim < prec) prec = lim; }
                                    // FLAC__lpc_quantize_coefficients
                                    const float *lpv = S.lp[order - 1];
                                    int p1 = (int)prec - 1;
                                    int qmax = (1 << p1) - 1, qmin = -(1 << p1);
                                    double cmax = 0.0;
                                    for (uint32_t i = 0; i < order; i++) { double d = fabs((double)lpv[i]); if (d > cmax) cmax = d; }
                                    if (cmax > 0.0) {
                                        int log2cmax; (void)frexp(cmax, &log2cmax); log2cmax--;
                                        int sh = p1 - log2cmax - 1;
                                        bool okq = true;
                                        if (sh > 15) sh = 15; else if (sh < -16) okq = false;
                                        if (okq) {
                                            Choice &C = S.cand;
                                            for (int j = 0; j < kMaxOrd; j++) C.coefs[j] = 0;
                                            double er = 0.0;
                                            if (sh >= 0) {
                                                for (uint32_t i = 0; i < order; i++) {
                                                    er = __dadd_rn(er, __dmul_rn((double)lpv[i], (double)(1 << sh)));
                                                    long long q = llround(er);
                                                    if (q > qmax) q = qmax; else if (q < qmin) q = qmin;
                                                    er = __dsub_rn(er, (double)q); C.coefs[i] = (int32_t)q;
                                                }
                                            } else {
                                                const int ns = -sh;
                                                for (uint32_t i = 0; i < order; i++) {
                                                    er = __dadd_rn(er, __ddiv_rn((double)lpv[i], (double)(1 << ns)));
                                                    long long q = llround(er);
                                                    if (q > qmax) q = qmax; else if (q < qmin) q = qmin;
                                                    er = __dsub_rn(er, (double)q); C.coefs[i] = (int32_t)q;
                                                }
                                                sh = 0;
                                            }
                                            C.type = 3; C.order = (int)order; C.wasted = (int)wasted; C.precision = (int)prec; C.shift = sh;
                                            S.flag = 1;
                                        }
                                    }
                                }
                            }
                        }
                        __syncthreads();
                        if (S.flag) {
                            cand_buf = (S.best_buf == 0 && (S.best.type >= 2)) ? 2 : 0;
                            const int order = S.cand.order, sh = S.cand.shift;
                            int32_t *R = S.buf[cand_buf];
                            bool ok = sbps <= 16 ? compute_residual<false>(X, R, n, order, sh, S.cand.coefs)
                                                        : compute_residual<true>(X, R, n, order, sh, S.cand.coefs);
                            int bad = __syncthreads_or(ok ? 0 : 1);
                            if (!bad) {
                                uint32_t rb = search_partitions(R, n, order, (uint32_t)cfg.max_po, k_limit, S);
                                uint32_t total = 8 + wasted + 4 + 5 + (uint32_t)order * ((uint32_t)S.cand.precision + bps) + rb;
                                consider_candidate(total, cand_buf, S);
                            }
                        }
                        __syncthreads();
                    }
                }
            }
        }
    }
    __syncthreads();

    // ---- exact bit lengths, fallback to VERBATIM, pack ----------------------------
    int type = S.best.type;
    const int order = S.best.order, po = S.best.po, method = S.best.method;
    const int32_t *R = S.buf[S.best_buf];
    const uint32_t plen = method ? 5u : 4u;
    const uint32_t psize = n >> po;
    uint32_t my_bits = 0;
    // folded residuals and their Rice parameters stay in registers between the length pass and the pack pass;
    // the partition index is tracked incrementally (one division per thread instead of two per sample)
    uint32_t u_reg[kSPT], k_reg[kSPT];
    uint32_t pstart_mask = 0;                    // bit s: sample i0+s is the first residual of its partition
    if (type >= 2 && i0 < n) {
        uint32_t p = i0 / psize;
        uint32_t next_b = (p + 1) * psize;
        uint32_t kcur = S.best.params[p];
#pragma unroll
        for (int s = 0; s < kSPT; s++) {
            const uint32_t i = i0 + s;
            u_reg[s] = 0; k_reg[s] = 0;
            if (i < n) {
                if (i == next_b) { p++; next_b += psize; kcur = S.best.params[p]; }
                if (i >= (uint32_t)order) {
                    const uint32_t u = zigzag(R[PX(i)]);
                    u_reg[s] = u; k_reg[s] = kcur;
                    my_bits += (u >> kcur) + 1 + kcur;
                    if (i + psize == next_b || i == (uint32_t)order) { my_bits += plen; pstart_mask |= 1u << s; }
                }
            }
        }
    }
    uint32_t hdr_bits = 8 + wasted;
    if (type == 0) hdr_bits += bps;
    else if (type == 2) hdr_bits += (uint32_t)order * bps + 6;
    else if (type == 3) hdr_bits += (uint32_t)order * bps + 9 + (uint32_t)(order * S.best.precision) + 6;
    uint32_t total_res = 0;
    uint32_t my_off = block_exscan(my_bits, &total_res, S);
    __syncthreads();
    if (type >= 2 && hdr_bits + total_res > verbatim_bits) type = 1;     // exactness guard
    uint32_t total_bits;
    if (type == 1) { hdr_bits = 8 + wasted; total_bits = verbatim_bits; }
    else total_bits = hdr_bits + total_res;

    // bit buffer: X + the non-best residual buffer (contiguous 32 KB); warm-up samples saved first
    int32_t warm[kMaxOrd];
    int32_t xfirst_shifted = 0;
    if (tid == 0) {
#pragma unroll
        for (int j = 0; j < kMaxOrd; j++) warm[j] = (j < order && (uint32_t)j < n) ? X[PX(j)] : 0;
        xfirst_shifted = n ? X[0] : 0;
    }
    uint32_t *bitbuf;
    int32_t xv_verb[kSPT];
    if (type == 1) {
#pragma unroll
        for (int s = 0; s < kSPT; s++) { const uint32_t i = i0 + s; xv_verb[s] = (i < n) ? X[PX(i)] : 0; }
        bitbuf = (uint32_t *)S.buf[1];              // X + resB: nothing else is needed any more
    } else {
        bitbuf = (S.best_buf == 0) ? (uint32_t *)S.buf[1] : (uint32_t *)S.buf[0];
    }
    __syncthreads();
    const uint32_t nwords = (total_bits + 31) / 32;
    for (uint32_t wd = tid; wd < nwords + 1 && wd < 2 * kBufWords; wd += kEncThreads) bitbuf[wd] = 0;
    __syncthreads();

    const uint32_t mask_bps = bps >= 32 ? 0xFFFFFFFFu : ((1u << bps) - 1u);
    SmemBitWriter bw;
    if (tid == 0) {
        bw.init(bitbuf, 0);
        uint32_t typecode = type == 0 ? 0u : type == 1 ? 1u : type == 2 ? (8u | (uint32_t)order) : (32u | (uint32_t)(order - 1));
        bw.put((typecode << 1) | (wasted ? 1u : 0u), 8);
        if (wasted) { bw.zeros(wasted - 1); bw.put(1, 1); }
        // (bps == 33: the side subframe of a two-channel 32-bps stream; its int32 samples are sign-extended by one bit)
        auto put_sample = [&](int32_t x) { if (bps > 32) { bw.put(x < 0 ? 1u : 0u, bps - 32); bw.put((uint32_t)x, 32); } else bw.put((uint32_t)x & mask_bps, bps); };
        if (type == 0) put_sample((int32_t)xfirst_shifted);
        else if (type >= 2) {
#pragma unroll
            for (int j = 0; j < kMaxOrd; j++) if (j < order) put_sample((int32_t)warm[j]);
            if (type == 3) {
                const uint32_t prec = (uint32_t)S.best.precision;
                bw.put(prec - 1, 4);
                bw.put((uint32_t)S.best.shift & 31u, 5);
#pragma unroll
                for (int j = 0; j < kMaxOrd; j++) if (j < order) bw.put((uint32_t)S.best.coefs[j] & ((1u << prec) - 1u), prec);
            }
            bw.put((uint32_t)method, 2);
            bw.put((uint32_t)po, 4);
        }
        bw.finish();
    }
    if (type == 1) {
        bw.init(bitbuf, hdr_bits + i0 * bps);
#pragma unroll
        for (int s = 0; s < kSPT; s++) {
            const uint32_t i = i0 + s;
            if (i < n) { if (bps > 32) { bw.put(xv_verb[s] < 0 ? 1u : 0u, bps - 32); bw.put((uint32_t)xv_verb[s], 32); } else bw.put((uint32_t)xv_verb[s] & mask_bps, bps); }
        }
        bw.finish();
    } else if (type >= 2) {
        bw.init(bitbuf, hdr_bits + my_off);
#pragma unroll
        for (int s = 0; s < kSPT; s++) {
            const uint32_t i = i0 + s;
            if (i < n && i >= (uint32_t)order) {
                const uint32_t k = k_reg[s], u = u_reg[s];
                if (pstart_mask & (1u << s)) bw.put(k, plen);
                const uint32_t q = u >> k;
                const uint32_t tailv = (1u << k) | (u & ((1u << k) - 1u));
                if (q + k + 1 <= 32) bw.put(tailv, q + k + 1);       // zeros, stop bit and LSBs in one write
                else { bw.zeros(q); bw.put(tailv, k + 1); }
            }
        }
        bw.finish();
    }
    __syncthreads();
    // ---- slot store (128-bit, coalesced) -------------------------------------------
    uint32_t *slot = slots + (size_t)task * slot_words;
    const uint32_t nq = (nwords + 1 + 3) / 4;          // one extra word so the emitter can funnel-read past the end
    const uint4 *b4 = reinterpret_cast<const uint4 *>(bitbuf);
    uint4 *s4 = reinterpret_cast<uint4 *>(slot);
    for (uint32_t q = tid; q < nq && q * 4 < slot_words; q += kEncThreads) s4[q] = b4[q];
    if (tid == 0) { sub_bits[task] = total_bits; if (sub_est) sub_est[task] = S.best.bits; }
}

#include "frb_encode_fast.cuh"

// ---- frame sizes / scans -------------------------------------------------------
__device__ __forceinline__ uint32_t frame_header_bytes(uint32_t n, uint32_t sample_rate, uint64_t number) {
    int bh, sh;
    (void)blocksize_code(n, &bh);
    (void)samplerate_code(sample_rate, &sh);
    return 4 + (uint32_t)utf8_len(number) + (uint32_t)bh + (sh == 0 ? 0u : sh == 1 ? 1u : 2u) + 1;
}

// ---- two-channel streams: libFLAC's stereo decorrelation --------------------------------------------------------
// The four candidate subframes of a frame -- left, right, mid = (L+R)>>1, side = L-R (one more bit per sample) -- are
// encoded as four VIRTUAL channels (k_ms_expand builds their planar audio, every analysis kernel runs unchanged on
// them); k_ms_choose then picks the channel assignment per frame from libFLAC's ESTIMATED subframe bits, exactly as
// process_subframes_ does: independent, left/side, right/side, mid/side in that order, strict improvement only; the
// "loose" presets (levels 1 and 4) decide once every loose_frames frames and keep independent or switch to
// mid/side in between.  frame_sel[f]: 0 independent, 1 left/side, 2 right/side, 3 mid/side; the frame is assembled
// from two of the four slots.
__host__ __device__ __forceinline__ uint32_t ms_slot(uint32_t sel, uint32_t c) {
    // virtual channels: 0 L, 1 R, 2 M, 3 S
    return sel == 0 ? c : sel == 1 ? (c == 0 ? 0u : 3u) : sel == 2 ? (c == 0 ? 3u : 1u) : (c == 0 ? 2u : 3u);
}
__host__ __device__ __forceinline__ uint32_t ms_channel_code(uint32_t sel) { return sel == 0 ? 1u : 7u + sel; }   // 1, 8, 9, 10

__global__ void __launch_bounds__(256)
k_ms_expand(const EncStreamDev *__restrict__ streams, const EncStreamDev *__restrict__ vstreams,
            const EncSrc audio, int32_t *__restrict__ vaudio, uint32_t parts, uint32_t *__restrict__ err_flag) {
    // flattened grid, `parts` CTAs per stream (gridDim.y stops at 65535 streams)
    const uint32_t si = blockIdx.x / parts, part = blockIdx.x - si * parts;
    const EncStreamDev st = streams[si], vs = vstreams[si];
    TaskLoc l, r;
    l.n = r.n = 0; l.a16 = r.a16 = audio.a16;
    l.src = audio_at(audio, st.audio_base); r.src = audio_at(audio, st.audio_base + (int64_t)st.n_samples);
    int32_t *o = vaudio + vs.audio_base;
    const uint64_t n = st.n_samples;
    bool bad = false;
    for (uint64_t i = (uint64_t)part * blockDim.x + threadIdx.x; i < n; i += (uint64_t)parts * blockDim.x) {
        const int32_t a = sample_at(l, (uint32_t)i), b = sample_at(r, (uint32_t)i);
        o[i] = a; o[n + i] = b; o[2 * n + i] = (int32_t)(((long long)a + b) >> 1); o[3 * n + i] = a - b;
        bad |= ((long long)a - b) != (long long)(a - b);
    }
    if (bad) atomicOr(err_flag + 1, 1u);      // a side sample does not fit int32: the caller's range promise was wrong
}

__global__ void __launch_bounds__(256)
k_ms_choose(const EncStreamDev *__restrict__ streams, uint32_t n_streams, uint32_t blocksize, uint32_t total_frames, uint32_t loose,
            const uint32_t *__restrict__ sub_est, uint8_t *__restrict__ frame_sel) {
    const uint32_t f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= total_frames) return;
    uint32_t lo = 0, hi = n_streams - 1;
    while (lo < hi) {
        uint32_t mid = (lo + hi + 1) >> 1;
        if (streams[mid].frame_base <= f) lo = mid; else hi = mid - 1;
    }
    const EncStreamDev st = streams[lo];
    const uint32_t k = f - st.frame_base;
    auto decide = [&](uint32_t fr) -> uint32_t {
        const uint32_t *e = sub_est + (size_t)fr * 4;
        const unsigned long long b[4] = {(unsigned long long)e[0] + e[1], (unsigned long long)e[0] + e[3],
                                         (unsigned long long)e[1] + e[3], (unsigned long long)e[2] + e[3]};
        uint32_t best = 0;
        for (uint32_t a = 1; a < 4; a++) if (b[a] < b[best]) best = a;
        return best;
    };
    uint32_t sel;
    if (!loose) sel = decide(f);
    else {
        // FLAC__stream_encoder: loose_mid_side_stereo_frames = (uint32_t)(sample_rate * 0.4 / blocksize + 0.5), at least 1
        uint32_t lf = (uint32_t)((double)st.sample_rate * 0.4 / (double)blocksize + 0.5);
        if (lf == 0) lf = 1;
        const uint32_t r = k % lf;
        if (r == 0) sel = decide(f);
        else sel = decide(f - r) == 0 ? 0u : 3u;
    }
    frame_sel[f] = (uint8_t)sel;
}

__global__ void __launch_bounds__(256)
k_frame_sizes(const EncStreamDev *__restrict__ streams, uint32_t n_streams, uint32_t channels, uint32_t blocksize,
              uint32_t total_frames, const uint32_t *__restrict__ sub_bits, uint32_t *__restrict__ frame_bytes,
              uint32_t vch, const uint8_t *__restrict__ frame_sel) {
    const uint32_t f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= total_frames) return;
    uint32_t lo = 0, hi = n_streams - 1;
    while (lo < hi) {
        uint32_t mid = (lo + hi + 1) >> 1;
        if (streams[mid].frame_base <= f) lo = mid; else hi = mid - 1;
    }
    const EncStreamDev st = streams[lo];
    const uint32_t k = f - st.frame_base;
    const uint32_t n = (k + 1 < st.n_frames) ? blocksize : (uint32_t)(st.n_samples - (uint64_t)k * blocksize);
    uint64_t bits = 0;
    for (uint32_t c = 0; c < channels; c++) bits += sub_bits[(size_t)f * vch + (frame_sel ? ms_slot(frame_sel[f], c) : c)];
    frame_bytes[f] = frame_header_bytes(n, st.sample_rate, k) + (uint32_t)((bits + 7) >> 3) + 2;
}

// Seek index of the coded streams (frb_encode_index): for every frame the bit offset of each of its subframes from the
// frame's first byte (entry 0 = the frame header's length).  Thread per frame; same sums as k_frame_sizes.
__global__ void __launch_bounds__(256)
k_export_index(const EncStreamDev *__restrict__ streams, uint32_t n_streams, uint32_t channels, uint32_t blocksize,
               uint32_t total_frames, const uint32_t *__restrict__ sub_bits, uint32_t vch, const uint8_t *__restrict__ frame_sel,
               uint32_t *__restrict__ sub_bitoff) {
    const uint32_t f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= total_frames) return;
    uint32_t lo = 0, hi = n_streams - 1;
    while (lo < hi) {
        uint32_t mid = (lo + hi + 1) >> 1;
        if (streams[mid].frame_base <= f) lo = mid; else hi = mid - 1;
    }
    const EncStreamDev st = streams[lo];
    const uint32_t k = f - st.frame_base;
    const uint32_t n = (k + 1 < st.n_frames) ? blocksize : (uint32_t)(st.n_samples - (uint64_t)k * blocksize);
    uint32_t bits = 8u * frame_header_bytes(n, st.sample_rate, k);
    for (uint32_t c = 0; c < channels; c++) {
        sub_bitoff[(size_t)f * channels + c] = bits;
        bits += sub_bits[(size_t)f * vch + (frame_sel ? ms_slot(frame_sel[f], c) : c)];
    }
}

// one CTA per stream: exclusive scan of its frame sizes -> frame_off, total -> stream_bytes
__global__ void __launch_bounds__(1024)
k_stream_scan(const EncStreamDev *__restrict__ streams, const uint32_t *__restrict__ frame_bytes,
              unsigned long long *__restrict__ frame_off, unsigned long long *__restrict__ stream_bytes) {
    __shared__ unsigned long long s_warp[32];
    __shared__ unsigned long long s_carry;
    const EncStreamDev st = streams[blockIdx.x];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < st.n_frames; base += blockDim.x) {
        const uint32_t i = base + threadIdx.x;
        unsigned long long v = i < st.n_frames ? frame_bytes[st.frame_base + i] : 0ull;
        unsigned long long inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { unsigned long long t = __shfl_up_sync(0xFFFFFFFFu, inc, o); if (lane >= o) inc += t; }
        if (lane == 31) s_warp[warp] = inc;
        __syncthreads();
        unsigned long long wbase = 0, tot = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); w++) { unsigned long long s = s_warp[w]; if (w < warp) wbase += s; tot += s; }
        const unsigned long long carry = s_carry;
        if (i < st.n_frames) frame_off[st.frame_base + i] = carry + wbase + inc - v;
        __syncthreads();
        if (threadIdx.x == 0) s_carry = carry + tot;
        __syncthreads();
    }
    if (threadIdx.x == 0) stream_bytes[blockIdx.x] = s_carry;
}

// out_offset of every stream = exclusive scan of the stream sizes (streams packed back to back in stream order): what the
// caller of frb_encode_emit would compute on the host from the downloaded sizes -- done here so that the step has no
// host round trip between analysis and frame assembly.  One CTA walks the streams in chunks of its size.
__global__ void __launch_bounds__(1024)
k_pack_out_offsets(EncStreamDev *__restrict__ streams, const unsigned long long *__restrict__ stream_bytes, uint32_t n) {
    __shared__ unsigned long long s_warp[32];
    __shared__ unsigned long long s_carry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < n; base += blockDim.x) {
        const uint32_t i = base + threadIdx.x;
        const unsigned long long v = i < n ? stream_bytes[i] : 0ull;
        unsigned long long inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const unsigned long long t = __shfl_up_sync(0xFFFFFFFFu, inc, o); if (lane >= o) inc += t; }
        if (lane == 31) s_warp[warp] = inc;
        __syncthreads();
        unsigned long long wbase = 0, tot = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); w++) { const unsigned long long x = s_warp[w]; if (w < warp) wbase += x; tot += x; }
        const unsigned long long carry = s_carry;
        if (i < n) streams[i].out_offset = carry + wbase + inc - v;
        __syncthreads();
        if (threadIdx.x == 0) s_carry = carry + tot;
        __syncthreads();
    }
}

__global__ void k_set_out_offsets(EncStreamDev *streams, const unsigned long long *offs, uint32_t n) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) streams[i].out_offset = offs[i];
}

// ---- frame assembly ------------------------------------------------------------------------------
// One warp per frame (a 128-thread CTA per frame on request).  The frame's bytes are produced in 16-byte chunks aligned to the
// GLOBAL address (coalesced 128-bit stores; the first/last chunk of a frame is partial and produced by the whole warp, a byte
// per lane), each chunk gathered from the header words / subframe slots with funnel shifts.  CRC-16: a lane folds its chunks
// (rows of 30, or 120 for the CTA form) without tables (CrcFold, frb_crc16.cuh), then weights x^(128*(ROW-1-t)) and small tail
// powers, XOR-reduced over the group.
// v1 stored single bytes and ran a byte-serial CRC per thread: 13.8 ms on C3 (profiles/r01_launches_c3_v1.csv).
constexpr int kEmitThreads = 128;
#ifndef FRB_EMIT_VLOAD
#define FRB_EMIT_VLOAD 1
#endif
// rows ahead whose slot words a thread asks for while it works on the current chunk (0 = off); see do_chunk
#ifndef FRB_EMIT_PF_L1
#define FRB_EMIT_PF_L1 1
#endif
#ifndef FRB_EMIT_PF_L2
#define FRB_EMIT_PF_L2 0
#endif

struct EmitGroup {                           // state of the frame a thread group (a CTA or a warp) is assembling
    uint32_t hdr[6];
    uint32_t seg_start[FRB_MAX_CHANNELS + 2];
    uint32_t slot_of[FRB_MAX_CHANNELS];      // slot (virtual channel) that holds subframe c of this frame
};
struct EmitShared {
    CrcTables T;
    EmitGroup g[kEmitThreads / 32];
    uint32_t red[kEmitThreads / 32];
};

// 32 bits of the frame bitstream starting at bit position P (P + 32 may run past the end: zero padded)
__device__ __forceinline__ uint32_t emit_gather32(uint32_t P, const EmitGroup &S, uint32_t channels, uint32_t hdr_bits,
                                                  uint32_t end_bits, const uint32_t *__restrict__ slots_f, uint32_t slot_words) {
    uint32_t need = 32, val = 0;
    while (need) {
        uint32_t take, bits;
        if (P < hdr_bits) {
            take = min(need, hdr_bits - P);
            const uint32_t wi = P >> 5, sh = P & 31;
            const uint32_t v = __funnelshift_l(S.hdr[wi + 1], S.hdr[wi], sh);
            bits = take == 32 ? v : (v >> (32 - take));
        } else if (P < end_bits) {
            uint32_t c = 0;
            while (S.seg_start[c + 1] <= P) c++;
            const uint32_t o = P - S.seg_start[c];
            take = min(need, S.seg_start[c + 1] - P);
            const uint32_t *sl = slots_f + (size_t)S.slot_of[c] * slot_words;
            const uint32_t wi = o >> 5, sh = o & 31;
            const uint32_t v = __funnelshift_l(__ldg(sl + wi + 1), __ldg(sl + wi), sh);
            bits = take == 32 ? v : (v >> (32 - take));
        } else { take = need; bits = 0; }
        val = take == 32 ? bits : ((val << take) | bits);
        need -= take; P += take;
    }
    return val;
}

// TPF = threads per frame: 128 (the whole CTA; large multi-channel frames) or 32 (a warp per frame, no CTA barriers:
// small frames, where the per-frame barriers and the serial header dominated -- C5's 6 KB frames took 2.16 ms).
template <int TPF>
__global__ void __launch_bounds__(kEmitThreads)
k_emit_frames(const EncStreamDev *__restrict__ streams, uint32_t n_streams, uint32_t channels, uint32_t bps_stream,
              uint32_t blocksize, uint32_t total_frames, const uint32_t *__restrict__ sub_bits,
              const uint32_t *__restrict__ slots, uint32_t slot_words, const uint32_t *__restrict__ frame_bytes,
              const unsigned long long *__restrict__ frame_off, uint8_t *__restrict__ out, uint64_t out_capacity,
              uint32_t *__restrict__ err_flag, uint32_t vch, const uint8_t *__restrict__ frame_sel,
              const FrameDesc *__restrict__ frame_table) {
    __shared__ __align__(16) EmitShared SS;
    constexpr int kGroups = kEmitThreads / TPF;
    const int tid = threadIdx.x % TPF, grp = threadIdx.x / TPF;
    EmitGroup &S = SS.g[grp];
    auto group_sync = [&]() { if (TPF == kEmitThreads) __syncthreads(); else __syncwarp(); };
    crc_tables_to_smem(&SS.T);
    __syncthreads();                                      // tables staged
    // persistent CTAs: the CRC tables (6 KB: slice-by-4 for ragged rows and tails, powers of x) are staged once, then every group walks frames with stride gridDim.x * kGroups
    for (uint32_t f = blockIdx.x * kGroups + grp; f < total_frames; f += gridDim.x * kGroups) {
    group_sync();                                         // previous frame's shared state consumed
    // the frame's stream from the descriptor table of the analysis (one load instead of a binary search of log2(n_streams)
    // dependent loads per frame: with 4096 streams of 64 small frames, C5, that search was a fifth of a frame's time)
    const uint32_t lo = frame_table[f].stream;
    const EncStreamDev st = streams[lo];
    const uint32_t k = f - st.frame_base;
    const uint32_t n = (k + 1 < st.n_frames) ? blocksize : (uint32_t)(st.n_samples - (uint64_t)k * blocksize);
    const uint32_t total = frame_bytes[f];
    const uint64_t dst_off = st.out_offset + frame_off[f];
    if (tid == 0) {
        uint8_t hb[16];
        int bh, sh;
        const uint32_t bsc = blocksize_code(n, &bh), src = samplerate_code(st.sample_rate, &sh);
        uint32_t i = 0;
        hb[i++] = 0xFF; hb[i++] = 0xF8;
        hb[i++] = (uint8_t)((bsc << 4) | src);
        const uint32_t sel = frame_sel ? frame_sel[f] : 0u;
        hb[i++] = (uint8_t)(((frame_sel ? ms_channel_code(sel) : channels - 1) << 4) | (bps_code(bps_stream) << 1));
        {
            uint64_t v = k; int len = utf8_len(v);
            if (len == 1) hb[i++] = (uint8_t)v;
            else {
                const uint8_t lead[8] = {0, 0, 0xC0, 0xE0, 0xF0, 0xF8, 0xFC, 0xFE};
                for (int q = len - 1; q > 0; q--) { hb[i + q] = (uint8_t)(0x80 | (v & 0x3F)); v >>= 6; }
                hb[i] = (uint8_t)(lead[len] | v);
                i += len;
            }
        }
        if (bh == 1) hb[i++] = (uint8_t)(n - 1);
        else if (bh == 2) { hb[i++] = (uint8_t)((n - 1) >> 8); hb[i++] = (uint8_t)(n - 1); }
        if (sh == 1) hb[i++] = (uint8_t)(st.sample_rate / 1000);
        else if (sh == 2) { hb[i++] = (uint8_t)(st.sample_rate >> 8); hb[i++] = (uint8_t)st.sample_rate; }
        else if (sh == 3) { hb[i++] = (uint8_t)((st.sample_rate / 10) >> 8); hb[i++] = (uint8_t)(st.sample_rate / 10); }
        uint8_t crc = 0;
        for (uint32_t q = 0; q < i; q++) crc = c_crc8[crc ^ hb[q]];
        hb[i++] = crc;
        for (uint32_t q = i; q < 16; q++) hb[q] = 0;
        for (int w = 0; w < 4; w++) S.hdr[w] = ((uint32_t)hb[4 * w] << 24) | ((uint32_t)hb[4 * w + 1] << 16) | ((uint32_t)hb[4 * w + 2] << 8) | hb[4 * w + 3];
        S.hdr[4] = 0; S.hdr[5] = 0;
        uint32_t pos = i * 8;
        S.seg_start[0] = pos;
        for (uint32_t c = 0; c < channels; c++) {
            const uint32_t sl = frame_sel ? ms_slot(sel, c) : c;
            S.slot_of[c] = sl;
            pos += sub_bits[(size_t)f * vch + sl]; S.seg_start[c + 1] = pos;
        }
        if (((pos + 7) >> 3) + 2 != total || dst_off + total > out_capacity) atomicExch(err_flag, 1u);
    }
    group_sync();
    if (dst_off + total > out_capacity) continue;
    const uint32_t payload = total - 2;                        // bytes covered by the CRC-16
    const uint32_t hdr_bits = S.seg_start[0], end_bits = S.seg_start[channels];
    const uint32_t *slots_f = slots + (size_t)f * vch * slot_words;
    uint8_t *dst = out + dst_off;
    const uint32_t a = (uint32_t)(reinterpret_cast<uintptr_t>(dst) & 15u);   // bytes of the first chunk that are not ours
    uint8_t *g0 = dst - a;
    const uint32_t span = a + payload;
    const uint32_t nfull = span >> 4, tl = span & 15;
    // rows of ROW 16-byte chunks, one chunk per thread and row: 30 of a warp's 32 lanes / 120 of a CTA's 128 threads, because x^(128 * ROW)
    // is then a two-term multiplier and the CRC-16 needs no table in the loop (CrcFold, frb_crc16.cuh)
    constexpr int ROW = TPF == 32 ? 30 : 120;
    const uint32_t rows = nfull / (uint32_t)ROW, rem = nfull - rows * (uint32_t)ROW;
    const CrcTables &T = SS.T;

    // A thread visits its chunks in increasing order, so the subframe that holds a chunk only moves forward: the
    // segment search resumes where the previous chunk left it (it restarted from 0 for every chunk: 19 % of the kernel's
    // instructions, profiles/r01_ncu_emit_v7.txt).  seg_start[] entries and the chunk's register state: per frame.
    uint32_t ch = 0, seg_lo = S.seg_start[0], seg_hi = S.seg_start[1];
    const uint32_t *seg_sl = slots_f + (size_t)S.slot_of[0] * slot_words;
    // Warp-per-frame groups: a frame's partial head and tail chunks (its start and end are not 16-byte aligned) were produced
    // byte by byte by ONE lane (~50 instructions per byte, up to 30 bytes per frame) while the other 31 waited -- for 6 KB
    // frames (C5) about a third of the kernel.  Here the warp produces them together, one byte per lane, and assembles the
    // chunk's four words with warp-wide ORs; every lane gets the words, lane 0 (head) / lane 31 (tail) feed them to the CRC.
    // (CTA-per-frame groups do the same inside the warp that owns the chunk -- warp 0 for the head, the last warp for the tail:
    // there the single lane was the straggler every other thread waited for at the frame's closing barrier.)
    const int lane = tid & 31;
    auto coop_partial = [&](int32_t b_first /* frame byte of the chunk's byte 0 */, uint32_t nbytes, uint8_t *gdst, uint32_t (&w)[4]) {
        const bool valid = (uint32_t)lane < nbytes && b_first + lane >= 0;      // called by all 32 lanes of ONE warp
        uint32_t contrib = 0;
        if (valid) {
            const uint32_t byte = emit_gather32(8u * (uint32_t)(b_first + lane), S, channels, hdr_bits, end_bits, slots_f, slot_words) >> 24;
            gdst[lane] = (uint8_t)byte;
            contrib = byte << (24 - 8 * (lane & 3));
        }
#pragma unroll
        for (int q = 0; q < 4; q++) w[q] = __reduce_or_sync(0xFFFFFFFFu, (lane >> 2) == q ? contrib : 0u);
    };
    uint32_t w_head[4] = {0, 0, 0, 0};
    const bool head_pre = a > 0 && nfull >= 1;                   // uniform over the group
    if (head_pre && (tid >> 5) == 0) coop_partial(-(int32_t)a, 16, g0, w_head);
    // produce chunk c: returns its four big-endian words (head-masked), stores its bytes
    auto do_chunk = [&](uint32_t c, uint32_t (&w)[4], uint32_t nbytes /* valid bytes from the chunk start, 16 = full */) {
        const int32_t b0 = (int32_t)(16 * c) - (int32_t)a;    // frame byte of the chunk's first byte (negative in the head chunk)
        if (head_pre && c == 0) {
#pragma unroll
            for (int q = 0; q < 4; q++) w[q] = w_head[q];
            return;
        }
        if (b0 >= 0 && nbytes == 16) {
            const uint32_t P = 8u * (uint32_t)b0;
            // common case: all 128 bits lie inside one subframe -> five slot words, four funnel shifts.  The subframe's bounds and
            // slot address sit in registers and are looked up again only when a chunk leaves it (a subframe is a dozen rows long):
            // the three shared-memory loads and the 64-bit multiply per chunk were at the head of the chunk's dependent chain.
            if (P >= seg_hi) {
                while (ch + 1 < channels && S.seg_start[ch + 1] <= P) ch++;
                seg_lo = S.seg_start[ch];
                seg_hi = S.seg_start[ch + 1];
                seg_sl = slots_f + (size_t)S.slot_of[ch] * slot_words;
            }
            if (P >= hdr_bits && P + 128 <= seg_hi) {
                const uint32_t o = P - seg_lo;
                const uint32_t *sl = seg_sl + (o >> 5);
                const uint32_t sh = o & 31;
#if FRB_EMIT_VLOAD
                // the five words as TWO aligned 16-byte loads (slots are 16-byte aligned and over-allocated by a vector): five
                // 4-byte loads at a 16-byte lane stride cost 20 L1 wavefronts per warp against 8.  The word offset inside the
                // vector is the same for every lane of a warp inside one subframe, so the switch does not diverge.
                const uint32_t k = (uint32_t)((reinterpret_cast<uintptr_t>(sl) >> 2) & 3u);
                const uint4 *al = reinterpret_cast<const uint4 *>(sl - k);
                const uint4 a4 = __ldg(al), b4 = __ldg(al + 1);
                // The loop is one dependent chain per chunk (segment lookup -> two loads from DRAM -> funnel shifts -> store -> CRC
                // fold) and a thread has one chunk in flight: ask for the words of the chunk it will need N rows on while this one is
                // on its way.  Same subframe only, so the address is inside this frame's slot.  Same-box A/B (tools/enc_kernels_ab.py): C3
                // 0.836 -> 0.703 ms, C5 1.111 -> 0.991 ms with one row ahead into L1; two rows ahead or L2 prefetches measure the same or worse.
#if FRB_EMIT_PF_L1
                if (P + 128u * ROW * FRB_EMIT_PF_L1 + 128 <= seg_hi)
                    asm volatile("prefetch.global.L1 [%0];" ::"l"(al + ROW * FRB_EMIT_PF_L1 + 1));
#endif
#if FRB_EMIT_PF_L2
                if (P + 128u * ROW * FRB_EMIT_PF_L2 + 128 <= seg_hi)
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(al + ROW * FRB_EMIT_PF_L2 + 1));
#endif
                uint32_t v0, v1, v2, v3, v4;
                switch (k) {
                    case 0: v0 = a4.x; v1 = a4.y; v2 = a4.z; v3 = a4.w; v4 = b4.x; break;
                    case 1: v0 = a4.y; v1 = a4.z; v2 = a4.w; v3 = b4.x; v4 = b4.y; break;
                    case 2: v0 = a4.z; v1 = a4.w; v2 = b4.x; v3 = b4.y; v4 = b4.z; break;
                    default: v0 = a4.w; v1 = b4.x; v2 = b4.y; v3 = b4.z; v4 = b4.w; break;
                }
#else
                uint32_t v0 = __ldg(sl), v1 = __ldg(sl + 1), v2 = __ldg(sl + 2), v3 = __ldg(sl + 3), v4 = __ldg(sl + 4);
#endif
                w[0] = __funnelshift_l(v1, v0, sh); w[1] = __funnelshift_l(v2, v1, sh);
                w[2] = __funnelshift_l(v3, v2, sh); w[3] = __funnelshift_l(v4, v3, sh);
            } else if (P >= seg_lo && P < seg_hi && ch + 1 < channels && P + 128 <= S.seg_start[ch + 2]) {
                // the chunk runs from subframe ch into subframe ch + 1 (seven such chunks per 8-channel frame, one lane of a row of 30):
                // every word is A's bits, B's bits or t bits of A followed by B's first 32 - t -- both fetched for every word, so the 16
                // loads are independent.  Through the general path (a loop of dependent segment searches and loads per word) this one
                // lane held its row up for several memory latencies.
                const uint32_t *slB = slots_f + (size_t)S.slot_of[ch + 1] * slot_words;
                auto fetch32 = [](const uint32_t *sl, uint32_t o) {
                    const uint32_t wi = o >> 5;
                    return __funnelshift_l(__ldg(sl + wi + 1), __ldg(sl + wi), o & 31);
                };
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    const uint32_t Pq = P + 32u * q;
                    const bool inA = Pq < seg_hi;
                    const uint32_t a = fetch32(seg_sl, inA ? Pq - seg_lo : 0u), b = fetch32(slB, inA ? 0u : Pq - seg_hi);
                    const uint32_t t = seg_hi - Pq;                 // bits of A in this word (meaningful when inA)
                    w[q] = !inA ? b : t >= 32 ? a : ((a & ~(0xFFFFFFFFu >> t)) | (b >> t));
                }
            } else {
#pragma unroll
                for (int q = 0; q < 4; q++) w[q] = emit_gather32(P + 32u * q, S, channels, hdr_bits, end_bits, slots_f, slot_words);
            }
            *reinterpret_cast<uint4 *>(g0 + 16 * (size_t)c) = make_uint4(bswap32(w[0]), bswap32(w[1]), bswap32(w[2]), bswap32(w[3]));
        } else {
#pragma unroll
            for (int q = 0; q < 4; q++) w[q] = 0;
            for (uint32_t j = 0; j < nbytes; j++) {
                const int32_t b = b0 + (int32_t)j;
                if (b < 0) continue;
                const uint32_t byte = emit_gather32(8u * (uint32_t)b, S, channels, hdr_bits, end_bits, slots_f, slot_words) >> 24;
                w[j >> 2] |= byte << (24 - 8 * (j & 3));
                g0[16 * (size_t)c + j] = (uint8_t)byte;
            }
        }
    };

    uint32_t v = 0;
    if (tid < ROW) {
        CrcFold F;
        crcfold_init(F);
        for (uint32_t m = 0; m < rows; m++) {
            uint32_t w[4];
            do_chunk(m * ROW + tid, w, 16);
            crcfold_step<ROW>(F, w);
        }
        // x^16 (message -> CRC register), the chunks of the last full row after this thread's, then everything after the full rows
        if (rows) v = gf16_mul(gf16_mul(crcfold_finish(F), T.xp[16 * (ROW - 1 - tid) + 2]), T.xp[16 * rem + tl]);
        if ((uint32_t)tid < rem) {
            uint32_t w[4];
            do_chunk(rows * ROW + tid, w, 16);
            v ^= gf16_mul(crc16_words4(0, w, T.s4), T.xp[16 * (rem - 1 - tid) + tl]);
        }
    }
    if (tl && (tid >> 5) == ((TPF - 1) >> 5)) {              // the group's last warp, all 32 lanes; tl is uniform over the group
        uint32_t w[4];
        coop_partial((int32_t)(16 * nfull) - (int32_t)a, tl, g0 + 16 * (size_t)nfull, w);
        if (tid == TPF - 1) {
            uint32_t c = 0;
            for (uint32_t q = 0; q < tl; q++) {
                const uint32_t byte = (w[q >> 2] >> (24 - 8 * (q & 3))) & 0xFF;
                c = ((c << 8) & 0xFFFFu) ^ T.s4[((c >> 8) ^ byte) & 0xFF];
            }
            v ^= c;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v ^= __shfl_xor_sync(0xFFFFFFFFu, v, o);
    if (TPF == kEmitThreads) {
        if ((tid & 31) == 0) SS.red[tid >> 5] = v;
        __syncthreads();
        if (tid == 0) {
            uint32_t crc = 0;
            for (int w = 0; w < kEmitThreads / 32; w++) crc ^= SS.red[w];
            dst[payload] = (uint8_t)(crc >> 8);
            dst[payload + 1] = (uint8_t)crc;
        }
    } else if (tid == 0) {
        dst[payload] = (uint8_t)(v >> 8);
        dst[payload + 1] = (uint8_t)v;
    }
    }
}

// ---- workspace -----------------------------------------------------------------
struct EncWorkspace {
    EncStreamDev *streams;
    uint32_t *sub_bits;
    uint32_t *frame_bytes;
    unsigned long long *frame_off;
    unsigned long long *stream_bytes;
    unsigned long long *out_offs;
    uint32_t *err_flag;
    float *window;
    EncSubStats *stats;
    double *autoc;
    EncCand *cands;
    uint32_t *slow_tasks;
    FrameDesc *frame_table;
    unsigned long long *fx_fin;
    uint32_t *slots;
    EncStreamDev *vstreams;      // two-channel streams: stream table of the four virtual channels (L, R, M, S)
    uint32_t *sub_est;           //   estimated bits per virtual subframe (libFLAC's decision metric)
    uint8_t *frame_sel;          //   chosen channel assignment per frame
    int32_t *vaudio;             //   planar audio of the virtual channels
};
// Two-channel streams are analysed as four virtual channels (see k_ms_choose); the workspace is laid out for that
// whenever channels == 2, whether or not the level / bit depth ends up using it.
static inline uint32_t enc_virtual_channels(const frb_encode_params *p) { return p->channels == 2 ? 4u : p->channels; }
static inline uint32_t enc_slot_bps(const frb_encode_params *p) { return p->bps + (p->channels == 2 ? 1u : 0u); }
static inline size_t enc_ws_layout(const frb_encode_params *p, uint64_t total_frames, void *base, EncWorkspace *w) {
    size_t off = 0;
    uint8_t *b = (uint8_t *)base;
    const uint64_t subs = total_frames * enc_virtual_channels(p);
#define FRB_TAKE(field, type, count)                                         \
    if (w) w->field = (type *)(b + off);                                      \
    off += align256(sizeof(type) * (size_t)(count));
    FRB_TAKE(streams, EncStreamDev, p->n_streams)
    FRB_TAKE(sub_bits, uint32_t, subs)
    FRB_TAKE(frame_bytes, uint32_t, total_frames)
    FRB_TAKE(frame_off, unsigned long long, total_frames)
    FRB_TAKE(stream_bytes, unsigned long long, p->n_streams)
    FRB_TAKE(out_offs, unsigned long long, p->n_streams)
    FRB_TAKE(err_flag, uint32_t, 64)
    FRB_TAKE(window, float, FRB_MAX_BLOCKSIZE)
    FRB_TAKE(stats, EncSubStats, subs)
    FRB_TAKE(autoc, double, subs * kMaxSets * kLags)
    FRB_TAKE(cands, EncCand, subs * kMaxCands)
    FRB_TAKE(slow_tasks, uint32_t, subs)
    FRB_TAKE(frame_table, FrameDesc, total_frames)
    FRB_TAKE(fx_fin, unsigned long long, subs * 64)
    FRB_TAKE(slots, uint32_t, subs * slot_words_for(p->blocksize, enc_slot_bps(p)))
    FRB_TAKE(vstreams, EncStreamDev, p->n_streams)
    FRB_TAKE(sub_est, uint32_t, subs)
    FRB_TAKE(frame_sel, uint8_t, total_frames)
    FRB_TAKE(vaudio, int32_t, p->channels == 2 ? total_frames * (uint64_t)p->blocksize * 4u : 0u)
#undef FRB_TAKE
    return off;
}

static inline void make_tukey(float *w, int L, float p) {
    // FLAC__window_tukey
    for (int n = 0; n < L; n++) w[n] = 1.0f;
    if (p <= 0.0f) return;
    const int Np = (int)(p / 2.0f * L) - 1;
    if (Np > 0) {
        for (int n = 0; n <= Np; n++) {
            w[n] = (float)(0.5f - 0.5f * cosf((float)(M_PI * n / Np)));
            w[L - Np - 1 + n] = (float)(0.5f - 0.5f * cosf((float)(M_PI * (n + Np) / Np)));
        }
    }
}

// libFLAC's stereo decorrelation applies to exactly two channels at the presets with do_mid_side; the GPU path covers
// 16-bit streams (17-bit side channel)
// ... and 32-bps streams whose caller vouches that every sample is below 2^30 in magnitude (FRB_ENC_RANGE_30: the tile path's
// 24-bit audio of float32 / 32-bit rasters), so that the 33-bit side channel L - R is held exactly by the int32 planar audio.
static inline bool enc_mid_side(const frb_encode_params *p) {
    return p->channels == 2 && level_cfg(p->level).mid_side && (p->bps == 16 || (p->bps == 32 && (p->reserved & 2u)));
}

// frb_encode_emit needs the frame count frb_encode_analyse computed; it is remembered per host thread for the usual
// analyse -> emit sequence on one workspace (otherwise emit reads it back from the stream table: one more round trip)
struct LastAnalyse { const void *ws = nullptr; uint64_t frames = 0; uint32_t n_streams = 0; };
static thread_local LastAnalyse t_last_analyse;

static inline bool enc_params_ok(const frb_encode_params *p) {
    return p && p->n_streams >= 1 && p->channels >= 1 && p->channels <= FRB_MAX_CHANNELS &&
           (p->bps == 16 || p->bps == 32) && p->blocksize >= 16 && p->blocksize <= FRB_MAX_BLOCKSIZE && p->level <= 8;
}

}  // namespace frb

extern "C" int frb_encode_workspace_size(const frb_encode_params *p, uint64_t total_frames, size_t *bytes) {
    if (!frb::enc_params_ok(p) || !bytes) return FRB_ERR_INVALID_ARG;
    *bytes = frb::enc_ws_layout(p, total_frames, nullptr, nullptr);
    return FRB_OK;
}

extern "C" int frb_encode_analyse(const frb_encode_params *p, const void *d_audio,
                                  const uint64_t *h_n_samples, const uint32_t *h_sample_rate,
                                  const int64_t *h_audio_base, void *d_workspace, size_t workspace_bytes,
                                  uint64_t *d_stream_bytes, uint64_t *h_stream_bytes, void *stream) {
    using namespace frb;
    if (!enc_params_ok(p) || !d_audio || !h_n_samples || !h_sample_rate || !h_audio_base || !d_workspace) return FRB_ERR_INVALID_ARG;
    int rc = ensure_tables_impl();
    if (rc) return rc;
    std::vector<EncStreamDev> hs(p->n_streams);
    uint64_t frames = 0;
    for (uint32_t i = 0; i < p->n_streams; i++) {
        if (h_n_samples[i] == 0) return FRB_ERR_INVALID_ARG;
        EncStreamDev d;
        d.n_samples = h_n_samples[i]; d.audio_base = h_audio_base[i]; d.out_offset = 0;
        d.sample_rate = h_sample_rate[i]; d.frame_base = (uint32_t)frames;
        d.n_frames = (uint32_t)((h_n_samples[i] + p->blocksize - 1) / p->blocksize); d.pad = 0;
        frames += d.n_frames;
        hs[i] = d;
    }
    if (frames == 0 || frames * p->channels > 0x7FFFFFFFull) return FRB_ERR_INVALID_ARG;
    EncWorkspace w;
    if (enc_ws_layout(p, frames, d_workspace, &w) > workspace_bytes) return FRB_ERR_OVERFLOW;
    cudaStream_t s = (cudaStream_t)stream;
    // analysis window of this (blocksize, apodization count): computed once per host thread and kept
    static thread_local std::vector<float> win;
    static thread_local uint32_t win_bs = 0, win_n = 0;
    if (win_bs != p->blocksize || win_n != (uint32_t)level_cfg(p->level).windows) {
        win.assign(FRB_MAX_BLOCKSIZE, 1.0f);
        make_tukey(win.data(), (int)p->blocksize, 0.5f / (float)level_cfg(p->level).windows);
        win_bs = p->blocksize; win_n = (uint32_t)level_cfg(p->level).windows;
    }
    // two-channel streams at a mid/side preset: analyse the four virtual channels L, R, M, S (an_* below)
    const bool ms = enc_mid_side(p);
    const uint32_t an_ch = ms ? 4u : p->channels;
    std::vector<EncStreamDev> vhs;
    if (ms) {
        vhs = hs;
        uint64_t cum = 0;
        for (uint32_t i = 0; i < p->n_streams; i++) { vhs[i].audio_base = (int64_t)(4 * cum); cum += hs[i].n_samples; }
        if (cum > frames * (uint64_t)p->blocksize) return FRB_ERR_INVALID_ARG;
        FRB_TRY(small_upload(w.vstreams, vhs.data(), sizeof(EncStreamDev) * vhs.size(), s));
    }
    FRB_TRY(small_upload(w.streams, hs.data(), sizeof(EncStreamDev) * hs.size(), s));
    FRB_TRY(small_upload(w.window, win.data(), sizeof(float) * FRB_MAX_BLOCKSIZE, s));
    FRB_TRY(small_fill(w.err_flag, 0u, 256, s));
    // (small_upload copies its source into pinned staging before it returns: no synchronisation needed here)
    const std::vector<EncStreamDev> &ahs = ms ? vhs : hs;
    const EncStreamDev *an_streams = ms ? w.vstreams : w.streams;
    // reserved bit 0: d_audio holds int16 elements (16-bps streams only); the mid/side expansion always writes int32
    const bool a16 = (p->reserved & 1u) != 0;
    if (a16 && p->bps != 16) return FRB_ERR_INVALID_ARG;
    const EncSrc in_audio = {d_audio, a16 ? 1u : 0u};
    const EncSrc an_audio = ms ? EncSrc{w.vaudio, 0u} : in_audio;
    const uint32_t an_esz = an_audio.a16 ? 2u : 4u;
    const uint32_t side_ch = ms ? 3u : 0xFFFFFFFFu;
    uint32_t *sub_est = ms ? w.sub_est : nullptr;
    if (ms) {
        uint64_t max_n = 0;
        for (uint32_t i = 0; i < p->n_streams; i++) max_n = std::max<uint64_t>(max_n, hs[i].n_samples);
        uint32_t gx = (uint32_t)std::min<uint64_t>((max_n + 256 * 8 - 1) / (256 * 8), std::max<uint32_t>(1u, (uint32_t)kNumSMs * 16 / p->n_streams));
        if (gx < 1) gx = 1;
        k_ms_expand<<<gx * p->n_streams, 256, 0, s>>>(w.streams, w.vstreams, in_audio, w.vaudio, gx, w.err_flag);
        FRB_LAUNCH_CHECK("k_ms_expand");
    }
    const uint32_t slot_words = slot_words_for(p->blocksize, enc_slot_bps(p));
    static bool attr_set[64] = {false};
    if (first_call_on_device(attr_set)) {
        FRB_CUDA(cudaFuncSetAttribute(k_encode_subframes, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(EncShared)));
        // the analysis kernels spill to local memory (L1-resident) and use little shared memory: give L1 the rest
        // (same-box A/B: 86.0 -> 87.1 GSamples/s on C3)
        cudaFuncSetAttribute(k_enc_code<false>, cudaFuncAttributePreferredSharedMemoryCarveout, 20);
        cudaFuncSetAttribute(k_enc_stats<false, 9>, cudaFuncAttributePreferredSharedMemoryCarveout, 5);
        cudaFuncSetAttribute(k_enc_stats<false, 13>, cudaFuncAttributePreferredSharedMemoryCarveout, 5);
        cudaFuncSetAttribute(k_enc_stats<false, 0>, cudaFuncAttributePreferredSharedMemoryCarveout, 5);
        cudaGetLastError();
    }
    // Full, 16-byte aligned 4096-sample blocks go through the three-kernel fast path; everything else (the short
    // last frame of a stream, channels that start at an unaligned sample) is listed for the one-kernel encoder.
    const LevelCfg cfg = level_cfg(p->level);
    const bool fast = p->blocksize == (uint32_t)kMaxBlock && cfg.max_po >= 3 && cfg.max_po <= 6;
    std::vector<uint32_t> slow;
    const uint32_t total_tasks = (uint32_t)(frames * an_ch);
    if (fast) {
        const uint64_t base_addr = (uint64_t)reinterpret_cast<uintptr_t>(an_audio.audio);
        if (base_addr & (an_esz - 1)) return FRB_ERR_INVALID_ARG;
        for (uint32_t i = 0; i < p->n_streams; i++) {
            const EncStreamDev &d = ahs[i];
            const bool tail = (d.n_samples % p->blocksize) != 0;
            for (uint32_t c = 0; c < an_ch; c++) {
                const bool aligned = ((base_addr + ((uint64_t)d.audio_base + (uint64_t)c * d.n_samples) * an_esz) & (an_esz == 2 ? 7u : 15u)) == 0;
                for (uint32_t k = aligned ? (tail ? d.n_frames - 1 : d.n_frames) : 0; k < d.n_frames; k++)
                    slow.push_back((d.frame_base + k) * an_ch + c);
            }
        }
        if (!slow.empty()) {
            if (4 * slow.size() <= (1u << 20)) FRB_TRY(small_upload(w.slow_tasks, slow.data(), 4 * slow.size(), s));
            else {
                FRB_CUDA(cudaMemcpyAsync(w.slow_tasks, slow.data(), 4 * slow.size(), cudaMemcpyHostToDevice, s));
                FRB_CUDA(cudaStreamSynchronize(s));
            }
        }
    }
    // per-frame descriptors (stream index, sample position): the analysis kernels and the frame assembly look frames up
    // here instead of searching the stream table per CTA
    k_frame_table<<<(uint32_t)((frames + 255) / 256), 256, 0, s>>>(an_streams, p->n_streams, p->blocksize, (uint32_t)frames, w.frame_table);
    FRB_LAUNCH_CHECK("k_frame_table");
    prof_begin(6, s);
    if (fast && slow.size() < total_tasks) {
        const uint32_t windows = (uint32_t)cfg.windows, max_lpc = (uint32_t)cfg.max_lpc_order;
        const uint32_t n_cands = max_lpc == 0 ? 0u : windows == 1 ? 1u : windows == 2 ? 3u : 9u;     // LPC candidates
        const bool wide = p->bps > 16;
        // one CTA per subframe; with mid/side the 17-bit side channel (virtual channel 3) runs in the 64-bit kernels
        const dim3 grid((uint32_t)frames, ms ? 3u : p->channels), grid_side((uint32_t)frames, 1);
        // 16-bit subframes: one warp each, FIXED search included (k_enc_stats_warp); FRB_STATS_CTA=1 selects the CTA kernel
        // and k_enc_fixed for them as well (A/B runs).  The 32-bps and side-channel subframes always take the CTA kernel.
        static int stats_cta = -1;
        if (stats_cta < 0) { const char *e = getenv("FRB_STATS_CTA"); stats_cta = e ? atoi(e) : 0; }
        const bool warp_stats = !wide && stats_cta != 1;
        const uint32_t main_ch = ms ? 3u : p->channels;
        prof_begin(4, s);
#define FRB_STATS(W, NL, G, C0, EX) k_enc_stats<W, NL><<<G, kEncThreads, 0, s>>>(w.frame_table, an_ch, p->bps, windows, (uint32_t)cfg.max_po, an_audio, \
            w.window, w.stats, w.autoc, w.fx_fin, C0, EX)
#define FRB_STATS_WARP(NL) k_enc_stats_warp<NL><<<(uint32_t)((frames * main_ch + kStatsWarps - 1) / kStatsWarps), kStatsWarps * 32, 0, s>>>( \
            w.frame_table, an_ch, main_ch, (uint32_t)(frames * main_ch), p->bps, windows, (uint32_t)cfg.max_po, an_audio, w.window, w.stats, w.autoc)
#define FRB_STATS_L(NL) do { if (warp_stats) FRB_STATS_WARP(NL); else if (wide) FRB_STATS(true, NL, grid, 0u, 0u); else FRB_STATS(false, NL, grid, 0u, 0u); \
                             if (ms) FRB_STATS(true, NL, grid_side, 3u, 1u); } while (0)
        if (max_lpc == 0) FRB_STATS_L(0);
        else if (max_lpc <= 8) FRB_STATS_L(9);
        else FRB_STATS_L(13);
#undef FRB_STATS_L
#undef FRB_STATS_WARP
#undef FRB_STATS
        FRB_LAUNCH_CHECK("k_enc_stats");
        // the FIXED search of the subframes k_enc_stats analysed: all of them, or only the side channel
        const uint32_t fx_c0 = warp_stats ? 3u : 0u, fx_nch = warp_stats ? 1u : an_ch;
        if (!warp_stats || ms) {
            const uint32_t fx_total = (uint32_t)(frames * fx_nch);
            k_enc_fixed<<<(fx_total + 3) / 4, 128, 0, s>>>(w.frame_table, an_ch, fx_c0, fx_nch, p->bps, (uint32_t)cfg.max_po, fx_total,
                                                         an_audio, w.stats, w.fx_fin, side_ch);
            FRB_LAUNCH_CHECK("k_enc_fixed");
        }
        prof_end(4, s);
        const uint32_t n_slots = n_cands;
        const uint32_t model_threads = total_tasks * n_slots;
        if (n_cands) {
#define FRB_MODEL(MO) k_enc_model<MO><<<(model_threads + 127) / 128, 128, 0, s>>>(w.frame_table, an_ch, p->bps, \
            p->blocksize, windows, max_lpc, n_slots, total_tasks, an_audio, w.stats, w.autoc, w.cands, side_ch)
        if (max_lpc <= 8) FRB_MODEL(8); else FRB_MODEL(12);
#undef FRB_MODEL
        FRB_LAUNCH_CHECK("k_enc_model");
        }
        prof_begin(0, s);
#define FRB_CODE(W, G, C0, EX) k_enc_code<W><<<G, kEncThreads, 0, s>>>(w.frame_table, an_ch, p->bps, (uint32_t)cfg.max_po, n_cands, an_audio, \
            w.stats, w.cands, slot_words, w.slots, w.sub_bits, C0, EX, sub_est)
        if (wide) FRB_CODE(true, grid, 0u, 0u); else FRB_CODE(false, grid, 0u, 0u);
        if (ms) FRB_CODE(true, grid_side, 3u, 1u);
#undef FRB_CODE
        prof_end(0, s);
        FRB_LAUNCH_CHECK("k_enc_code");
    }
    if (!fast || !slow.empty()) {
        const uint32_t grid = fast ? (uint32_t)slow.size() : total_tasks;
        k_encode_subframes<<<grid, kEncThreads, sizeof(EncShared), s>>>(
            an_streams, p->n_streams, an_ch, p->bps, p->blocksize, p->level, an_audio, w.window, slot_words, w.slots, w.sub_bits,
            fast ? w.slow_tasks : nullptr, side_ch, sub_est);
        FRB_LAUNCH_CHECK("k_encode_subframes");
    }
    prof_end(6, s);
    if (ms) {
        k_ms_choose<<<(uint32_t)((frames + 255) / 256), 256, 0, s>>>(w.streams, p->n_streams, p->blocksize, (uint32_t)frames,
                                                                   (uint32_t)cfg.loose, w.sub_est, w.frame_sel);
        FRB_LAUNCH_CHECK("k_ms_choose");
    }
    k_frame_sizes<<<(uint32_t)((frames + 255) / 256), 256, 0, s>>>(w.streams, p->n_streams, p->channels, p->blocksize,
                                                                 (uint32_t)frames, w.sub_bits, w.frame_bytes, an_ch, ms ? w.frame_sel : nullptr);
    FRB_LAUNCH_CHECK("k_frame_sizes");
    t_last_analyse.ws = d_workspace; t_last_analyse.frames = frames; t_last_analyse.n_streams = p->n_streams;
    k_stream_scan<<<p->n_streams, 1024, 0, s>>>(w.streams, w.frame_bytes, w.frame_off, w.stream_bytes);
    FRB_LAUNCH_CHECK("k_stream_scan");
    if (d_stream_bytes)
        FRB_CUDA(cudaMemcpyAsync(d_stream_bytes, w.stream_bytes, 8 * (size_t)p->n_streams, cudaMemcpyDeviceToDevice, s));
    if (h_stream_bytes) {
        FRB_TRY(small_download(h_stream_bytes, w.stream_bytes, 8 * (size_t)p->n_streams, s));
    }
    return FRB_OK;
}

extern "C" int frb_encode_emit(const frb_encode_params *p, void *d_workspace, size_t workspace_bytes,
                               const uint64_t *h_out_offset, uint8_t *d_out, size_t out_capacity,
                               uint32_t *d_frame_bytes, void *stream) {
    using namespace frb;
    if (!enc_params_ok(p) || !d_workspace || !d_out) return FRB_ERR_INVALID_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    // recover the frame count from the stream table written by analyse
    EncWorkspace w0;
    (void)enc_ws_layout(p, 0, d_workspace, &w0);
    uint64_t frames;
    if (t_last_analyse.ws == d_workspace && t_last_analyse.n_streams == p->n_streams && t_last_analyse.frames) frames = t_last_analyse.frames;
    else {
        EncStreamDev last;
        FRB_TRY(small_download(&last, w0.streams + (p->n_streams - 1), sizeof last, s));
        frames = (uint64_t)last.frame_base + last.n_frames;
    }
    EncWorkspace w;
    if (enc_ws_layout(p, frames, d_workspace, &w) > workspace_bytes) return FRB_ERR_OVERFLOW;
    if (h_out_offset) {
        FRB_TRY(small_upload(w.out_offs, h_out_offset, 8 * (size_t)p->n_streams, s));
        k_set_out_offsets<<<(p->n_streams + 255) / 256, 256, 0, s>>>(w.streams, w.out_offs, p->n_streams);
        FRB_LAUNCH_CHECK("k_set_out_offsets");
    } else {        // packed: stream s starts where stream s-1 ends, computed on the device
        k_pack_out_offsets<<<1, 1024, 0, s>>>(w.streams, w.stream_bytes, p->n_streams);
        FRB_LAUNCH_CHECK("k_pack_out_offsets");
    }
    prof_begin(2, s);
    {
        // a warp per frame; the whole CTA per frame only on request (FRB_EMIT_TPF=128, A/B runs): with the table-free CRC the warp form
        // is the faster one for large frames as well (C3's 48 KB frames: 0.83 against 1.02 ms; C5's 6 KB frames: 1.11 against 1.97 ms)
        static int tpf_cfg = -1;
        if (tpf_cfg < 0) { const char *e = getenv("FRB_EMIT_TPF"); tpf_cfg = e ? atoi(e) : 0; }
        const bool warp_per_frame = tpf_cfg != 128;
        const uint32_t vch = enc_mid_side(p) ? 4u : p->channels;
        const uint8_t *sel = enc_mid_side(p) ? w.frame_sel : nullptr;
        const uint32_t sw = slot_words_for(p->blocksize, enc_slot_bps(p));
        if (warp_per_frame)
            k_emit_frames<32><<<(uint32_t)std::min<uint64_t>((frames + 3) / 4, (uint64_t)kNumSMs * 16), kEmitThreads, 0, s>>>(
                w.streams, p->n_streams, p->channels, p->bps, p->blocksize, (uint32_t)frames, w.sub_bits, w.slots, sw,
                w.frame_bytes, w.frame_off, d_out, (uint64_t)out_capacity, w.err_flag, vch, sel, w.frame_table);
        else
            k_emit_frames<kEmitThreads><<<(uint32_t)std::min<uint64_t>(frames, (uint64_t)kNumSMs * 16), kEmitThreads, 0, s>>>(
                w.streams, p->n_streams, p->channels, p->bps, p->blocksize, (uint32_t)frames, w.sub_bits, w.slots, sw,
                w.frame_bytes, w.frame_off, d_out, (uint64_t)out_capacity, w.err_flag, vch, sel, w.frame_table);
    }
    prof_end(2, s);
    FRB_LAUNCH_CHECK("k_emit_frames");
    if (d_frame_bytes)
        FRB_CUDA(cudaMemcpyAsync(d_frame_bytes, w.frame_bytes, 4 * (size_t)frames, cudaMemcpyDeviceToDevice, s));
    uint32_t h_err[2] = {0, 0};
    FRB_TRY(small_download(h_err, w.err_flag, 8, s));
    if (h_err[1]) return FRB_ERR_INVALID_ARG;     // FRB_ENC_RANGE_30 was set but a side sample did not fit int32
    if (h_err[0]) return FRB_ERR_OVERFLOW;
    return FRB_OK;
}
extern "C" int frb_encode_index(const frb_encode_params *p, void *d_workspace, size_t workspace_bytes,
                                uint32_t *d_frame_bytes, uint32_t *d_sub_bitoff, void *stream) {
    using namespace frb;
    if (!enc_params_ok(p) || !d_workspace || (!d_frame_bytes && !d_sub_bitoff)) return FRB_ERR_INVALID_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    if (!(t_last_analyse.ws == d_workspace && t_last_analyse.n_streams == p->n_streams && t_last_analyse.frames)) return FRB_ERR_INVALID_ARG;
    const uint64_t frames = t_last_analyse.frames;           // the index describes the analyse that just ran on this workspace
    EncWorkspace w;
    if (enc_ws_layout(p, frames, d_workspace, &w) > workspace_bytes) return FRB_ERR_OVERFLOW;
    if (d_frame_bytes) FRB_CUDA(cudaMemcpyAsync(d_frame_bytes, w.frame_bytes, 4 * (size_t)frames, cudaMemcpyDeviceToDevice, s));
    if (d_sub_bitoff) {
        const bool ms = enc_mid_side(p);
        k_export_index<<<(uint32_t)((frames + 255) / 256), 256, 0, s>>>(w.streams, p->n_streams, p->channels, p->blocksize, (uint32_t)frames,
                                                                       w.sub_bits, ms ? 4u : p->channels, ms ? w.frame_sel : nullptr, d_sub_bitoff);
        FRB_LAUNCH_CHECK("k_export_index");
    }
    return FRB_OK;
}
static_assert(sizeof(frb::EncShared) <= 100 * 1024, "EncShared must allow >= 2 CTAs per SM");
