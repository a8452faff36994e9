// frb_encode_fast.cuh -- three-kernel subframe encoder for full 4096-sample blocks (the common case:
// every frame of a stream except its last one).  Included by frb_encode.cuh inside namespace frb.
//
// The one-kernel encoder (k_encode_subframes, kept for short tail frames and unaligned channels) executed
// 16.6 warp instructions per sample at 48 % issue utilisation (profiles/r01_ncu_enc_v2_*): every phase went
// through padded shared-memory sample/residual buffers with per-element bounds checks, all reductions were
// 64-bit shuffles, and 255 of 256 threads idled at a barrier while lane 0 ran Levinson-Durbin, the order
// estimate (logarithms) and the coefficient quantisation in fp64.  Here the work is split where the data
// dependencies are:
//   k_enc_stats_warp  WARP per 16-bit subframe, 4 subframes per 128-thread CTA, no barrier: lane l walks the
//                 16-sample chunks 32j + l (j = 0..7) in registers (+12 halo samples read straight from
//                 global/L1): wasted bits, constant check, fixed-predictor abs sums (32-bit, REDUX warp
//                 sums), windowed autocorrelation for every apodization of the level (fp64 FMA chain in
//                 registers), and the FIXED candidate's Rice search -> ~200 bytes of statistics per subframe
//   k_enc_stats   the same per CTA (16 samples per thread) for the 32-bps and side-channel subframes (and
//                 every subframe with FRB_STATS_CTA=1); k_enc_fixed then runs their FIXED search
//   k_enc_model   ONE THREAD per (subframe, apodization): Levinson-Durbin, libFLAC's order estimate
//                 and coefficient quantisation -- the serial fp64 section now runs 32 subframes per
//                 warp instead of one lane per CTA -> candidate predictors (64 bytes each)
//   k_enc_code    CTA per subframe: residual of each candidate in registers, partition sums by a
//                 segmented warp butterfly, libFLAC's Rice estimate, winner selection, exact bit
//                 lengths, CTA scan, 64-bit per-thread bit accumulator with plain interior word stores,
//                 128-bit slot copy
// All decisions are the same as the one-kernel encoder's (and the oracle's): same estimates, same
// tie-breaks, same fp64 operation order in the model; the autocorrelation uses the same per-thread /
// butterfly / cross-warp summation tree as before (in k_enc_stats_warp: per chunk / butterfly / running sum
// over the chunk rows, the same additions).
#pragma once

constexpr int kMaxSets = 6;        // autocorrelation sets per subframe: root, 2 halves, 3 thirds (level 8)
constexpr int kMaxCands = 9;       // LPC candidates per subframe (level 8: 1 + 2 + 6); the FIXED candidate is searched before k_enc_code
constexpr int kLags = kMaxOrd + 1;

struct EncSubStats {
    unsigned long long e[5];       // fixed-predictor abs sums over i in [4, n)
    uint32_t wasted, flags;        // flags bit 0: constant signal, bit 1: FIXED candidate evaluated (fx_* valid)
    uint32_t fx_order, fx_bits, fx_po, fx_bad;     // guessed FIXED order, its estimated subframe bits, partition order; residual overflow
    uint8_t fx_params[64];         // Rice parameters of the FIXED candidate's best partition order
};
struct EncCand {                   // type 0 = no candidate, 2 FIXED, 3 LPC
    int32_t type, order, precision, shift;
    int32_t coefs[kMaxOrd];
};

// Per-frame descriptor table (k_frame_table, one binary search per FRAME): the three kernels index it
// directly instead of searching the stream table once per CTA (7 dependent loads before any work).
struct FrameDesc {
    int64_t src0;          // audio index of channel 0's first sample of this frame
    uint64_t ns;           // samples per channel of the stream (channel stride)
    uint32_t n, stream;    // samples in this frame, stream index
};
__global__ void __launch_bounds__(256)
k_frame_table(const EncStreamDev *__restrict__ streams, uint32_t n_streams, uint32_t blocksize, uint32_t total_frames,
              FrameDesc *__restrict__ out) {
    const uint32_t f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= total_frames) return;
    uint32_t lo = 0, hi = n_streams - 1;
    while (lo < hi) {
        const uint32_t mid = (lo + hi + 1) >> 1;
        if (streams[mid].frame_base <= f) lo = mid; else hi = mid - 1;
    }
    const EncStreamDev st = streams[lo];
    const uint32_t kf = f - st.frame_base;
    FrameDesc d;
    d.src0 = st.audio_base + (int64_t)kf * blocksize;
    d.ns = st.n_samples;
    d.n = (kf + 1 < st.n_frames) ? blocksize : (uint32_t)(st.n_samples - (uint64_t)kf * blocksize);
    d.stream = lo;
    out[f] = d;
}

__device__ __forceinline__ TaskLoc locate_task(const FrameDesc *__restrict__ frames, const EncSrc &S, uint32_t f, uint32_t c) {
    const FrameDesc d = frames[f];
    TaskLoc L;
    L.n = d.n;
    L.a16 = S.a16;
    L.src = audio_at(S, d.src0 + (int64_t)c * (int64_t)d.ns);
    return L;
}
// The fast path handles full 4096-sample blocks whose first sample is 16-byte aligned (the host lists every
// other subframe for the one-kernel encoder with the same predicate, see frb_encode_analyse).
// (int16 audio: 8-byte alignment is enough -- a channel that starts at a sample index of 4 mod 8 is read with 8-byte loads; with
// 16 bytes required, tiles of h*w = 4 mod 8 pixels would have sent every other band to the one-kernel encoder)
__device__ __forceinline__ bool fast_eligible(const TaskLoc &L) {
    return L.n == (uint32_t)kMaxBlock && (reinterpret_cast<uintptr_t>(L.src) & (L.a16 ? 7u : 15u)) == 0;
}

// compile-time choice between two arrays of the same type (a reference, so that the unused one stays dead)
template <bool FIRST, typename T>
__device__ __forceinline__ const T &pick_ref(const T &a, const T &b) { if constexpr (FIRST) return a; else return b; }

// two sign-extended int16 samples of a 32-bit word, one instruction each (the compiler emits PRMT with sign replication /
// an arithmetic shift; __byte_perm cannot express it: it masks the selector nibbles to 3 bits)
__device__ __forceinline__ int32_t s16_lo(uint32_t w) { return (int32_t)(int16_t)(uint16_t)w; }
__device__ __forceinline__ int32_t s16_hi(uint32_t w) { return (int32_t)w >> 16; }

// 16 own samples at xs[12..27], 12 halo samples (previous thread's tail, zeros for thread 0) at xs[0..11]
__device__ __forceinline__ void load_samples28(const TaskLoc &L, int tid, int32_t (&xs)[28]) {
    if (L.a16) {
        // int16 audio: the thread's 16 samples are 32 bytes (two 16-byte loads), the halo 24 bytes (three 8-byte loads)
        const uint4 *p = reinterpret_cast<const uint4 *>(reinterpret_cast<const int16_t *>(L.src) + tid * kSPT);
        const bool al16 = (reinterpret_cast<uintptr_t>(p) & 15u) == 0;          // uniform over the CTA (tid * 32 bytes)
#pragma unroll
        for (int q = 0; q < 2; q++) {
            uint4 v;
            if (al16) v = __ldg(p + q);
            else {
                const uint2 a = __ldg(reinterpret_cast<const uint2 *>(p) + 2 * q), b = __ldg(reinterpret_cast<const uint2 *>(p) + 2 * q + 1);
                v = make_uint4(a.x, a.y, b.x, b.y);
            }
            xs[12 + 8 * q] = s16_lo(v.x); xs[13 + 8 * q] = s16_hi(v.x); xs[14 + 8 * q] = s16_lo(v.y); xs[15 + 8 * q] = s16_hi(v.y);
            xs[16 + 8 * q] = s16_lo(v.z); xs[17 + 8 * q] = s16_hi(v.z); xs[18 + 8 * q] = s16_lo(v.w); xs[19 + 8 * q] = s16_hi(v.w);
        }
        if (tid > 0) {
            const uint2 *h = reinterpret_cast<const uint2 *>(p) - 3;
#pragma unroll
            for (int q = 0; q < 3; q++) {
                const uint2 v = __ldg(h + q);
                xs[4 * q] = s16_lo(v.x); xs[4 * q + 1] = s16_hi(v.x); xs[4 * q + 2] = s16_lo(v.y); xs[4 * q + 3] = s16_hi(v.y);
            }
        } else {
#pragma unroll
            for (int q = 0; q < 12; q++) xs[q] = 0;
        }
        return;
    }
    const int4 *p = reinterpret_cast<const int4 *>(reinterpret_cast<const int32_t *>(L.src) + tid * kSPT);
#pragma unroll
    for (int q = 0; q < 4; q++) {
        const int4 v = __ldg(p + q);
        xs[12 + 4 * q] = v.x; xs[13 + 4 * q] = v.y; xs[14 + 4 * q] = v.z; xs[15 + 4 * q] = v.w;
    }
    if (tid > 0) {
#pragma unroll
        for (int q = 0; q < 3; q++) {
            const int4 v = __ldg(p - 3 + q);
            xs[4 * q] = v.x; xs[4 * q + 1] = v.y; xs[4 * q + 2] = v.z; xs[4 * q + 3] = v.w;
        }
    } else {
#pragma unroll
        for (int q = 0; q < 12; q++) xs[q] = 0;
    }
}

// Sum N doubles per lane over the warp with the SAME pairing tree as a plain xor butterfly (16, 8, 4, 2, 1),
// but lanes split the values between them while there is more than one left: 8 values cost 9 double
// shuffles instead of 40.  On return lane L holds in v[0] the warp total of value index
// ((L>>4)&1)*4 + ((L>>3)&1)*2 + ((L>>2)&1) (for N == 8; N == 4 uses bits 4,3; N == 1 is the plain butterfly).
__device__ __forceinline__ double shfl_xor_f64(double v, int o) { return __shfl_xor_sync(0xFFFFFFFFu, v, o); }
template <int N>
__device__ __forceinline__ void warp_sum_split(double (&v)[N], int lane) {
    static_assert(N == 8 || N == 4 || N == 1, "power of two up to 8");
    int o = 16;
    if (N >= 8) {
        const bool up = lane & o;
#pragma unroll
        for (int i = 0; i < 4; i++) { const double send = up ? v[i] : v[i + 4], keep = up ? v[i + 4] : v[i]; v[i] = keep + shfl_xor_f64(send, o); }
        o >>= 1;
    }
    if (N >= 4) {
        const bool up = lane & o;
#pragma unroll
        for (int i = 0; i < 2; i++) { const double send = up ? v[i] : v[i + 2], keep = up ? v[i + 2] : v[i]; v[i] = keep + shfl_xor_f64(send, o); }
        o >>= 1;
        const bool up2 = lane & o;
        { const double send = up2 ? v[0] : v[1], keep = up2 ? v[1] : v[0]; v[0] = keep + shfl_xor_f64(send, o); }
        o >>= 1;
    }
    for (; o > 0; o >>= 1) v[0] += shfl_xor_f64(v[0], o);
}

// ------------------------------------------------------------------------------------------------ Rice search
// libFLAC's Rice parameter estimate and bit estimate for one partition (set_partitioned_rice_ with the
// 18-bit fixed-point mean): np samples, abs sum `sum`.
__device__ __forceinline__ void rice_estimate(unsigned long long sum, uint32_t np, uint32_t k_limit, uint32_t *k_out, uint32_t *bits_out) {
    const uint32_t div = 0x40000u / np;
    const unsigned long long t = sum < 2 ? 0ull : (((sum - 1) * div) >> 18);
    uint32_t k = t == 0 ? 0u : (uint32_t)ilog2_u64(t) + 1u;
    if (k >= k_limit) k = k_limit - 1;
    *k_out = k;
    *bits_out = rice_bits_estimate(k, np, sum);
}

struct SearchShared {
    unsigned long long fin[64];                 // |residual| sums of the finest partitions (order P)
    uint8_t params[64];                         // Rice parameters of the chosen order
    uint32_t rb, best_l;                        // estimated residual bits (incl. the 6 method/order bits), chosen level
};
__device__ __forceinline__ unsigned long long shfl_xor_u64(unsigned long long v, int o) { return __shfl_xor_sync(0xFFFFFFFFu, v, o); }

// sum over the warp of capped 32-bit values without overflow (two REDUX on 16-bit halves)
__device__ __forceinline__ unsigned long long warp_sum_u32(uint32_t lo16sum, uint32_t hi16sum) {
    return ((unsigned long long)__reduce_add_sync(0xFFFFFFFFu, hi16sum) << 16) + __reduce_add_sync(0xFFFFFFFFu, lo16sum);
}

// find_best_partition_order_ for one full block (n = 4096, 256 threads x 16 samples) in two parts.
// (1) finest_sums, all 256 threads: s64 = this thread's |residual| sum (warm-up samples excluded); tpp_log
//     xor-shuffle steps give the 2^P finest partition sums (P = 3..6), stored by the group leaders.
// (2) warp_search, ONE warp: lane i owns the finest pair (2i, 2i+1): levels 0 and 1 directly, levels >= 2
//     from an xor butterfly over the pair sums (the entry of level j >= 2 and group g is estimated by the
//     lane of that group with j-2 trailing one bits, so every lane estimates at most one of them); when the
//     pairs fill only half the warp (P <= 5) the upper half takes the second entry of each pair and the
//     levels >= 2, so the four estimates become two; per-level totals with REDUX, order choice, parameters.
// v2 estimated the in-warp levels in all eight warps and the upper levels redundantly in every warp (~330
// instructions in every thread): the search is ~5 % of the arithmetic of a subframe but was a third of its
// instructions (profiles/r01_ncu_enc_v4_*).
__device__ __forceinline__ void finest_sums(unsigned long long s64, uint32_t P, int tid, unsigned long long *fin) {
    const int lane = tid & 31;
    const uint32_t tpp_log = 8 - P;             // log2(threads per finest partition): 2..5
#pragma unroll
    for (int step = 0; step < 5; step++)
        if ((uint32_t)step < tpp_log) s64 += shfl_xor_u64(s64, 1 << step);
    if (((uint32_t)lane & ((1u << tpp_log) - 1u)) == 0) fin[(uint32_t)tid >> tpp_log] = s64;
}

__device__ __forceinline__ void warp_search(const unsigned long long *fin, uint32_t order, uint32_t P, uint32_t k_limit, int lane,
                                            uint8_t *params, uint32_t *rb_out, uint32_t *best_l_out) {
    constexpr uint32_t n = kMaxBlock;
    const uint32_t M = 1u << (P - 1);           // pairs of finest partitions: 4..32 lanes
    const bool act = (uint32_t)lane < M;
    const unsigned long long a = act ? fin[2 * lane] : 0ull, b = act ? fin[2 * lane + 1] : 0ull;
    // levels >= 2: butterfly over the pair sums; lane with t trailing ones takes level t + 2
    const uint32_t t1 = (uint32_t)__ffs(~lane) - 1u;       // trailing ones of the lane index (0..5)
    const uint32_t myl = t1 + 2;
    unsigned long long v = a + b, mine = 0;
#pragma unroll
    for (int step = 0; step < 5; step++) {
        v += shfl_xor_u64(v, 1 << step);
        if ((uint32_t)step == t1) mine = v;
    }
    const bool actd = act && myl <= P;
    const uint32_t np0 = n >> P, np1 = n >> (P - 1);
    uint32_t ka = 0, kb = 0, kc = 0, kd = 0, ba = 0, bb = 0, bc = 0, bd = 0;
    if (P <= 5) {
        // the upper half-warp mirrors lane - 16: first call (a | b), second call (pair sum | level >= 2)
        const int src = lane & 15;
        const bool hi = lane >= 16;
        const unsigned long long b_m = __shfl_sync(0xFFFFFFFFu, b, src), mine_m = __shfl_sync(0xFFFFFFFFu, mine, src);
        const uint32_t myl_m = __shfl_sync(0xFFFFFFFFu, myl, src);
        const bool act_m = (uint32_t)src < M, actd_m = act_m && myl_m <= P;
        uint32_t k1 = 0, b1 = 0, k2 = 0, b2 = 0;
        if (act_m) rice_estimate(hi ? b_m : a, (!hi && lane == 0) ? np0 - order : np0, k_limit, &k1, &b1);
        if (hi ? actd_m : act_m) {
            uint32_t np = hi ? (n >> (P - myl_m)) : np1;
            if (hi ? (((uint32_t)src >> (myl_m - 1)) == 0) : (lane == 0)) np -= order;
            rice_estimate(hi ? mine_m : a + b, np, k_limit, &k2, &b2);
        }
        // hand the mirrored results back to the owning lanes
        const uint32_t kb_u = __shfl_sync(0xFFFFFFFFu, k1, src + 16), bb_u = __shfl_sync(0xFFFFFFFFu, b1, src + 16);
        const uint32_t kd_u = __shfl_sync(0xFFFFFFFFu, k2, src + 16), bd_u = __shfl_sync(0xFFFFFFFFu, b2, src + 16);
        if (!hi) { ka = k1; ba = b1; kb = kb_u; bb = bb_u; kc = k2; bc = b2; kd = kd_u; bd = bd_u; }
    } else {
        if (act) {
            rice_estimate(a, lane == 0 ? np0 - order : np0, k_limit, &ka, &ba);
            rice_estimate(b, np0, k_limit, &kb, &bb);
            rice_estimate(a + b, lane == 0 ? np1 - order : np1, k_limit, &kc, &bc);
        }
        if (actd) {
            uint32_t np = n >> (P - myl);
            if (((uint32_t)lane >> (myl - 1)) == 0) np -= order;
            rice_estimate(mine, np, k_limit, &kd, &bd);
        }
    }
    // totals per level (each + 6 bits for method and order), strict improvement from the finest order downwards
    unsigned long long tot = warp_sum_u32((ba & 0xFFFFu) + (bb & 0xFFFFu), (ba >> 16) + (bb >> 16)) + 6;
    uint32_t rb = tot > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t)tot, best_l = 0;
    tot = warp_sum_u32(bc & 0xFFFFu, bc >> 16) + 6;
    { const uint32_t c = tot > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t)tot; if (c < rb) { rb = c; best_l = 1; } }
#pragma unroll
    for (int l = 2; l <= 6; l++) {
        if ((uint32_t)l <= P) {
            const uint32_t x = (actd && myl == (uint32_t)l) ? bd : 0u;
            tot = warp_sum_u32(x & 0xFFFFu, x >> 16) + 6;
            const uint32_t c = tot > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t)tot;
            if (c < rb) { rb = c; best_l = (uint32_t)l; }
        }
    }
    if (best_l == 0) { if (act) { params[2 * lane] = (uint8_t)ka; params[2 * lane + 1] = (uint8_t)kb; } }
    else if (best_l == 1) { if (act) params[lane] = (uint8_t)kc; }
    else if (actd && myl == best_l) params[(uint32_t)lane >> (myl - 1)] = (uint8_t)kd;
    *rb_out = rb; *best_l_out = best_l;
}

// ------------------------------------------------------------------------------------------------ autocorrelation
// One chunk = the 16 samples [16t, 16t + 16) of a block (k_enc_stats' thread t), at xs[12..27] with the 12 samples before
// them at xs[0..11] (zeros for t = 0).  Both statistics kernels form the windowed autocorrelation of a chunk with these
// helpers, so their fp64 partials are the same bits.

// full-length window for the chunk's samples and its HALO samples
template <int HALO>
__device__ __forceinline__ void load_window_chunk(const float *__restrict__ window, int t, float (&wv)[kSPT + HALO + 1]) {
    const float4 *wp = reinterpret_cast<const float4 *>(window + t * kSPT) - HALO / 4;
#pragma unroll
    for (int q = 0; q < (kSPT + HALO) / 4; q++) {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (t > 0 || q >= HALO / 4) v = __ldg(wp + q);
        wv[4 * q] = v.x; wv[4 * q + 1] = v.y; wv[4 * q + 2] = v.z; wv[4 * q + 3] = v.w;
    }
}

// windowed samples (libFLAC windows in single precision): the full window (set 0) ...
template <int HALO>
__device__ __forceinline__ void window_full(const int32_t (&xs)[28], const float (&wv)[kSPT + HALO + 1], float (&df)[kSPT + HALO]) {
    // chunk 0's halo samples are zero, so no range checks are needed
#pragma unroll
    for (int j = 0; j < kSPT + HALO; j++) df[j] = __fmul_rn((float)xs[12 - HALO + j], wv[j]);
}
// ... and a subdivide_tukey part: window[0, part) and its last `part` values around a flat top, over [wshift, wshift + wlen)
template <int HALO>
__device__ __forceinline__ void window_part(const int32_t (&xs)[28], uint32_t i0, uint32_t wshift, uint32_t wlen, uint32_t part,
                                            const float *__restrict__ window, float (&df)[kSPT + HALO]) {
    constexpr uint32_t n = kMaxBlock;
#pragma unroll
    for (int j = 0; j < kSPT + HALO; j++) {
        const int idx = (int)i0 - HALO + j;
        float v = 0.0f;
        if (idx >= (int)wshift && (uint32_t)idx < wshift + wlen) {
            const uint32_t local = (uint32_t)idx - wshift;
            float w1;
            if (local < part) w1 = __ldg(window + local);
            else if (local < 2 * part) w1 = __ldg(window + (n - 2 * part + local));
            else w1 = 0.0f;
            v = __fmul_rn((float)xs[12 - HALO + j], w1);
        }
        df[j] = v;
    }
}

// the chunk's partial autocorrelation: sliding window of the last NLAGS samples in double (one conversion per sample, few
// live registers), one FMA chain per lag from ac[] (the callers start it at 0.0)
template <int NLAGS>
__device__ __forceinline__ void autoc_fma(const float (&df)[kSPT + NLAGS - 1], double (&ac)[NLAGS]) {
    constexpr int HALO = NLAGS - 1;
    double win[NLAGS];
#pragma unroll
    for (int l = 1; l < NLAGS; l++) win[l] = (double)df[HALO - l];
#pragma unroll
    for (int s = 0; s < kSPT; s++) {
        if (s > 0) {
#pragma unroll
            for (int l = NLAGS - 1; l >= 1; l--) win[l] = win[l - 1];
        }
        win[0] = (double)df[HALO + s];
#pragma unroll
        for (int l = 0; l < NLAGS; l++) ac[l] = fma(win[0], win[l], ac[l]);
    }
}

// Warp totals of the 32 lanes' partials (same pairing tree as an xor butterfly per lag): lags 0-7 split over the lanes (lag
// autoc_lag8(lane) in g8, complete in the lanes with lane % 4 == 0), lag 8 in every lane (g1), lags 9-12 when NLAGS == 13
// (lag autoc_lag4(lane) in g4, complete in the lanes with lane % 8 == 0).
__device__ __forceinline__ int autoc_lag8(int lane) { return ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1); }
__device__ __forceinline__ int autoc_lag4(int lane) { return 9 + ((lane >> 4) & 1) * 2 + ((lane >> 3) & 1); }
template <int NLAGS>
__device__ __forceinline__ void autoc_warp_sums(const double (&ac)[NLAGS], int lane, double &g8, double &g1, double &g4) {
    double v8[8];
#pragma unroll
    for (int l = 0; l < 8; l++) v8[l] = ac[l];
    warp_sum_split<8>(v8, lane);
    double v1[1] = {ac[8]};
    warp_sum_split<1>(v1, lane);
    g8 = v8[0]; g1 = v1[0]; g4 = 0.0;
    if constexpr (NLAGS > 9) {
        double v4[4];
#pragma unroll
        for (int l = 0; l < 4; l++) v4[l] = ac[9 + l];
        warp_sum_split<4>(v4, lane);
        g4 = v4[0];
    }
}

// libFLAC's "bits per sample" estimate of the guessed FIXED order (FLAC__fixed_compute_best_predictor); the FIXED candidate
// is not tried when it reaches the subframe's bps
__device__ __forceinline__ float fixed_bits_estimate(unsigned long long eg) {
    constexpr uint32_t n = kMaxBlock;
    return (float)(eg > 0 ? log(0.69314718055994530942 * (double)eg / (double)(n - 4)) / 0.69314718055994530942 : 0.0);
}

// ------------------------------------------------------------------------------------------------ stats
struct StatsShared {
    uint32_t orv[8], diff[8];
    unsigned long long e[8][5];
    double ac[8][kLags];
};

#ifndef FRB_STATS_MINB
#define FRB_STATS_MINB 4
#endif
#ifndef FRB_CODE_MINB
#define FRB_CODE_MINB 4
#endif
#ifndef FRB_CODE_RELOAD
#define FRB_CODE_RELOAD 1
#endif
#ifndef FRB_STATS_LATEWIN
#define FRB_STATS_LATEWIN 0
#endif
#ifndef FRB_STATS_RELOAD
#define FRB_STATS_RELOAD 1
#endif
template <bool WIDE, int NLAGS>
__global__ void __launch_bounds__(kEncThreads, (NLAGS > 9 || WIDE) ? 2 : FRB_STATS_MINB)
k_enc_stats(const FrameDesc *__restrict__ frames, uint32_t channels, uint32_t bps_stream,
            uint32_t windows, uint32_t max_po_cfg, const EncSrc audio,
            const float *__restrict__ window, EncSubStats *__restrict__ stats, double *__restrict__ autoc_out,
            unsigned long long *__restrict__ fx_fin, uint32_t c0, uint32_t side_extra) {
    // c0 / side_extra: channel offset of this launch and 1 when its subframes carry one more bit than the stream (the
    // side channel of a two-channel stream, see frb_encode_analyse); bps_stream stays the STREAM's value
    __shared__ StatsShared S;
    const uint32_t cch = blockIdx.y + c0, sbps = bps_stream + side_extra;
    const uint32_t task = blockIdx.x * channels + cch;
    const TaskLoc L = locate_task(frames, audio, blockIdx.x, cch);
    if (!fast_eligible(L)) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr uint32_t n = kMaxBlock;
    constexpr int HALO = NLAGS > 0 ? NLAGS - 1 : 0;         // 8 or 12: multiples of 4, so the window reads stay 16-byte aligned
    int32_t xs[28];
    load_samples28(L, tid, xs);
    // full-length window for this thread's samples and halo
    float wv[kSPT + HALO + 1];
    auto load_window = [&]() {
        if constexpr (NLAGS > 0) load_window_chunk<HALO>(window, tid, wv);
    };
#if !FRB_STATS_LATEWIN
    load_window();          // fetched together with the samples
#endif
    // ---- wasted bits / constant ----
    uint32_t orv = 0, diff = 0;
    const int32_t x_first = sample_at(L, 0);
#pragma unroll
    for (int s = 0; s < kSPT; s++) { orv |= (uint32_t)xs[12 + s]; diff |= (uint32_t)(xs[12 + s] ^ x_first); }
    orv = __reduce_or_sync(0xFFFFFFFFu, orv);
    diff = __reduce_or_sync(0xFFFFFFFFu, diff);
    if (lane == 0) { S.orv[warp] = orv; S.diff[warp] = diff; }
    __syncthreads();
    orv = 0; diff = 0;
#pragma unroll
    for (int w = 0; w < 8; w++) { orv |= S.orv[w]; diff |= S.diff[w]; }
    uint32_t wasted = orv ? (uint32_t)(__ffs((int)orv) - 1) : 0;
    if (wasted > sbps) wasted = sbps;
    if (wasted) {
#pragma unroll
        for (int j = 0; j < 28; j++) xs[j] >>= wasted;
    }
    // ---- fixed predictor abs-error sums over i in [4, n) (libFLAC's order guess) and, for thread 0, the extra
    // terms i in [q, 4) that belong to the order-q residual but not to the guess statistic ----
    unsigned long long e[5], pe[5];           // warp-reduced / per-thread
    uint32_t fx_badmask = 0;                  // WIDE: bit q set if an order-q residual of this thread does not fit int32
    if (!WIDE) {
        // successive differences in 32 bits: |4th difference| <= 16 * 2^15, 16 samples per thread, 32 per warp
        uint32_t e32[5] = {0, 0, 0, 0, 0}, x32[4] = {0, 0, 0, 0};
        // |d| accumulates with one VABSDIFF (|a - b| + c); the 4th difference is never materialised
        int32_t d1[kSPT + 3], d2[kSPT + 2], d3[kSPT + 1];
#pragma unroll
        for (int j = 0; j < kSPT + 3; j++) d1[j] = xs[9 + j] - xs[8 + j];
#pragma unroll
        for (int j = 0; j < kSPT + 2; j++) d2[j] = d1[j + 1] - d1[j];
#pragma unroll
        for (int j = 0; j < kSPT + 1; j++) d3[j] = d2[j + 1] - d2[j];
#pragma unroll
        for (int s = 0; s < kSPT; s++) {
            if (s >= 4 || tid > 0) {
                e32[0] = __sad(xs[12 + s], 0, e32[0]); e32[1] = __sad(xs[12 + s], xs[11 + s], e32[1]);
                e32[2] = __sad(d1[s + 3], d1[s + 2], e32[2]); e32[3] = __sad(d2[s + 2], d2[s + 1], e32[3]);
                e32[4] = __sad(d3[s + 1], d3[s], e32[4]);
            } else {
                x32[0] = __sad(xs[12 + s], 0, x32[0]);
                if (s >= 1) x32[1] = __sad(xs[12 + s], xs[11 + s], x32[1]);
                if (s >= 2) x32[2] = __sad(d1[s + 3], d1[s + 2], x32[2]);
                if (s >= 3) x32[3] = __sad(d2[s + 2], d2[s + 1], x32[3]);
            }
        }
#pragma unroll
        for (int q = 0; q < 5; q++) { pe[q] = e32[q] + (q < 4 ? x32[q < 4 ? q : 0] : 0u); e[q] = __reduce_add_sync(0xFFFFFFFFu, e32[q]); }
    } else {
        unsigned long long xe[4] = {0, 0, 0, 0};
#pragma unroll
        for (int q = 0; q < 5; q++) e[q] = 0;
#pragma unroll
        for (int s = 0; s < kSPT; s++) {
            const long long a = xs[12 + s], b = xs[11 + s], cc = xs[10 + s], d = xs[9 + s], ee = xs[8 + s];
            const long long r0 = a, r1 = a - b, r2 = a - 2 * b + cc, r3 = a - 3 * b + 3 * cc - d, r4 = a - 4 * b + 6 * cc - 4 * d + ee;
            const unsigned long long a0 = (unsigned long long)(r0 < 0 ? -r0 : r0), a1 = (unsigned long long)(r1 < 0 ? -r1 : r1),
                                     a2 = (unsigned long long)(r2 < 0 ? -r2 : r2), a3 = (unsigned long long)(r3 < 0 ? -r3 : r3),
                                     a4 = (unsigned long long)(r4 < 0 ? -r4 : r4);
            if (s >= 4 || tid > 0) {
                e[0] += a0; e[1] += a1; e[2] += a2; e[3] += a3; e[4] += a4;
                // residual must satisfy INT32_MIN < r <= INT32_MAX (the oracle's / libFLAC's limit)
                fx_badmask |= (r0 > 2147483647ll || r0 <= -2147483648ll) ? 1u : 0u;
                fx_badmask |= (r1 > 2147483647ll || r1 <= -2147483648ll) ? 2u : 0u;
                fx_badmask |= (r2 > 2147483647ll || r2 <= -2147483648ll) ? 4u : 0u;
                fx_badmask |= (r3 > 2147483647ll || r3 <= -2147483648ll) ? 8u : 0u;
                fx_badmask |= (r4 > 2147483647ll || r4 <= -2147483648ll) ? 16u : 0u;
            } else {
                xe[0] += a0; fx_badmask |= (r0 > 2147483647ll || r0 <= -2147483648ll) ? 1u : 0u;
                if (s >= 1) { xe[1] += a1; fx_badmask |= (r1 > 2147483647ll || r1 <= -2147483648ll) ? 2u : 0u; }
                if (s >= 2) { xe[2] += a2; fx_badmask |= (r2 > 2147483647ll || r2 <= -2147483648ll) ? 4u : 0u; }
                if (s >= 3) { xe[3] += a3; fx_badmask |= (r3 > 2147483647ll || r3 <= -2147483648ll) ? 8u : 0u; }
            }
        }
#pragma unroll
        for (int q = 0; q < 5; q++) pe[q] = e[q] + (q < 4 ? xe[q < 4 ? q : 0] : 0ull);
#pragma unroll
        for (int q = 0; q < 5; q++)
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) e[q] += __shfl_xor_sync(0xFFFFFFFFu, e[q], o);
    }
    if (lane == 0)
#pragma unroll
        for (int q = 0; q < 5; q++) S.e[warp][q] = e[q];
    if (tid == 6) stats[task].fx_bad = 0;
    __syncthreads();
    // every warp totals the five sums on its own (lanes 0..4) and broadcasts them: no further barrier
    unsigned long long et = 0;
    if (lane < 5) {
#pragma unroll
        for (int w = 0; w < 8; w++) et += S.e[w][lane];
    }
#pragma unroll
    for (int q = 0; q < 5; q++) e[q] = __shfl_sync(0xFFFFFFFFu, et, q);
    if (tid < 5) stats[task].e[tid] = et;
    uint32_t flags = diff == 0 ? 1u : 0u;
    if (diff != 0) {
        // ---- FIXED candidate: libFLAC's order guess; the per-thread |residual| sums of that order are already in
        // registers, so only the finest partition sums are stored and k_enc_fixed (one warp per subframe) runs the
        // Rice search: no residual pass and no idle warps for it ----
        uint32_t guess;
        const unsigned long long m1234 = min(min(e[1], e[2]), min(e[3], e[4]));
        const unsigned long long m234 = min(e[2], min(e[3], e[4]));
        const unsigned long long m34 = min(e[3], e[4]);
        if (e[0] <= m1234) guess = 0; else if (e[1] <= m234) guess = 1; else if (e[2] <= m34) guess = 2; else if (e[3] <= e[4]) guess = 3; else guess = 4;
        const unsigned long long ps = guess == 0 ? pe[0] : guess == 1 ? pe[1] : guess == 2 ? pe[2] : guess == 3 ? pe[3] : pe[4];
        finest_sums(ps, max_po_cfg, tid, fx_fin + (size_t)task * 64);
        if (WIDE && ((fx_badmask >> guess) & 1u)) atomicOr(&stats[task].fx_bad, 1u);
        if (tid == 6) stats[task].fx_order = guess;
        flags |= 2u;
    }
    if (tid == 5) { stats[task].wasted = wasted; stats[task].flags = flags; }
    if (diff == 0) return;
    if constexpr (NLAGS > 0) {
    // ---- windowed autocorrelation, one set per apodization (root, halves, thirds) ----
#if FRB_STATS_LATEWIN
    // the window (16 KB, shared by every CTA: L1 hits) and, with FRB_STATS_RELOAD, the samples are fetched only now: the
    // fixed-predictor phase above and this one no longer hold each other's registers
    load_window();
#endif
    const uint32_t i0 = tid * kSPT;
    const int32_t (&xs0)[28] = xs;
    int set = 0;
    for (uint32_t b = 1; b <= windows; b++) {
        const uint32_t nsub = (b == 1) ? 1u : b;
        for (uint32_t sub = 0; sub < nsub; sub++, set++) {
            uint32_t wshift = 0, wlen = n, part = 0;
            if (b > 1) { part = n / b / 2; wshift = (sub * n) / b; wlen = n / b; }
            double ac[NLAGS];
#pragma unroll
            for (int l = 0; l < NLAGS; l++) ac[l] = 0.0;
            // threads whose 16 samples lie outside the window contribute nothing
            if (i0 + kSPT > wshift && i0 < wshift + wlen) {
                float df[kSPT + HALO];
                // 16-bit kernels at the 64-register cap: the samples are fetched again per window set (L1 hits) so that they
                // are dead once df[] is formed, instead of staying in 28 registers next to the fp64 window and accumulators
                // for the next set.  (The 64-bit / 13-lag instantiations run at 128 registers and keep them: reloading
                // there only adds work, C4 24.7 against 23.5 ms.)
                constexpr bool RELOAD = FRB_STATS_RELOAD != 0 && !WIDE && NLAGS <= 9;
                int32_t xr[28];
                if constexpr (RELOAD) {
                    load_samples28(L, tid, xr);
                    if (wasted) {
#pragma unroll
                        for (int j = 0; j < 28; j++) xr[j] >>= wasted;
                    }
                }
                const int32_t (&xs)[28] = pick_ref<RELOAD>(xr, xs0);
                if (b == 1) window_full<HALO>(xs, wv, df);
                else window_part<HALO>(xs, i0, wshift, wlen, part, window, df);
                autoc_fma<NLAGS>(df, ac);
            }
            double g8, g1, g4;
            autoc_warp_sums<NLAGS>(ac, lane, g8, g1, g4);
            __syncthreads();                          // previous set's S.ac has been consumed
            if ((lane & 3) == 0) S.ac[warp][autoc_lag8(lane)] = g8;
            if (lane == 0) S.ac[warp][8] = g1;
            if (NLAGS > 9 && (lane & 7) == 0) S.ac[warp][autoc_lag4(lane)] = g4;
            __syncthreads();
            if (tid < NLAGS) {
                double s = 0.0;
#pragma unroll
                for (int w = 0; w < 8; w++) s += S.ac[w][tid];
                autoc_out[((size_t)task * kMaxSets + set) * kLags + tid] = s;
            }
        }
    }
    }
}

// ------------------------------------------------------------------------------------------------ fixed search
// One warp per subframe: libFLAC's "is FIXED worth trying" estimate and the Rice search of the FIXED candidate
// from the finest partition sums k_enc_stats stored.  Runs over channels [c0, c0 + nch) of every frame (the subframes
// k_enc_stats analysed; k_enc_stats_warp searches its own).
__global__ void __launch_bounds__(128)
k_enc_fixed(const FrameDesc *__restrict__ frames, uint32_t channels, uint32_t c0, uint32_t nch, uint32_t bps_stream, uint32_t max_po_cfg,
            uint32_t total, const EncSrc audio, EncSubStats *__restrict__ stats, const unsigned long long *__restrict__ fx_fin,
            uint32_t side_ch) {
    const int lane = threadIdx.x & 31;
    const uint32_t g = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (g >= total) return;
    const uint32_t f = g / nch, ch = c0 + (g - f * nch), task = f * channels + ch;
    const TaskLoc L = locate_task(frames, audio, f, ch);
    if (!fast_eligible(L)) return;
    EncSubStats *st = stats + task;
    const uint32_t flags = st->flags;
    if (!(flags & 2u)) return;
    const uint32_t wasted = st->wasted, guess = st->fx_order;
    const uint32_t bps = bps_stream + (ch == side_ch ? 1u : 0u) - wasted;
    // FLAC__fixed_compute_best_predictor's estimate for the guessed order; >= bps means "do not even try"
    const unsigned long long eg = st->e[guess];
    if (fixed_bits_estimate(eg) >= (float)bps || st->fx_bad) {
        __syncwarp();
        if (lane == 0) st->flags = flags & ~2u;
        return;
    }
    uint32_t rb, best_l;
    warp_search(fx_fin + (size_t)task * 64, guess, max_po_cfg, bps_stream > 16 ? 31u : 15u, lane, st->fx_params, &rb, &best_l);
    if (lane == 0) { st->fx_bits = 8 + wasted + guess * bps + rb; st->fx_po = max_po_cfg - best_l; }
}

// ------------------------------------------------------------------------------------------------ stats, warp per subframe
// k_enc_stats and k_enc_fixed for a 16-bit subframe (!WIDE) in ONE warp, with no CTA barrier: lane l walks chunks j = 0..7,
// chunk (j, l) being the 16 samples of k_enc_stats' thread t = 32j + l, with the same halo and window values, so every
// partial sum is the one that thread formed.
//  * one pass over the samples gives the OR / XOR for wasted bits and constant, the fixed-predictor sums and the root
//    window's autocorrelation, all from the UNSHIFTED samples; the wasted-bits shift is applied afterwards, exactly:
//    every sample is a multiple of 2^w, so a |residual| sum shifts right by w without remainder, and in the window product,
//    the fp64 FMA chain and the sums every value scales by a power of two with no rounding change (no value comes near
//    the subnormal range), so the root set times 2^-2w is the same bits as k_enc_stats' result from shifted samples;
//  * the per-chunk warp totals of the autocorrelation (warp_sum_split, as k_enc_stats) go into a running total per lag in
//    chunk order from 0.0: k_enc_stats' cross-warp sum over its 8 warps, the same additions in the same order;
//  * the five per-chunk |residual| sums go to shared memory, so the guessed order's finest partition sums (64..512
//    samples = 4..32 chunks) need no second pass, and the FIXED candidate's Rice search (warp_search) runs here.
// The subdivide_tukey sets (levels 6-8) take one more pass each over the chunk rows they overlap, from shifted samples.
struct StatsWarpShared {
    uint32_t ch[5][kEncThreads];            // |order-q residual| sum of chunk t = 32j + lane (unshifted samples)
    unsigned long long fin[64];             // finest partition sums of the guessed order
};
constexpr int kStatsWarps = 4;              // warps (subframes) per CTA

#ifndef FRB_STATS_WARP_MINB
#define FRB_STATS_WARP_MINB 6
#endif
template <int NLAGS>
__global__ void __launch_bounds__(kStatsWarps * 32, FRB_STATS_WARP_MINB)
k_enc_stats_warp(const FrameDesc *__restrict__ frames, uint32_t channels, uint32_t nch, uint32_t total, uint32_t bps_stream,
                 uint32_t windows, uint32_t max_po_cfg, const EncSrc audio, const float *__restrict__ window,
                 EncSubStats *__restrict__ stats, double *__restrict__ autoc_out) {
    // subframe g of this launch: frame g / nch, channel g % nch (channels [0, nch) of every frame)
    __shared__ __align__(16) StatsWarpShared Sh[kStatsWarps];
    const int lane = threadIdx.x & 31;
    const uint32_t g = blockIdx.x * kStatsWarps + (threadIdx.x >> 5);
    if (g >= total) return;
    const uint32_t f = g / nch, ch = g - f * nch, task = f * channels + ch;
    const TaskLoc L = locate_task(frames, audio, f, ch);
    if (!fast_eligible(L)) return;
    StatsWarpShared &S = Sh[threadIdx.x >> 5];
    constexpr uint32_t n = kMaxBlock;
    constexpr int HALO = NLAGS > 0 ? NLAGS - 1 : 0;
    constexpr int NL = NLAGS > 0 ? NLAGS : 1;
    const int32_t x_first = sample_at(L, 0);
    uint32_t orv = 0, diff = 0, e32[5] = {0, 0, 0, 0, 0};
    double r8 = 0.0, r1 = 0.0, r4 = 0.0;    // running totals of the root set: lag autoc_lag8(lane), lag 8, lag autoc_lag4(lane)
#pragma unroll 1
    for (int j = 0; j < 8; j++) {
        const int t = 32 * j + lane;
        int32_t xs[28];
        load_samples28(L, t, xs);
        float wv[kSPT + HALO + 1];
        if constexpr (NLAGS > 0) load_window_chunk<HALO>(window, t, wv);
        // fixed-predictor |residual| sums over all 16 samples (chunk 0's zero halo is corrected below); |4th difference|
        // <= 16 * 2^15, so a lane's 128 samples and the warp's 4096 fit 32 bits
        uint32_t c32[5] = {0, 0, 0, 0, 0};
        int32_t d1[kSPT + 3], d2[kSPT + 2], d3[kSPT + 1];
#pragma unroll
        for (int k = 0; k < kSPT + 3; k++) d1[k] = xs[9 + k] - xs[8 + k];
#pragma unroll
        for (int k = 0; k < kSPT + 2; k++) d2[k] = d1[k + 1] - d1[k];
#pragma unroll
        for (int k = 0; k < kSPT + 1; k++) d3[k] = d2[k + 1] - d2[k];
#pragma unroll
        for (int s = 0; s < kSPT; s++) {
            orv |= (uint32_t)xs[12 + s]; diff |= (uint32_t)(xs[12 + s] ^ x_first);
            c32[0] = __sad(xs[12 + s], 0, c32[0]); c32[1] = __sad(xs[12 + s], xs[11 + s], c32[1]);
            c32[2] = __sad(d1[s + 3], d1[s + 2], c32[2]); c32[3] = __sad(d2[s + 2], d2[s + 1], c32[3]);
            c32[4] = __sad(d3[s + 1], d3[s], c32[4]);
        }
#pragma unroll
        for (int q = 0; q < 5; q++) { S.ch[q][t] = c32[q]; e32[q] += c32[q]; }
        if constexpr (NLAGS > 0) {
            float df[kSPT + HALO];
            window_full<HALO>(xs, wv, df);
            double ac[NL];
#pragma unroll
            for (int l = 0; l < NLAGS; l++) ac[l] = 0.0;
            autoc_fma<NLAGS>(df, ac);
            double g8, g1, g4;
            autoc_warp_sums<NLAGS>(ac, lane, g8, g1, g4);
            r8 += g8; r1 += g1;
            if (NLAGS > 9) r4 += g4;
        }
    }
    orv = __reduce_or_sync(0xFFFFFFFFu, orv);
    diff = __reduce_or_sync(0xFFFFFFFFu, diff);
    uint32_t wasted = orv ? (uint32_t)(__ffs((int)orv) - 1) : 0;
    if (wasted > bps_stream) wasted = bps_stream;
    if (lane == 0) {
        // chunk 0 summed its first 4 samples against a zero history: those terms are not part of the order guess's
        // statistic (i in [4, n)), and the terms i < q are not part of the order-q residual
        int32_t r[4] = {x_first, sample_at(L, 1), sample_at(L, 2), sample_at(L, 3)};
#pragma unroll
        for (int q = 0; q < 5; q++) {
            uint32_t all = 0, pre = 0;
#pragma unroll
            for (int s = 0; s < 4; s++) { const uint32_t u = __sad(r[s], 0, 0u); all += u; if (s < q) pre += u; }
            e32[q] -= all;
            S.ch[q][0] -= pre;
#pragma unroll
            for (int s = 3; s >= 1; s--) r[s] -= r[s - 1];          // next order's residual, zero history
        }
    }
    unsigned long long e[5];
#pragma unroll
    for (int q = 0; q < 5; q++) e[q] = __reduce_add_sync(0xFFFFFFFFu, e32[q]) >> wasted;
    EncSubStats *st = stats + task;
    if (lane < 5) st->e[lane] = lane == 0 ? e[0] : lane == 1 ? e[1] : lane == 2 ? e[2] : lane == 3 ? e[3] : e[4];
    uint32_t flags = diff == 0 ? 1u : 0u;
    if (diff != 0) {
        // ---- FIXED candidate: libFLAC's order guess, its "worth trying" estimate and the Rice search (k_enc_fixed) ----
        uint32_t guess;
        const unsigned long long m1234 = min(min(e[1], e[2]), min(e[3], e[4]));
        const unsigned long long m234 = min(e[2], min(e[3], e[4]));
        const unsigned long long m34 = min(e[3], e[4]);
        if (e[0] <= m1234) guess = 0; else if (e[1] <= m234) guess = 1; else if (e[2] <= m34) guess = 2; else if (e[3] <= e[4]) guess = 3; else guess = 4;
        const uint32_t bps = bps_stream - wasted;
        const unsigned long long eg = guess == 0 ? e[0] : guess == 1 ? e[1] : guess == 2 ? e[2] : guess == 3 ? e[3] : e[4];
        if (!(fixed_bits_estimate(eg) >= (float)bps)) {
            __syncwarp();
            // lane l sums chunks [8l, 8l + 8) in two halves; finest partitions are 2^(8 - P) chunks
            const uint4 u = *reinterpret_cast<const uint4 *>(&S.ch[guess][8 * lane]);
            const uint4 v = *reinterpret_cast<const uint4 *>(&S.ch[guess][8 * lane + 4]);
            const uint32_t a = (u.x + u.y + u.z + u.w) >> wasted, b = (v.x + v.y + v.z + v.w) >> wasted;
            if (max_po_cfg == 6) { S.fin[2 * lane] = a; S.fin[2 * lane + 1] = b; }
            else {
                const uint32_t lg = 5 - max_po_cfg;                  // octets per finest partition: 2^0..2^2
                uint32_t p = a + b;
#pragma unroll
                for (int step = 0; step < 2; step++)
                    if ((uint32_t)step < lg) p += __shfl_xor_sync(0xFFFFFFFFu, p, 1 << step);
                if (((uint32_t)lane & ((1u << lg) - 1u)) == 0) S.fin[(uint32_t)lane >> lg] = p;
            }
            __syncwarp();
            uint32_t rb, best_l;
            warp_search(S.fin, guess, max_po_cfg, bps_stream > 16 ? 31u : 15u, lane, st->fx_params, &rb, &best_l);
            if (lane == 0) { st->fx_bits = 8 + wasted + guess * bps + rb; st->fx_po = max_po_cfg - best_l; }
            flags |= 2u;
        }
        if (lane == 0) st->fx_order = guess;
    }
    if (lane == 0) { st->wasted = wasted; st->flags = flags; st->fx_bad = 0; }
    if constexpr (NLAGS > 0) {
        if (diff == 0) return;
        const double sc = ldexp(1.0, -2 * (int)wasted);
        double *out = autoc_out + (size_t)task * kMaxSets * kLags;
        if ((lane & 3) == 0) out[autoc_lag8(lane)] = r8 * sc;
        if (lane == 0) out[8] = r1 * sc;
        if (NLAGS > 9 && (lane & 7) == 0) out[autoc_lag4(lane)] = r4 * sc;
        // ---- subdivide_tukey sets: halves (b = 2), thirds (b = 3) ----
        int set = 1;
        for (uint32_t b = 2; b <= windows; b++) {
            for (uint32_t sub = 0; sub < b; sub++, set++) {
                const uint32_t part = n / b / 2, wshift = (sub * n) / b, wlen = n / b;
                r8 = 0.0; r1 = 0.0; r4 = 0.0;
#pragma unroll 1
                for (int j = 0; j < 8; j++) {
                    // a row of chunks wholly outside the window adds +0.0 to every running total (never -0.0): skipped
                    if (!(512u * j + 512u > wshift && 512u * j < wshift + wlen)) continue;
                    const int t = 32 * j + lane;
                    const uint32_t i0 = (uint32_t)t * kSPT;
                    double ac[NL];
#pragma unroll
                    for (int l = 0; l < NLAGS; l++) ac[l] = 0.0;
                    if (i0 + kSPT > wshift && i0 < wshift + wlen) {
                        int32_t xs[28];
                        load_samples28(L, t, xs);
                        if (wasted) {
#pragma unroll
                            for (int k = 0; k < 28; k++) xs[k] >>= wasted;
                        }
                        float df[kSPT + HALO];
                        window_part<HALO>(xs, i0, wshift, wlen, part, window, df);
                        autoc_fma<NLAGS>(df, ac);
                    }
                    double g8, g1, g4;
                    autoc_warp_sums<NLAGS>(ac, lane, g8, g1, g4);
                    r8 += g8; r1 += g1;
                    if (NLAGS > 9) r4 += g4;
                }
                double *o = autoc_out + ((size_t)task * kMaxSets + set) * kLags;
                if ((lane & 3) == 0) o[autoc_lag8(lane)] = r8;
                if (lane == 0) o[8] = r1;
                if (NLAGS > 9 && (lane & 7) == 0) o[autoc_lag4(lane)] = r4;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------ model
// Levinson-Durbin with fully static indexing (registers): runs the recursion up to `upto` orders and
// returns the number of orders actually computed (stops early when the error reaches zero).
template <int MAXO>
__device__ __forceinline__ uint32_t levinson_static(const double (&autoc)[MAXO + 1], uint32_t upto, double (&lpc)[MAXO],
                                                    double (&lp_err)[MAXO]) {
    double err = autoc[0];
    uint32_t mo = upto;
    bool done = false;
#pragma unroll
    for (int i = 0; i < MAXO; i++) {
        if (!done && (uint32_t)i < upto) {
            double r = -autoc[i + 1];
#pragma unroll
            for (int j = 0; j < i; j++) r = __dsub_rn(r, __dmul_rn(lpc[j], autoc[i - j]));
            r = __ddiv_rn(r, err);
            lpc[i] = r;
#pragma unroll
            for (int j = 0; j < (i >> 1); j++) {
                const double tmp = lpc[j];
                lpc[j] = __dadd_rn(lpc[j], __dmul_rn(r, lpc[i - 1 - j]));
                lpc[i - 1 - j] = __dadd_rn(lpc[i - 1 - j], __dmul_rn(r, tmp));
            }
            if (i & 1) lpc[i >> 1] = __dadd_rn(lpc[i >> 1], __dmul_rn(lpc[i >> 1], r));
            err = __dmul_rn(err, __dsub_rn(1.0, __dmul_rn(r, r)));
            lp_err[i] = err;
            if (err == 0.0) { mo = i + 1; done = true; }
        }
    }
    return mo;
}

template <int MAXO>
__device__ __forceinline__ void model_one(const double (&autoc)[MAXO + 1], uint32_t max_lpc, uint32_t n, uint32_t bps,
                                          uint32_t qprec_cfg, EncCand &C) {
    C.type = 0;
    if (autoc[0] == 0.0) return;
    double lpc[MAXO], lp_err[MAXO];
#pragma unroll
    for (int j = 0; j < MAXO; j++) { lpc[j] = 0.0; lp_err[j] = 0.0; }
    const uint32_t mo = levinson_static<MAXO>(autoc, max_lpc, lpc, lp_err);
    // FLAC__lpc_compute_best_order and the "don't even try" estimate
    uint32_t best_i = 0;
    double best_b = 4294967295.0, best_eb2 = 0.0;
#pragma unroll
    for (int i = 0; i < MAXO; i++) {
        if ((uint32_t)i < mo) {
            const double le = lp_err[i];
            const uint32_t ord = (uint32_t)i + 1;
            const double scale = 0.5 / (double)n, scale2 = 0.5 / (double)(n - ord);
            double eb, eb2;
            if (le > 0.0) {
                eb = 0.5 * log(scale * le) / 0.69314718055994530942; if (eb < 0.0) eb = 0.0;
                eb2 = 0.5 * log(scale2 * le) / 0.69314718055994530942; if (eb2 < 0.0) eb2 = 0.0;
            } else if (le < 0.0) { eb = 1e32; eb2 = 1e32; } else { eb = 0.0; eb2 = 0.0; }
            const double bits = eb * (double)(n - ord) + (double)(ord * (bps + qprec_cfg));
            if (bits < best_b) { best_b = bits; best_i = (uint32_t)i; best_eb2 = eb2; }
        }
    }
    if (mo == 0) return;
    const uint32_t order = best_i + 1;
    if (best_eb2 >= (double)bps) return;
    uint32_t prec = qprec_cfg;
    if (bps <= 17) { const uint32_t lim = 32 - bps - (uint32_t)ilog2_u32(order); if (lim < prec) prec = lim; }
    // coefficients of the chosen order: rerun the (deterministic) recursion up to it
#pragma unroll
    for (int j = 0; j < MAXO; j++) lpc[j] = 0.0;
    (void)levinson_static<MAXO>(autoc, order, lpc, lp_err);
    float lpv[MAXO];
#pragma unroll
    for (int j = 0; j < MAXO; j++) lpv[j] = (float)(-lpc[j]);
    // FLAC__lpc_quantize_coefficients
    const int p1 = (int)prec - 1;
    const int qmax = (1 << p1) - 1, qmin = -(1 << p1);
    double cmax = 0.0;
#pragma unroll
    for (int i = 0; i < MAXO; i++) if ((uint32_t)i < order) { const double d = fabs((double)lpv[i]); if (d > cmax) cmax = d; }
    if (!(cmax > 0.0)) return;
    int log2cmax; (void)frexp(cmax, &log2cmax); log2cmax--;
    int sh = p1 - log2cmax - 1;
    if (sh > 15) sh = 15; else if (sh < -16) return;
#pragma unroll
    for (int j = 0; j < kMaxOrd; j++) C.coefs[j] = 0;
    double er = 0.0;
    if (sh >= 0) {
#pragma unroll
        for (int i = 0; i < MAXO; i++) if ((uint32_t)i < order) {
            er = __dadd_rn(er, __dmul_rn((double)lpv[i], (double)(1 << sh)));
            long long q = llround(er);
            if (q > qmax) q = qmax; else if (q < qmin) q = qmin;
            er = __dsub_rn(er, (double)q); C.coefs[i] = (int32_t)q;
        }
    } else {
        const int ns = -sh;
#pragma unroll
        for (int i = 0; i < MAXO; i++) if ((uint32_t)i < order) {
            er = __dadd_rn(er, __ddiv_rn((double)lpv[i], (double)(1 << ns)));
            long long q = llround(er);
            if (q > qmax) q = qmax; else if (q < qmin) q = qmin;
            er = __dsub_rn(er, (double)q); C.coefs[i] = (int32_t)q;
        }
        sh = 0;
    }
    C.type = 3; C.order = (int)order; C.precision = (int)prec; C.shift = sh;
}

// thread per (subframe, LPC candidate slot), slots in libFLAC's evaluation order
// (b = 1: full window; b = 2: halves; b = 3: third, punch-out, third, punch-out, ...)
template <int MAXO>
__global__ void __launch_bounds__(128)
k_enc_model(const FrameDesc *__restrict__ frames, uint32_t channels, uint32_t bps_stream,
            uint32_t blocksize, uint32_t windows, uint32_t max_lpc_cfg, uint32_t n_cands, uint32_t total_tasks,
            const EncSrc audio, EncSubStats *__restrict__ stats, const double *__restrict__ autoc_in,
            EncCand *__restrict__ cands, uint32_t side_ch) {
    const uint32_t gid = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t task = gid / n_cands, slot = gid - task * n_cands;
    if (task >= total_tasks) return;
    const uint32_t f = task / channels;
    const TaskLoc L = locate_task(frames, audio, f, task - f * channels);
    if (!fast_eligible(L)) return;
    constexpr uint32_t n = kMaxBlock;
    EncCand C;
    C.type = 0; C.order = 0; C.precision = 0; C.shift = 0;
#pragma unroll
    for (int j = 0; j < kMaxOrd; j++) C.coefs[j] = 0;
    const EncSubStats *stp = stats + task;
    const uint32_t st_flags = stp->flags;
    const uint32_t bps = bps_stream + (task - f * channels == side_ch ? 1u : 0u) - stp->wasted;
    if (!(st_flags & 1u)) {
        if constexpr (MAXO > 0) {
            // map the slot to (set, punch-out?)
            uint32_t set = 0;
            bool punch = false;
            if (slot == 0) set = 0;
            else if (slot <= 2) set = slot;                        // halves: sets 1, 2
            else { const uint32_t ci = slot - 3; set = 3 + ci / 2; punch = (ci & 1u) != 0; }   // thirds: sets 3, 4, 5
            const double *a = autoc_in + ((size_t)task * kMaxSets + set) * kLags;
            double autoc[MAXO + 1];
#pragma unroll
            for (int l = 0; l <= MAXO; l++) autoc[l] = a[l];
            const uint32_t max_lpc = max_lpc_cfg;
            if (punch) {
                const double *root = autoc_in + (size_t)task * kMaxSets * kLags;
                // libFLAC subtracts lags [0, max_lpc_order) only; the last lag keeps the partial window's value
#pragma unroll
                for (int l = 0; l < MAXO; l++) if ((uint32_t)l < max_lpc) autoc[l] = root[l] - autoc[l];
            }
            model_one<MAXO>(autoc, max_lpc, n, bps, qlp_precision_for(bps_stream, blocksize), C);
        }
    }
    cands[(size_t)task * kMaxCands + slot] = C;
}

// ------------------------------------------------------------------------------------------------ code
template <bool WIDE>
struct CodeShared {
    uint32_t bitbuf[WIDE ? 4232 : 2052];       // VERBATIM upper bound: 8 + 32 + 4096 x 33 bits (the 33-bit side subframe of a 32-bps stream)
    SearchShared search;
    uint8_t best_params[64];
    uint32_t scan[kEncThreads / 32];
};

// v < 2^len, 1 <= len <= 32: OR the bits into a zeroed MSB-first word buffer at bit position pos
__device__ __forceinline__ void put_bits_atomic(uint32_t *buf, uint32_t pos, uint32_t v, uint32_t len) {
    const uint32_t o = pos & 31u;
    const unsigned long long x = (unsigned long long)v << (64u - o - len);
    const uint32_t hi = (uint32_t)(x >> 32), lo = (uint32_t)x;
    if (hi) atomicOr(&buf[pos >> 5], hi);
    if (lo) atomicOr(&buf[(pos >> 5) + 1], lo);
}

// A sample of a subframe with `bps` bits per sample, bps up to 33 (the side subframe of a two-channel 32-bps stream): the
// samples are int32 (the caller guarantees that the side channel fits), so a 33rd bit is the sign.
__device__ __forceinline__ void put_sample_atomic(uint32_t *buf, uint32_t pos, int32_t x, uint32_t bps) {
    if (bps > 32) { put_bits_atomic(buf, pos, x < 0 ? 1u : 0u, bps - 32); put_bits_atomic(buf, pos + bps - 32, (uint32_t)x, 32); }
    else if (bps) put_bits_atomic(buf, pos, (uint32_t)x & (bps == 32 ? 0xFFFFFFFFu : ((1u << bps) - 1u)), bps);
}

// Per-thread bit accumulator over the zeroed shared word buffer (MSB first).  `hi` holds the pending bits of
// the current word (top `fill` < 32 bits); a code of len <= 32 bits is split into the part that still fits and
// the spill-over, and a completed word is OR-ed in with a predicated reduction (a thread's first and last
// word can be shared with its neighbours, and a data-dependent branch would diverge in almost every step).
// v1 kept a 64-bit window and branched on the flush: ~26 instructions per code (profiles/r01_ncu_enc_v5_lines_code.txt).
struct PackWriter {
    uint32_t addr, fill, hi;     // shared-space byte address of the current word
    __device__ __forceinline__ void init(uint32_t *b, uint32_t bitpos) {
        addr = (uint32_t)__cvta_generic_to_shared(b) + ((bitpos >> 5) << 2); fill = bitpos & 31u; hi = 0;
    }
    __device__ __forceinline__ void put(uint32_t v, uint32_t len) {        // 1 <= len <= 32, v < 2^len
        const uint32_t vh = v << (32u - len);                              // left-aligned code
        hi |= vh >> fill;
        const uint32_t lo = __funnelshift_lc(0u, vh, 32u - fill);          // spill-over: vh << (32 - fill), 0 when fill == 0
        fill += len;
        asm volatile("{\n\t.reg .pred p;\n\t"
                     "setp.ge.u32 p, %1, 32;\n\t"
                     "@p red.shared.or.b32 [%2], %0;\n\t"
                     "@p mov.b32 %0, %3;\n\t"
                     "@p add.u32 %2, %2, 4;\n\t"
                     "@p sub.u32 %1, %1, 32;\n\t"
                     "}\n" : "+r"(hi), "+r"(fill), "+r"(addr) : "r"(lo) : "memory");
    }
    // the same for 0 <= len <= 32 (len == 0 with v == 0 writes nothing): the left-aligning shift is a PTX shift, whose
    // count clamps at 32 (the C++ operator is undefined there)
    __device__ __forceinline__ void put0(uint32_t v, uint32_t len) {
        uint32_t vh;
        asm("shl.b32 %0, %1, %2;" : "=r"(vh) : "r"(v), "r"(32u - len));
        hi |= vh >> fill;
        const uint32_t lo = __funnelshift_lc(0u, vh, 32u - fill);
        fill += len;
        asm volatile("{\n\t.reg .pred p;\n\t"
                     "setp.ge.u32 p, %1, 32;\n\t"
                     "@p red.shared.or.b32 [%2], %0;\n\t"
                     "@p mov.b32 %0, %3;\n\t"
                     "@p add.u32 %2, %2, 4;\n\t"
                     "@p sub.u32 %1, %1, 32;\n\t"
                     "}\n" : "+r"(hi), "+r"(fill), "+r"(addr) : "r"(lo) : "memory");
    }
    __device__ __forceinline__ void zeros(uint32_t q) {
        fill += q;
        while (fill >= 32) {
            if (hi) asm volatile("red.shared.or.b32 [%0], %1;\n" ::"r"(addr), "r"(hi) : "memory");
            hi = 0; addr += 4; fill -= 32;
        }
    }
    __device__ __forceinline__ void finish() {
        if (hi) asm volatile("red.shared.or.b32 [%0], %1;\n" ::"r"(addr), "r"(hi) : "memory");
    }
};

// Rare path of the packing loop (a thread that holds a code longer than 32 bits: long unary runs), out of line and
// rolled up so that it costs no instruction-cache space in the hot kernel.
__device__ __noinline__ void pack_codes_long(uint32_t addr, uint32_t fill, uint32_t hi, uint32_t kcur, uint32_t skip,
                                             int32_t r0, int32_t r1, int32_t r2, int32_t r3, int32_t r4, int32_t r5, int32_t r6, int32_t r7,
                                             int32_t r8, int32_t r9, int32_t r10, int32_t r11, int32_t r12, int32_t r13, int32_t r14, int32_t r15) {
    const int32_t r[kSPT] = {r0, r1, r2, r3, r4, r5, r6, r7, r8, r9, r10, r11, r12, r13, r14, r15};
    PackWriter bw;
    bw.addr = addr; bw.fill = fill; bw.hi = hi;
    const uint32_t kbit = 1u << kcur, kmask = kbit - 1u, k1 = kcur + 1;
#pragma unroll 1
    for (uint32_t s = skip; s < (uint32_t)kSPT; s++) {
        const uint32_t u = (uint32_t)r[s];
        const uint32_t q = u >> kcur;
        const uint32_t tailv = kbit | (u & kmask);
        if (q + k1 <= 32) bw.put(tailv, q + k1);
        else { bw.zeros(q); bw.put(tailv, k1); }
    }
    bw.finish();
}

// Residual of this thread's 16 samples.  Returns the OR of |r| (>= 2^30 means an exact overflow check is needed).
template <bool WIDE, int TAPS>
__device__ __forceinline__ uint32_t residual16(const int32_t (&xs)[28], const int32_t (&cf)[kMaxOrd], int shift, int32_t (&r)[kSPT],
                                               uint32_t *hi_mismatch) {
    uint32_t ora = 0, bad = 0;
#pragma unroll
    for (int s = 0; s < kSPT; s++) {
        if (WIDE) {
            long long acc = 0;
#pragma unroll
            for (int j = 0; j < TAPS; j++) acc += (long long)cf[j] * (long long)xs[12 + s - 1 - j];
            const long long v = (long long)xs[12 + s] - (acc >> shift);
            r[s] = (int32_t)v;
            bad |= (uint32_t)((int32_t)(v >> 32) ^ (r[s] >> 31));        // non-zero iff v is not the sign extension of r
        } else {
            // <= 16-bit samples, precision <= 32 - bps - ilog2(order): every partial sum fits int32 (libFLAC's rule);
            // the subtraction may wrap only if |prediction| >= 2^31 - 2^16, which leaves |r| >= 2^30: caught through ora
            int32_t acc = 0;
#pragma unroll
            for (int j = 0; j < TAPS; j++) acc += cf[j] * xs[12 + s - 1 - j];
            r[s] = (int32_t)((uint32_t)xs[12 + s] - (uint32_t)(acc >> shift));
        }
        ora |= (uint32_t)abs(r[s]);
    }
    *hi_mismatch = bad;
    return ora;
}

// Rare path (a residual magnitude reached 2^30): the oracle's exact test r > INT32_MAX || r <= INT32_MIN in 64-bit
// arithmetic for this thread's samples, read back from global memory so the hot path keeps its arrays in registers.
__device__ __noinline__ bool residual_overflows(const void *src, uint32_t a16, uint32_t wasted, const EncCand *__restrict__ C, int tid) {
    const int order = C->order, shift = C->shift;
    TaskLoc L;
    L.src = src; L.a16 = a16; L.n = kMaxBlock;
    bool bad = false;
    for (int s = 0; s < kSPT; s++) {
        const int i = tid * kSPT + s;
        if (i < order) continue;
        long long acc = 0;
        for (int j = 0; j < order; j++) acc += (long long)C->coefs[j] * (long long)(sample_at(L, (uint32_t)(i - 1 - j)) >> wasted);
        const long long v = (long long)(sample_at(L, (uint32_t)i) >> wasted) - (acc >> shift);
        if (v > 2147483647ll || v <= -2147483648ll) bad = true;
    }
    return bad;
}

template <bool WIDE>
__global__ void __launch_bounds__(kEncThreads, WIDE ? 2 : FRB_CODE_MINB)
k_enc_code(const FrameDesc *__restrict__ frames, uint32_t channels, uint32_t bps_stream,
           uint32_t max_po_cfg, uint32_t n_cands, const EncSrc audio,
           const EncSubStats *__restrict__ stats, const EncCand *__restrict__ cands, uint32_t slot_words,
           uint32_t *__restrict__ slots, uint32_t *__restrict__ sub_bits, uint32_t c0, uint32_t side_extra,
           uint32_t *__restrict__ sub_est) {
    __shared__ __align__(16) CodeShared<WIDE> S;
    const uint32_t cch = blockIdx.y + c0;
    const uint32_t task = blockIdx.x * channels + cch;
    const TaskLoc L = locate_task(frames, audio, blockIdx.x, cch);
    if (!fast_eligible(L)) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr uint32_t n = kMaxBlock;
    const uint32_t k_limit = bps_stream > 16 ? 31u : 15u;
    const EncSubStats *stp = stats + task;
    const uint32_t wasted = stp->wasted, st_flags = stp->flags;
    const uint32_t bps = bps_stream + side_extra - wasted;
    // 16-bit kernel (64-register cap): the samples are fetched again for every evaluation (L1 / L2 hits) instead of living in
    // 28 registers across the Rice search and the packing phase, where nothing reads them.  The 64-bit kernel runs at 128
    // registers and keeps them (with nine candidates per subframe at level 8 the reloads only add work: C4 38.3 against 34.7 ms).
    constexpr bool RELOAD = FRB_CODE_RELOAD != 0 && !WIDE;
    int32_t xs0[28];
    if constexpr (!RELOAD) {
        load_samples28(L, tid, xs0);
        if (wasted) {
#pragma unroll
            for (int j = 0; j < 28; j++) xs0[j] >>= wasted;
        }
    }
    {   // zero the bit buffer
        constexpr int nq = (int)(sizeof(S.bitbuf) / 16);
        uint4 *b4 = reinterpret_cast<uint4 *>(S.bitbuf);
        for (int q = tid; q < nq; q += kEncThreads) b4[q] = make_uint4(0, 0, 0, 0);
    }
    const uint32_t verbatim_bits = 8 + wasted + n * bps;
    int best_type = 1, best_order = 0, best_prec = 0, best_shift = 0, best_slot = -1, best_po = 0;
    uint32_t best_bits = verbatim_bits;
    int32_t r[kSPT];
    int cur_slot = -1;           // LPC candidate whose residual is in r[]
    const uint32_t P = max_po_cfg;   // finest partition order (3..6 for n = 4096)

    // residual of candidate C into r[] (warm-up positions of thread 0 zeroed).  Returns OR |r|, sets *bad.
    auto eval_residual = [&](const EncCand &C, const EncCand *Cg, bool *bad_out) -> uint32_t {
        int32_t xr[28];
        if constexpr (RELOAD) {
            load_samples28(L, tid, xr);
            if (wasted) {
#pragma unroll
                for (int j = 0; j < 28; j++) xr[j] >>= wasted;
            }
        }
        const int32_t (&xs)[28] = pick_ref<RELOAD>(xr, xs0);
        int32_t cf[kMaxOrd];
#pragma unroll
        for (int j = 0; j < kMaxOrd; j++) cf[j] = C.coefs[j];
        uint32_t ora, him;
        if (C.order <= 4) ora = residual16<WIDE, 4>(xs, cf, C.shift, r, &him);
        else if (C.order <= 8) ora = residual16<WIDE, 8>(xs, cf, C.shift, r, &him);
        else ora = residual16<WIDE, 12>(xs, cf, C.shift, r, &him);
        if (tid == 0) {
            ora = 0;
#pragma unroll
            for (int s = 0; s < kSPT; s++) { if (s < C.order) r[s] = 0; ora |= (uint32_t)abs(r[s]); }   // order <= 12 < 16
        }
        bool bad = false;
        if (Cg != nullptr && ((WIDE && him) || ora >= 0x40000000u)) bad = residual_overflows(L.src, L.a16, wasted, Cg, tid);
        *bad_out = bad;
        return ora;
    };

    if (st_flags & 1u) {
        const uint32_t b = 8 + wasted + bps;
        if (b < best_bits) { best_type = 0; best_bits = b; }
    } else {
        // FIXED candidate: searched by k_enc_stats from the abs sums it had in registers
        if ((st_flags & 2u) && stp->fx_bits < best_bits) {
            best_bits = stp->fx_bits; best_type = 2; best_order = (int)stp->fx_order; best_po = (int)stp->fx_po; best_slot = -2;
            if (tid < 64) S.best_params[tid] = stp->fx_params[tid];
        }
        // Passes 0 .. n_cands-1 evaluate the LPC candidates; the last pass makes sure r[] holds the residual of the winner
        // (the FIXED candidate was searched by k_enc_stats without a residual pass; with several candidates the winner may
        // not be the one evaluated last).  ONE loop so that the residual code (three tap counts, 16 samples unrolled)
        // exists once: as three inlined copies the kernel was 96 KB of instructions, and four CTAs per SM in different
        // phases miss the instruction cache (stall "no_instruction").
        for (uint32_t slot = 0; slot <= n_cands; slot++) {
            const bool final_pass = slot == n_cands;
            const EncCand *Cg = nullptr;
            EncCand C;
            if (!final_pass) {
                Cg = cands + (size_t)task * kMaxCands + slot;
                C = *Cg;
                if (C.type == 0) continue;                   // uniform over the CTA
            } else {
                if (best_type < 2 || best_slot == cur_slot) break;
                if (best_slot == -2) {                       // its overflow check was done by k_enc_stats: no Cg
                    C.type = 2; C.order = best_order; C.precision = 0; C.shift = 0;
#pragma unroll
                    for (int j = 0; j < kMaxOrd; j++) C.coefs[j] = 0;
                    if (best_order == 1) { C.coefs[0] = 1; }
                    else if (best_order == 2) { C.coefs[0] = 2; C.coefs[1] = -1; }
                    else if (best_order == 3) { C.coefs[0] = 3; C.coefs[1] = -3; C.coefs[2] = 1; }
                    else if (best_order == 4) { C.coefs[0] = 4; C.coefs[1] = -6; C.coefs[2] = 4; C.coefs[3] = -1; }
                } else {
                    Cg = cands + (size_t)task * kMaxCands + best_slot;
                    C = *Cg;
                }
            }
            bool bad_lane;
            const uint32_t ora = eval_residual(C, Cg, &bad_lane);
            if (final_pass) break;
            cur_slot = (int)slot;
            const uint32_t order = (uint32_t)C.order;
            // ---- per-thread abs sum (32-bit unless a residual is huge) ----
            unsigned long long s64;
            if (ora < 0x08000000u) {
                uint32_t s32 = 0;
#pragma unroll
                for (int s = 0; s < kSPT; s++) s32 = __sad(r[s], 0, s32);
                s64 = s32;
            } else {
                s64 = 0;
#pragma unroll
                for (int s = 0; s < kSPT; s++) s64 += (unsigned long long)(uint32_t)abs(r[s]);
            }
            finest_sums(s64, P, tid, S.search.fin);
            if (__syncthreads_or(bad_lane ? 1 : 0)) continue;                // uniform
            if (warp == 0) {
                uint32_t rb, bl;
                warp_search(S.search.fin, order, P, k_limit, lane, S.search.params, &rb, &bl);
                if (lane == 0) { S.search.rb = rb; S.search.best_l = bl; }
            }
            __syncthreads();
            const uint32_t total = 8 + wasted + 4 + 5 + order * ((uint32_t)C.precision + bps) + S.search.rb;
            if (total < best_bits) {
                best_bits = total; best_type = 3; best_order = C.order; best_prec = C.precision; best_shift = C.shift;
                best_slot = (int)slot; best_po = (int)(P - S.search.best_l);
                // (the FIXED parameters, if any, were stored before the barriers inside partition_search; S.search.params is
                // rewritten by warp 0 only after the first barrier of the next search)
                if (tid < 64) S.best_params[tid] = S.search.params[tid];
            }
        }
    }
    __syncthreads();

    // ---- exact bit lengths, fallback to VERBATIM, pack -------------------------------------------
    int type = best_type;
    const int order = best_order;
    uint32_t my_bits = 0, kcur = 0, plen = 4, method = 0, qmax = 0;
    bool pstart = false;
    if (type >= 2) {
        const uint32_t tl = 8 - (uint32_t)best_po;           // log2 threads per partition (psize = 4096 >> po >= 16)
        kcur = S.best_params[(uint32_t)tid >> tl];
        if (WIDE) {
            // Rice2 (5-bit parameters) as soon as any parameter of the chosen order needs it
            const uint32_t cnt = 1u << best_po;
            method = __syncthreads_or(((uint32_t)tid < cnt && S.best_params[tid < 64 ? tid : 0] >= 15) ? 1 : 0) ? 1u : 0u;
        }
        plen = method ? 5u : 4u;
        pstart = ((uint32_t)tid & ((1u << tl) - 1u)) == 0;
        uint32_t qsum = 0;
#pragma unroll
        for (int s = 0; s < kSPT; s++) { r[s] = (int32_t)zigzag(r[s]); const uint32_t q = (uint32_t)r[s] >> kcur; qsum += q; qmax = max(qmax, q); }
        const uint32_t cnt = tid == 0 ? kSPT - (uint32_t)order : (uint32_t)kSPT;    // warm-up slots hold 0 and add nothing to qsum
        my_bits = qsum + cnt * (1 + kcur) + (pstart ? plen : 0u);
    }
    uint32_t hdr_bits = 8 + wasted;
    if (type == 0) hdr_bits += bps;
    else if (type == 2) hdr_bits += (uint32_t)order * bps + 6;
    else if (type == 3) hdr_bits += (uint32_t)order * bps + 9 + (uint32_t)(order * best_prec) + 6;
    // CTA exclusive scan of my_bits
    uint32_t total_res, my_off;
    {
        uint32_t inc = my_bits;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, o); if (lane >= o) inc += t; }
        if (lane == 31) S.scan[warp] = inc;
        __syncthreads();
        uint32_t base = 0, tot = 0;
#pragma unroll
        for (int w = 0; w < kEncThreads / 32; w++) { const uint32_t s = S.scan[w]; if (w < warp) base += s; tot += s; }
        total_res = tot; my_off = base + inc - my_bits;
    }
    if (type >= 2 && hdr_bits + total_res > verbatim_bits) type = 1;     // exactness guard
    uint32_t total_bits;
    if (type == 1) { hdr_bits = 8 + wasted; total_bits = verbatim_bits; }
    else total_bits = hdr_bits + total_res;

    // ---- subframe header, written cooperatively (one field per thread, atomic ORs into the zeroed buffer) ----
    const uint32_t mask_bps = bps >= 32 ? 0xFFFFFFFFu : ((1u << bps) - 1u);
    const uint32_t pos0 = 8 + wasted;                        // first bit after the type byte and the wasted-bits unary code
    if (tid == 0) {
        const uint32_t typecode = type == 0 ? 0u : type == 1 ? 1u : type == 2 ? (8u | (uint32_t)order) : (32u | (uint32_t)(order - 1));
        put_bits_atomic(S.bitbuf, 0, (typecode << 1) | (wasted ? 1u : 0u), 8);
        if (wasted) put_bits_atomic(S.bitbuf, 8 + wasted - 1, 1, 1);
        if (type == 0 && bps) put_sample_atomic(S.bitbuf, pos0, sample_at(L, 0) >> wasted, bps);
    }
    if (type >= 2) {
        if (tid >= 32 && tid < 32 + order)                   // warm-up sample j = tid - 32
            put_sample_atomic(S.bitbuf, pos0 + (uint32_t)(tid - 32) * bps, sample_at(L, (uint32_t)(tid - 32)) >> wasted, bps);
        const uint32_t pos1 = pos0 + (uint32_t)order * bps;
        if (type == 3) {
            const uint32_t prec = (uint32_t)best_prec;
            if (tid == 96) put_bits_atomic(S.bitbuf, pos1, ((prec - 1) << 5) | ((uint32_t)best_shift & 31u), 9);
            if (tid >= 64 && tid < 64 + order)
                put_bits_atomic(S.bitbuf, pos1 + 9 + (uint32_t)(tid - 64) * prec,
                                (uint32_t)cands[(size_t)task * kMaxCands + best_slot].coefs[tid - 64] & ((1u << prec) - 1u), prec);
        }
        if (tid == 128) put_bits_atomic(S.bitbuf, hdr_bits - 6, (method << 4) | (uint32_t)best_po, 6);
    }
    PackWriter bw;
    if (type == 1) {
        bw.init(S.bitbuf, hdr_bits + (uint32_t)tid * kSPT * bps);
        if (bps) {
            int32_t xr[28];
            if constexpr (RELOAD) {
                load_samples28(L, tid, xr);
#pragma unroll
                for (int j = 12; j < 28; j++) xr[j] >>= wasted;
            }
            const int32_t (&xs)[28] = pick_ref<RELOAD>(xr, xs0);
            if (WIDE && bps > 32) {
#pragma unroll
                for (int s = 0; s < kSPT; s++) { bw.put(xs[12 + s] < 0 ? 1u : 0u, bps - 32); bw.put((uint32_t)xs[12 + s], 32); }
            } else {
#pragma unroll
                for (int s = 0; s < kSPT; s++) bw.put((uint32_t)xs[12 + s] & mask_bps, bps);
            }
        }
        bw.finish();
    } else if (type >= 2) {
        bw.init(S.bitbuf, hdr_bits + my_off);
        if (pstart) bw.put(kcur, plen);
        const uint32_t kbit = 1u << kcur, kmask = kbit - 1u, k1 = kcur + 1;
        const uint32_t skip = tid == 0 ? (uint32_t)order : 0u;          // thread 0: its first `order` slots are warm-up samples, not codes
        // Per code the writer used to test "is this a warm-up slot" (re-reading %tid) and "does the code fit one 32-bit
        // write", each a branch around the writer's inline assembly: 26 instructions per code
        // (profiles/r02_ncu_lines_v1.txt).  Whether ANY of the thread's codes is longer than 32 bits is known from the
        // length pass (qmax), so the common loop has no length test, and a warm-up slot is a zero-length write of zero
        // (two selects) instead of a branch.
        if (qmax + k1 <= 32) {
#pragma unroll
            for (int s = 0; s < kSPT; s++) {
                const uint32_t u = (uint32_t)r[s];
                const uint32_t q = u >> kcur;
                const uint32_t tailv = kbit | (u & kmask);
                if (s < kMaxOrd) { const bool on = (uint32_t)s >= skip; bw.put0(on ? tailv : 0u, on ? q + k1 : 0u); }
                else bw.put(tailv, q + k1);                  // zeros, stop bit and LSBs in one write
            }
            bw.finish();
        } else {
            pack_codes_long(bw.addr, bw.fill, bw.hi, kcur, skip, r[0], r[1], r[2], r[3], r[4], r[5], r[6], r[7], r[8], r[9], r[10], r[11],
                            r[12], r[13], r[14], r[15]);
        }
    }
    __syncthreads();
    // ---- slot store (128-bit, coalesced) ----
    const uint32_t nwords = (total_bits + 31) / 32;
    uint32_t *slot = slots + (size_t)task * slot_words;
    const uint32_t nq = (nwords + 1 + 3) / 4;          // one extra word so the emitter can funnel-read past the end
    const uint4 *b4 = reinterpret_cast<const uint4 *>(S.bitbuf);
    uint4 *s4 = reinterpret_cast<uint4 *>(slot);
    for (uint32_t q = tid; q < nq && q * 4 < slot_words; q += kEncThreads) s4[q] = b4[q];
    if (tid == 0) { sub_bits[task] = total_bits; if (sub_est) sub_est[task] = best_bits; }      // estimate = libFLAC's decision metric
}
