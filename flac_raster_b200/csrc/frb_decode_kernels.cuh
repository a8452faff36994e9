// frb_decode_kernels.cuh -- included inside namespace frb by frb_decode.cuh.
//
// Decode pipeline after k_sync_scan (history: the v1 thread-per-frame kernel ran at 9.7 % occupancy on 8-band tiles and
// spent 228 instructions per sample, profiles/r01_ncu_dec_v1_raw_subset.csv; v2 split it into a skim kernel and a
// thread-per-subframe decode kernel; v3 fuses the two launches and optionally the denormalisation):
//   k_decode_subframes  ONE launch with two roles.  Skim CTAs (lowest block indices; channels > 1 only): one thread per
//                       frame walks the Rice codes without reconstructing anything and publishes each subframe's bit
//                       offset as soon as it is known.  Decode CTAs: one thread per SUBFRAME in channel-major order
//                       waits for its offset, then Rice decode + predictor restore from a register history (taps padded
//                       to the warp's order class 4/8/12, 64-bit MACs only when libFLAC's rule demands them); output is
//                       either the planar int32 audio (128-bit stores) or, fused, the denormalised pixels written
//                       straight into the tile's window of the raster
//   k_crc16_frames      one warp per frame, rows of 30 16-byte chunks, one chunk per lane and row, folded without tables
//                       (CrcFold, frb_crc16.cuh), lane weights and tail powers once per frame (side stream, launched
//                       behind the decode kernel)

// ---- cp.async / shared-memory helpers ------------------------------------------------------------------
constexpr int kDecThreads = 128;
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }
__device__ __forceinline__ uint32_t lds_u32(uint32_t smem_addr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];\n" : "=r"(v) : "r"(smem_addr) : "memory");
    return v;
}

__device__ __forceinline__ int32_t unzigzag(uint32_t u) {
    int32_t sgn;                                              // -(u & 1): a one-bit signed field extract instead of AND + negate
    asm("bfe.s32 %0, %1, 0, 1;" : "=r"(sgn) : "r"(u));
    return (int32_t)(u >> 1) ^ sgn;
}
// (defined here, in front of its first use: round 2's first build had the default further down, so `#if FRB_BFIND_I2F` saw an
// undefined macro and the library kept using bfind)
#ifndef FRB_BFIND_I2F
#define FRB_BFIND_I2F 1
#endif
// position of the most significant set bit (0xFFFFFFFF for 0): clz(w) = 31 - bfind(w), so the length of a Rice code with
// parameter k is (k + 32) - bfind(window) in one subtraction, and 33 + k (> 32, "too long") for an all-zero window
// Measured on B200 (tools/microbench/lat.cu, dependent chains): bfind/clz/popc ~20 cycles, an integer -> float conversion
// ~6 cycles, shifts / multiply-adds 4.5, adds 3.  The Rice walk is ONE chain of bfind -> length -> shift per code, so the
// position of the leading one is taken from the exponent of cvt.rz.f32.u32 (round toward zero: exactly floor(log2 w));
// w == 0 gives a huge value (0 - 127), like bfind's 0xFFFFFFFF, which the callers read as "code longer than 32 bits".
__device__ __forceinline__ uint32_t bfind_u32(uint32_t w) {
#if FRB_BFIND_I2F
    float f;
    asm("cvt.rz.f32.u32 %0, %1;" : "=f"(f) : "r"(w));
    return (__float_as_uint(f) >> 23) - 127u;
#else
    uint32_t r;
    asm("bfind.u32 %0, %1;" : "=r"(r) : "r"(w));
    return r;
#endif
}
__device__ __forceinline__ uint32_t shr_clamped(uint32_t v, uint32_t s) {      // v >> s with s >= 32 giving 0 (PTX semantics)
    uint32_t r;
    asm("shr.b32 %0, %1, %2;" : "=r"(r) : "r"(v), "r"(s));
    return r;
}

struct FrameLoc {
    uint64_t start, end;      // byte range [start, end) of the frame incl. CRC-16
    uint32_t k, n, stream;    // frame number in stream, blocksize of this frame
    bool ok;
};

__device__ __forceinline__ FrameLoc locate_frame(const DecStreamDev *__restrict__ streams, uint32_t n_streams,
                                                 uint32_t blocksize, uint32_t f,
                                                 const unsigned long long *__restrict__ frame_pos, DecStreamDev *st_out) {
    uint32_t lo = 0, hi = n_streams - 1;
    while (lo < hi) {
        const uint32_t mid = (lo + hi + 1) >> 1;
        if (streams[mid].frame_base <= f) lo = mid; else hi = mid - 1;
    }
    const DecStreamDev st = streams[lo];
    FrameLoc L;
    L.stream = lo;
    L.k = f - st.frame_base;
    const unsigned long long p0 = frame_pos[f];
    const unsigned long long p1 = (L.k + 1 < st.n_frames) ? frame_pos[f + 1] : (st.byte_offset + st.byte_length);
    L.n = (L.k + 1 < st.n_frames) ? blocksize : (uint32_t)(st.n_samples - (uint64_t)L.k * blocksize);
    L.ok = !(p0 == kNoPos || p1 == kNoPos || p1 <= p0 + 4);
    L.start = p0; L.end = p1;
    *st_out = st;
    return L;
}

// status words: 0 frames_missing, 1 crc16_errors, 2 parse_errors, 3 frames_decoded, 4 order_overflow

// ---- bit reader + skim: subframe bit offsets for multi-channel frames ------------------------------
// sub_bitoff[f*channels + c] = bit offset of subframe c from the frame start; 0 marks a bad frame.
// One thread per frame walks subframes 0..C-2 (the last one only needs its start; its end is checked by
// the decode kernel).
//
// With 32 independent frames per warp every data-dependent branch is taken by SOME lane in almost every
// step, so the warp pays for the union of all paths: the v3 skim (shared-memory word ring, one Rice code
// per loop trip, refill branch) and a v4 trial (16-byte ring slots + register queue) executed 50-100 warp
// instructions per code (5.8 / 12.8 ms on C3, profiles/r01_ncu_skim_v4.txt).  This version keeps the hot
// loop free of data-dependent branches:
//   * codes are skipped in batches of kSkimBatch with predication (lane inactive once its partition is
//     exhausted); a code longer than 32 bits is the only branch in the batch;
//   * the window is (hi, lo) plus a pre-loaded next word; crossing a word boundary is three selects and a
//     predicated 4-byte LDS from the thread's ring, never a wait;
//   * the ring (16-byte chunks, cp.async) is topped up ONCE per batch at a warp-uniform point with
//     predicated copies, and one wait_group per batch covers every word the batch can touch.
#ifndef FRB_SKIM_BATCH
#define FRB_SKIM_BATCH 8
#endif
#ifndef FRB_LPC_NEWEST_LAST
#define FRB_LPC_NEWEST_LAST 1
#endif
#ifndef FRB_DEC_SHIFTWIN
#define FRB_DEC_SHIFTWIN 0
#endif
constexpr int kSkimRing = 16;                                   // 16-byte chunks per thread (256 contiguous bytes)
constexpr int kSkimBatch = FRB_SKIM_BATCH;                      // codes per skim batch: <= kSkimBatch words = kSkimBatch / 4 chunks
static_assert(kSkimBatch == 8 || kSkimBatch == 16, "the 16-chunk ring feeds batches of 8 or 16 codes");

// Bit reader (skim and decode roles): three consecutive big-endian words of the stream in registers -- A (holds the
// next unread bit), B, and C still as loaded (raw little-endian) -- plus a running bit position bp.  Only bits 0..4 of
// bp address A; bit 5 flipping means the position moved into B and the words shift up (A=B, B=bswap(C), C=next ring
// word).  The window of the next 32 bits is ONE wrap-mode funnel shift of A:B and the bookkeeping for a Rice code is
// 9 predicated instructions.  Two shifting-window readers came before it: a 64-bit window (2 funnel shifts + a
// 13-instruction predicated merge per code: 27 % of the decode kernel's instructions,
// profiles/r01_ncu_dec_v5_lines_decode.txt) and a 96-bit one whose merge stayed off the clz chain (17 per code).  They
// had shorter dependent chains, which mattered while the kernels were latency-bound; the fused skim+decode kernel is
// issue-bound (ALU pipe 55-59 %, profiles/r01_ncu_dec_v6_fused.txt) and the instruction count decides: 4.04 -> 3.84 ms.
// Ring: the thread's 16 chunks are contiguous in shared memory (256-byte aligned), chunk index XOR-swizzled with the
// lane so that lanes reading the same word offset spread over the banks.
struct BitReader {
    const uint4 *gq;
    uint32_t sbase, swz, sx;
    uint32_t woff;           // 4 * (index of the next word to load); A is word woff/4 - 3
    uint32_t cissue, qlast;
    uint32_t A, B, Craw;
    uint32_t bp;             // (bp & 31) = offset of the next unread bit inside A
    __device__ __forceinline__ uint32_t load_raw4(uint32_t byte_off) const { return lds_u32(sx ^ (byte_off & 252u)); }
    __device__ __forceinline__ void copy_chunk(uint32_t c) const {
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sbase + (((c & (kSkimRing - 1)) << 4) ^ swz)),
                     "l"(gq + min(c, qlast)) : "memory");
    }
    // Tops the ring up by at most R chunks (R = what a batch of 4 R codes can consume at 32 bits each) without a branch:
    // predicated copies, so that the compiler can schedule them into the shadow of the Rice chain.  Afterwards at most
    // N copy groups stay in flight, N chosen so that the R + 1 chunks a batch (plus the skim's look-ahead) can touch are
    // complete: 15 - N R >= R + 1.
    template <int R>
    __device__ __forceinline__ void top_up_n() {
        const uint32_t lim = (woff >> 4) + kSkimRing - 1;
#pragma unroll
        for (int r = 0; r < R; r++) {
            asm volatile("{\n\t.reg .pred p;\n\tsetp.lt.u32 p, %0, %1;\n\t@p cp.async.cg.shared.global [%2], [%3], 16;\n\t}\n"
                         ::"r"(cissue), "r"(lim), "r"(sbase + (((cissue & (kSkimRing - 1)) << 4) ^ swz)), "l"(gq + min(cissue, qlast)) : "memory");
            cissue += cissue < lim ? 1u : 0u;
        }
        cp_async_commit();
        static_assert(R == 2 || R == 4, "ring depth table");
        cp_async_wait<R == 2 ? 5 : 2>();                         // 15 - N R >= R + 1
    }
    __device__ __forceinline__ void top_up() { top_up_n<2>(); }
    __device__ __forceinline__ void init(uint32_t ring_saddr, uint32_t lane, const uint8_t *base, uint64_t bitpos, uint64_t byte_end) {
        gq = (const uint4 *)base;
        sbase = ring_saddr;
        swz = (lane & 15u) << 4;
        sx = sbase ^ swz;
        const uint32_t w = (uint32_t)(bitpos >> 5);
        qlast = (uint32_t)(byte_end >> 4);
        cissue = w >> 2;
        for (int j = 0; j < kSkimRing - 1; j++) { copy_chunk(cissue); cissue++; }
        cp_async_commit();
        cp_async_wait<0>();
        A = bswap32(load_raw4(w << 2)); B = bswap32(load_raw4((w + 1) << 2)); Craw = load_raw4((w + 2) << 2);
        woff = (w + 3) << 2;
        bp = (uint32_t)bitpos & 31u;
    }
    __device__ __forceinline__ uint64_t bitpos() const { return (uint64_t)((woff >> 2) - 3u) * 32u + (bp & 31u); }
    __device__ __forceinline__ bool overrun() const { return (woff >> 4) > qlast + 2; }
    __device__ __forceinline__ uint32_t window() const { return __funnelshift_l(B, A, bp); }     // wrap mode: shift = bp & 31
    __device__ __forceinline__ void advance_predicated(uint32_t nb) {                             // nb <= 32
        asm volatile(
            "{\n\t.reg .pred p;\n\t.reg .b32 t, a;\n\t"
            "add.u32 t, %3, %6;\n\t"
            "xor.b32 a, t, %3;\n\t"
            "and.b32 a, a, 32;\n\t"
            "setp.ne.u32 p, a, 0;\n\t"
            "mov.u32 %3, t;\n\t"
            "@p mov.u32 %0, %1;\n\t"
            "@p prmt.b32 %1, %2, 0, 0x0123;\n\t"
            "@p and.b32 a, %4, 252;\n\t"
            "@p xor.b32 a, a, %5;\n\t"
            "@p ld.shared.u32 %2, [a];\n\t"
            "@p add.u32 %4, %4, 4;\n\t"
            "}\n"
            : "+r"(A), "+r"(B), "+r"(Craw), "+r"(bp), "+r"(woff)
            : "r"(sx), "r"(nb)
            : "memory");
    }
    __device__ __forceinline__ void consume(uint32_t nb) {         // nb <= 32
        const uint32_t t = bp + nb;
        if ((t ^ bp) & 32u) { A = B; B = bswap32(Craw); Craw = load_raw4(woff); woff += 4; }
        bp = t;
    }
    __device__ __forceinline__ uint32_t get(uint32_t nb) {          // nb in 0..32
        const uint32_t v = __funnelshift_lc(window(), 0u, nb);
        consume(nb);
        return v;
    }
    // nb in 0..33.  A 33-bit sample (side subframe of a two-channel 32-bps stream) is returned as int32: *ovf is set when its
    // 33rd bit is not the sign of the other 32, i.e. the value does not fit (full-range 32-bit stereo audio; the reference's
    // 24-bit audio always fits) -- the caller reports the subframe as undecodable instead of handing out a wrapped sample.
    __device__ __forceinline__ int32_t get_signed(uint32_t nb, bool *ovf = nullptr) {
        if (nb == 0) return 0;
        if (nb > 32) {
            const uint32_t top = get(nb - 32);
            const uint32_t v = get(32);
            if (ovf && top != (v >> 31)) *ovf = true;
            return (int32_t)v;
        }
        const uint32_t v = get(nb);
        const uint32_t sh = 32 - nb;
        return (int32_t)(v << sh) >> sh;
    }
    __device__ __forceinline__ uint32_t unary() {
        uint32_t q = 0;
        for (;;) {
            const uint32_t w = window();
            if (w) { const uint32_t z = __clz(w); consume(z + 1); return q + z; }
            q += 32; consume(32);
            top_up();
            if (overrun()) return q;
        }
    }
    __device__ __forceinline__ uint32_t rice_u(uint32_t k) {
        const uint32_t q = unary();
        const uint32_t low = get(k);
        return (q << k) | low;
    }
    __device__ __forceinline__ void seek(const uint8_t *base, uint64_t bits_forward, uint64_t byte_end) {
        const uint64_t target = bitpos() + bits_forward;
        cp_async_wait<0>();
        init(sbase, swz >> 4, base, target, byte_end);
    }
};

// Reader of the skim role.  The walk over a frame's Rice codes is ONE dependent chain of ~28 000 codes, and it gates
// every decode thread of that frame: with few frames in flight (a rank's share of a scene at N = 8, a single tile) the
// kernel's run time IS this chain (round 2, N = 2: 3.0 ms for half the frames against 3.8 ms for all of them).  The
// position-based BitReader above minimises instructions, but its chain per code is window -> bfind -> length ->
// position -> word-crossing test -> select -> window (8 dependent instructions, ~130 cycles per code measured).  Here
// the next 64 bits live in a shifting register pair (hi, lo) and a BitReader runs 64 bits AHEAD to supply the word that
// enters at the bottom: the chain per code is bfind -> subtract -> funnel shift; the look-ahead bookkeeping is off it.
struct SkimReader {
    BitReader br;            // positioned 64 bits ahead of the read position
    uint32_t hi, lo;         // bits [pos, pos + 32) and [pos + 32, pos + 64)
    __device__ __forceinline__ void prime() { hi = br.get(32); lo = br.get(32); }
    __device__ __forceinline__ void init(uint32_t ring_saddr, uint32_t lane, const uint8_t *base, uint64_t bitpos, uint64_t byte_end) {
        br.init(ring_saddr, lane, base, bitpos, byte_end);
        prime();
    }
    __device__ __forceinline__ uint64_t bitpos() const { return br.bitpos() - 64u; }
    __device__ __forceinline__ bool overrun() const { return br.overrun(); }
    __device__ __forceinline__ void top_up() { br.top_up_n<kSkimBatch / 4>(); }
    __device__ __forceinline__ uint32_t window() const { return hi; }
    __device__ __forceinline__ void skip_predicated(uint32_t nb) {     // nb <= 32; branch-free
        const uint32_t in = br.window();
        hi = __funnelshift_lc(lo, hi, nb);
        lo = __funnelshift_lc(in, lo, nb);
        br.advance_predicated(nb);
    }
    __device__ __forceinline__ void skip(uint32_t nb) {               // nb <= 32
        const uint32_t in = br.window();
        hi = __funnelshift_lc(lo, hi, nb);
        lo = __funnelshift_lc(in, lo, nb);
        br.consume(nb);
    }
    __device__ __forceinline__ uint32_t get(uint32_t nb) {            // nb in 0..32
        const uint32_t v = __funnelshift_lc(hi, 0u, nb);
        skip(nb);
        return v;
    }
    __device__ __forceinline__ uint32_t unary() {
        uint32_t q = 0;
        for (;;) {
            if (hi) { const uint32_t z = __clz(hi); skip(z + 1); return q + z; }
            q += 32; skip(32);
            top_up();
            if (overrun()) return q;
        }
    }
    __device__ __forceinline__ void seek(const uint8_t *base, uint64_t bits_forward, uint64_t byte_end) {
        const uint64_t target = bitpos() + bits_forward;
        cp_async_wait<0>();
        br.init(br.sbase, br.swz >> 4, base, target, byte_end);
        prime();
    }
};

// Publication protocol (fused skim + decode, see k_decode_subframes): sub_bitoff[] starts as kNotReady (host memset);
// the skim thread of a frame stores each subframe's bit offset with release semantics as soon as the walk reaches it
// (0 = bad frame, nothing to decode), the decode thread of that subframe polls it with acquire loads.
constexpr uint32_t kNotReady = 0xFFFFFFFFu;
__device__ __forceinline__ void st_release_u32(uint32_t *p, uint32_t v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;\n" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];\n" : "=r"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ void
skim_role(uint4 *s_ring, uint32_t cta, const uint8_t *__restrict__ bytes, const DecStreamDev *__restrict__ streams, uint32_t n_streams,
          uint32_t channels, uint32_t bps, uint32_t blocksize, uint32_t total_frames,
          const unsigned long long *__restrict__ frame_pos, uint32_t *__restrict__ sub_bitoff,
          uint8_t *__restrict__ frame_chassign, uint32_t *__restrict__ status, uint32_t lanes_per_warp) {
    // Only `lanes_per_warp` lanes of every warp take a frame: the walk is a long dependent chain, and there are far
    // fewer frames than the machine has thread slots, so spreading them over more warps buys latency hiding (and
    // less divergence per warp) for issue slots that would otherwise idle.
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t f = (cta * (blockDim.x >> 5) + (threadIdx.x >> 5)) * lanes_per_warp + lane;
    // No lane leaves before the walk is over: the loop below re-converges the whole warp at every trip
    // (__any_sync).  Without that, lanes in different phases (batch / partition change / subframe header) ran
    // their phases one after the other and a warp executed 3.3x the batches a single lane needs
    // (profiles/r01_ncu_skim_v5.txt).
    bool done = !(lane < lanes_per_warp && f < total_frames) || channels <= 1;
    DecStreamDev st;
    FrameLoc L; L.ok = false; L.start = L.end = 0; L.k = 0; L.n = 0; L.stream = 0;
    FrameHdr h; h.header_bytes = 0; h.ch_assign = 0;
    uint32_t *off_out = sub_bitoff + (size_t)(done ? 0 : f) * channels;
    uint64_t frame_bit0 = 0;
    uint32_t published = 0;                                   // entries [0, published) of off_out have been stored
    SkimReader br;
    br.br.gq = (const uint4 *)bytes; br.br.sbase = (uint32_t)__cvta_generic_to_shared(s_ring + threadIdx.x * kSkimRing); br.br.swz = (lane & 15u) << 4;
    br.br.sx = br.br.sbase ^ br.br.swz; br.br.woff = 12; br.br.cissue = 0; br.br.qlast = 0; br.br.A = br.br.B = br.br.Craw = 0; br.br.bp = 0;
    br.hi = br.lo = 0;
    if (lane < lanes_per_warp && f < total_frames && channels > 1) {
        L = locate_frame(streams, n_streams, blocksize, f, frame_pos, &st);
        if (!L.ok) { atomicAdd(&status[0], 1u); done = true; }
        else if (!parse_frame_header(bytes + L.start, L.end - L.start, 0, bps, &h)) { atomicAdd(&status[2], 1u); done = true; }
        else {
            frame_chassign[f] = (uint8_t)h.ch_assign;
            frame_bit0 = L.start * 8;
            st_release_u32(off_out, h.header_bytes * 8);
            published = 1;
            br.init(br.br.sbase, lane, bytes, frame_bit0 + (uint64_t)h.header_bytes * 8, L.end);
        }
        if (done) { for (uint32_t q = 0; q < channels; q++) st_release_u32(off_out + q, 0u); published = channels; }
    }
    const uint32_t n = L.n;
    bool err = false, in_res = false;
    uint32_t c = 0, left = 0, parts_left = 0, k = 0, plen = 4, esc = 15, psize = 0;
    while (__any_sync(0xFFFFFFFFu, !done)) {
        if (done) continue;
        br.top_up();
        if (left >= (uint32_t)kSkimBatch) {
            // ---- a full batch of Rice codes without data-dependent branches; a code longer than 32 bits (long unary
            // run or corrupt data) is detected once per batch and the batch is then redone one code at a time ----
            const SkimReader snap = br;
            const uint32_t kb = k + 32;
            uint32_t maxlen = 0;
#pragma unroll
            for (int i = 0; i < kSkimBatch; i++) {
                const uint32_t len = kb - bfind_u32(br.window());
                maxlen = max(maxlen, len);
                br.skip_predicated(len);
            }
            if (maxlen <= 32) { left -= kSkimBatch; continue; }
            br = snap;
        }
        if (left) {
            // ---- one batch of Rice codes, predicated on the lane still having codes in this partition ----
            const uint32_t m = left < (uint32_t)kSkimBatch ? left : (uint32_t)kSkimBatch;
            const uint32_t k1 = k + 1;
#pragma unroll
            for (int i = 0; i < kSkimBatch; i++) {
                const uint32_t w = br.window();
                uint32_t len = (uint32_t)__clz(w) + k1;
                const bool active = (uint32_t)i < m;
                if (active && len > 32) {                    // rare: long unary run (or a corrupt stream)
                    (void)br.unary();
                    len = k;
                    if (br.overrun()) { err = true; len = 0; }
                }
                br.skip(active ? len : 0u);
            }
            left -= m;
            if (err) done = true;
            continue;
        }
        if (in_res) {
            // partition exhausted: next partition, or the subframe is finished
            for (;;) {
                if (--parts_left == 0) { in_res = false; break; }
                left = psize;
                k = br.get(plen);
                if (k == esc) { const uint32_t raw = br.get(5); br.seek(bytes, (uint64_t)raw * left, L.end); left = 0; }
                if (left) break;
            }
            if (!in_res) { c++; st_release_u32(off_out + c, (uint32_t)(br.bitpos() - frame_bit0)); published = c + 1; }
            continue;
        }
        if (err || c + 1 >= channels) { done = true; continue; }
        {
            uint32_t sbps = bps;
            if ((h.ch_assign == 8 && c == 1) || (h.ch_assign == 9 && c == 0) || (h.ch_assign == 10 && c == 1)) sbps++;
            const uint32_t hd = br.get(8);
            const uint32_t t = (hd >> 1) & 0x3F;
            uint32_t wasted = 0;
            if (hd & 1) wasted = br.unary() + 1;
            if ((hd & 0x80) || wasted >= sbps) { err = true; done = true; continue; }
            sbps -= wasted;
            uint32_t order = 0;
            bool coded = false;
            if (t == 0) br.seek(bytes, sbps, L.end);
            else if (t == 1) br.seek(bytes, (uint64_t)sbps * n, L.end);
            else if (t >= 8 && t <= 12) { order = t - 8; coded = true; }
            else if (t >= 32) { order = t - 31; coded = true; }
            else { err = true; done = true; continue; }
            if (coded) {
                if (order > n) { err = true; done = true; continue; }
                br.seek(bytes, (uint64_t)order * sbps, L.end);
                if (t >= 32) {
                    const uint32_t prec = br.get(4) + 1;
                    if (prec == 16) { err = true; done = true; continue; }
                    br.seek(bytes, 5 + (uint64_t)order * prec, L.end);
                }
                const uint32_t m = br.get(2);
                const uint32_t po = br.get(4);
                plen = m ? 5u : 4u; esc = m ? 31u : 15u;
                psize = n >> po;
                if (m > 1 || (po > 0 && (n & ((1u << po) - 1))) || psize < order) { err = true; done = true; continue; }
                parts_left = 1u << po;
                left = psize - order;
                in_res = true;
                // settle on the first partition that actually holds Rice-coded residuals
                for (;;) {
                    k = br.get(plen);
                    if (k == esc) { const uint32_t raw = br.get(5); br.seek(bytes, (uint64_t)raw * left, L.end); left = 0; }
                    if (left) break;
                    if (--parts_left == 0) { in_res = false; break; }
                    left = psize;
                    if (psize == 0) { err = true; break; }
                }
            }
            if (!in_res) { c++; st_release_u32(off_out + c, (uint32_t)(br.bitpos() - frame_bit0)); published = c + 1; }
        }
        if (err) done = true;
    }
    const bool mine = lane < lanes_per_warp && f < total_frames && channels > 1 && L.ok && h.header_bytes != 0;
    if (mine && !err && br.bitpos() > L.end * 8) err = true;
    if (mine) {
        if (err) atomicAdd(&status[2], 1u);
        // whatever the walk did not reach is published as "bad" so that no decode thread waits for ever; subframes
        // already handed out are decoded (their threads notice the damage themselves) and the call reports the error
        for (uint32_t q = published; q < channels; q++) st_release_u32(off_out + q, 0u);
    }
}

// ---- subframe decode -------------------------------------------------------------------------------
template <int MAXORD, bool WIDE>
__device__ __forceinline__ int32_t lpc_predict(const int32_t (&cf)[MAXORD], const int32_t *Hj, int shift) {
    // Hj points at the newest history sample; taps walk backwards (static indices after unrolling)
#if FRB_LPC_NEWEST_LAST
    // oldest tap first: inside a batch the newest sample is the one just reconstructed, and with it last only one
    // multiply-add of the next sample waits for it
    if (WIDE) {
        long long acc = 0;
#pragma unroll
        for (int q = MAXORD - 1; q >= 0; q--) acc += (long long)cf[q] * (long long)Hj[-q];
        return (int32_t)(acc >> shift);
    } else {
        int32_t acc = 0;
#pragma unroll
        for (int q = MAXORD - 1; q >= 0; q--) acc += cf[q] * Hj[-q];
        return acc >> shift;
    }
#else
    if (WIDE) {
        long long acc = 0;
#pragma unroll
        for (int q = 0; q < MAXORD; q++) acc += (long long)cf[q] * (long long)Hj[-q];
        return (int32_t)(acc >> shift);
    } else {
        int32_t acc = 0;
#pragma unroll
        for (int q = 0; q < MAXORD; q++) acc += cf[q] * Hj[-q];
        return acc >> shift;
    }
#endif
}

// v << wasted (wasted-bits restore) with a check that nothing is shifted out: only a 33-bit side subframe of full-range
// 32-bit audio can do that (see BitReader::get_signed)
__device__ __forceinline__ int32_t shl_checked(int32_t v, uint32_t wasted, bool &err) {
    const int32_t r = (int32_t)((uint32_t)v << wasted);
    if ((r >> wasted) != v) err = true;
    return r;
}

// the prediction in 64 bits (the 64-bit instantiations check that prediction + residual still fits int32)
template <int MAXORD>
__device__ __forceinline__ long long lpc_predict64(const int32_t (&cf)[MAXORD], const int32_t *Hj, int shift) {
    long long acc = 0;
#if FRB_LPC_NEWEST_LAST
#pragma unroll
    for (int q = MAXORD - 1; q >= 0; q--) acc += (long long)cf[q] * (long long)Hj[-q];
#else
#pragma unroll
    for (int q = 0; q < MAXORD; q++) acc += (long long)cf[q] * (long long)Hj[-q];
#endif
    return acc >> shift;
}

// Optional fused denormalise: instead of the planar int32 audio buffer, a decode thread can write its samples straight
// into the window of the (bands,H,W) raster that its tile covers (denormalize_from_audio, normalization.py:222-249,
// same fp64 operation order as k_denormalize_tiles).  This removes the audio round trip through HBM (4 B written +
// 4 B read per sample) and the separate mapping kernel.  Uniform per launch:
struct SinkCfg {
    int dtype;               // FRB_U8..FRB_F64, or -1: plain audio output
    uint32_t esize;          // bytes per raster element
    uint32_t H, W;           // raster height / width
    const frb_tile *tiles;   // one per stream (stream i carries tile i, bands == channels)
    const double *minmax;    // {min,max} per tile
    uint8_t *raster;
    double scale, rcp;
    int fast;                // scale is one of the three reference constants (exact reciprocal division)
    int intpath;             // 8/16-bit integer raster + scale 32767: exact integer evaluation of the fp64 formula (sink_px)
    int window;              // window sink (frb_decode_window): raster is the (bands, H, W) window at image (win_row, win_col)
    uint32_t win_row, win_col;
};
// output of k_decode_subframes: planar int32 audio, the tiles' windows of a raster, or the part of them inside a window
constexpr int kSinkAudio = 0, kSinkTile = 1, kSinkWindow = 2;
struct RasterPos {           // per thread
    uint8_t *rowp;           // first pixel of the current row of this tile/band window
    uint32_t x, w, pitch;    // position inside the row, row length (pixels), raster row pitch in bytes
    double mn, range;        // fp64 path
    int32_t imn;             // integer path: data_min - 1, data_max - data_min (integers for integer rasters, range < 2^16)
    uint32_t irange, kround; // kround = 32767*range + 32767 + 65534 (see sink_px)
    // window sink: rowp/x address the current tile row as if the whole row were stored (x = column in the tile); only
    // rows [y0, y1) and columns [x0, x1) of the tile lie inside the window and are stored
    uint32_t y, y0, y1, x0, x1;
};

typedef BitReader DecReader;
struct SubCtx {
    DecReader br;
    RasterPos rp;
    int32_t *dst;            // first sample of this subframe in the planar audio buffer
    uint32_t n, order, sbps, wasted, type;
    bool aligned16;
    bool err;
};

constexpr int kDecBatch = 8;      // samples decoded per branch-free batch

__device__ __forceinline__ double sink_map(const SinkCfg &G, const RasterPos &R, int32_t a) {
    return G.fast ? denormalize_one_fast((double)a, G.scale, G.rcp, R.mn, R.range) : denormalize_one((double)a, G.scale, R.mn, R.range);
}
// Integer rasters behind 16-bit audio: the reference's value is v = ((a/32767 + 1)/2)*range + min in fp64, then
// np.round.  In exact arithmetic v = min + N/65534 with N = (a + 32767)*range, so its fraction is a multiple of
// 1/65534: either an exact tie or at least 1.5e-5 away from one, far more than the fp64 evaluation can drift (a few
// ulp of 2^17 ~ 1e-11).  Away from ties round(v) = min + floor((N + 32767)/65534).  With one more 65534 added to
// keep the numerator non-negative for a = -32768 (a foreign stream may hold it):
//     px = (min - 1) + (a*range + K) / 65534,  K = 32767*range + 32767 + 65534,   numerator in [0, 2^32)
// -- one multiply-add, a constant division and an add instead of ten fp64 / conversion instructions (the fused kernel
// is issue-bound).  A zero remainder marks an exact tie, where fp64 rounding decides: the caller redoes that sample
// with the fp64 formula (sink_px_tie).
__device__ __forceinline__ uint32_t sink_px(const RasterPos &R, int32_t a, bool &tie) {
    const uint32_t N = (uint32_t)a * R.irange + R.kround;
    const uint32_t q = N / 65534u;
    tie |= (N - q * 65534u) == 0u;
    return (uint32_t)R.imn + q;                               // imn holds min - 1
}
__device__ __noinline__ uint32_t sink_px_tie(double scale, double rcp, int32_t imn_minus_1, uint32_t irange, int32_t a) {
    return (uint32_t)(int32_t)__double2ll_rn(denormalize_one_fast((double)a, scale, rcp, (double)(imn_minus_1 + 1), (double)irange));
}
__device__ __forceinline__ void sink_store1(const SinkCfg &G, const RasterPos &R, int32_t a) {
    if (G.intpath) {
        bool tie = false;
        uint32_t v = sink_px(R, a, tie);
        if (tie) v = sink_px_tie(G.scale, G.rcp, R.imn, R.irange, a);
        if (G.esize == 2) reinterpret_cast<uint16_t *>(R.rowp)[R.x] = (uint16_t)v; else R.rowp[R.x] = (uint8_t)v;
    } else store_denorm(R.rowp, G.dtype, R.x, sink_map(G, R, a));
}
__device__ __forceinline__ void sink_put1(const SinkCfg &G, RasterPos &R, int32_t a) {
    sink_store1(G, R, a);
    if (++R.x == R.w) { R.x = 0; R.rowp += R.pitch; }
}
// rare slow path of sink_put_batch (a sample on an exact rounding tie, or a batch that straddles a row end): kept out of
// line so the hot loop stays small (the fused kernel showed instruction-cache stalls with everything inlined)
// (everything by value: a reference to the thread's RasterPos would force that struct into local memory)
__device__ __noinline__ void sink_put_batch_slow(uint8_t *rowp, uint32_t x, uint32_t w, uint32_t pitch, int dtype, int intpath, uint32_t esize,
                                                 int fast, double scale, double rcp, double mn, double range, int32_t imn, uint32_t irange,
                                                 uint32_t kround, int32_t a0, int32_t a1, int32_t a2, int32_t a3,
                                                 int32_t a4, int32_t a5, int32_t a6, int32_t a7) {
    const int32_t a[8] = {a0, a1, a2, a3, a4, a5, a6, a7};
    SinkCfg G;
    G.dtype = dtype; G.intpath = intpath; G.esize = esize; G.fast = fast; G.scale = scale; G.rcp = rcp;
    G.H = G.W = 0; G.tiles = nullptr; G.minmax = nullptr; G.raster = nullptr;
    RasterPos R;
    R.rowp = rowp; R.x = x; R.w = w; R.pitch = pitch; R.mn = mn; R.range = range; R.imn = imn; R.irange = irange; R.kround = kround;
#pragma unroll 1
    for (int j = 0; j < 8; j++) sink_put1(G, R, a[j]);
}
__device__ __forceinline__ void sink_advance(RasterPos &R, uint32_t n) {
    R.x += n;
    while (R.x >= R.w) { R.x -= R.w; R.rowp += R.pitch; }
}
#define FRB_SINK_SLOW(G, R, a)                                                                                                   \
    do {                                                                                                                         \
        sink_put_batch_slow((R).rowp, (R).x, (R).w, (R).pitch, (G).dtype, (G).intpath, (G).esize, (G).fast, (G).scale, (G).rcp,    \
                            (R).mn, (R).range, (R).imn, (R).irange, (R).kround, a[0], a[1], a[2], a[3], a[4], a[5], a[6], a[7]);   \
        sink_advance(R, kDecBatch);                                                                                              \
    } while (0)
// Rare paths of the 8/16-bit integer sink, out of line (one call site each) so that the hot loop stays small:
//  * a sample sits on an exact rounding tie: the whole batch is redone with the tied samples through the fp64 formula;
//  * the batch straddles the end of a tile row (edge tiles whose width is not a multiple of 8: their 32 frames per warp
//    reach row ends in different trips, so SOME lane is here in a quarter of the trips): element stores with the row
//    step in between -- ~50 instructions instead of the generic sample-by-sample path (~300).
__device__ __noinline__ uint4 sink_fix_ties(double scale, double rcp, int32_t imn, uint32_t irange, uint32_t kround, int shift16,
                                            int32_t a0, int32_t a1, int32_t a2, int32_t a3, int32_t a4, int32_t a5, int32_t a6, int32_t a7) {
    const int32_t a[8] = {a0, a1, a2, a3, a4, a5, a6, a7};
    uint32_t v[8];
#pragma unroll 1
    for (int j = 0; j < 8; j++) {
        const uint32_t N = (uint32_t)a[j] * irange + kround;
        const uint32_t q = N / 65534u;
        v[j] = (N - q * 65534u) == 0u ? sink_px_tie(scale, rcp, imn, irange, a[j]) : (uint32_t)imn + q;
    }
    if (shift16) return make_uint4(__byte_perm(v[0], v[1], 0x5410), __byte_perm(v[2], v[3], 0x5410), __byte_perm(v[4], v[5], 0x5410), __byte_perm(v[6], v[7], 0x5410));
    return make_uint4((v[0] & 0xFFu) | ((v[1] & 0xFFu) << 8) | ((v[2] & 0xFFu) << 16) | (v[3] << 24),
                      (v[4] & 0xFFu) | ((v[5] & 0xFFu) << 8) | ((v[6] & 0xFFu) << 16) | (v[7] << 24), 0u, 0u);
}
__device__ __noinline__ void sink_store_straddle(uint8_t *rowp, uint32_t x, uint32_t w, uint32_t pitch, int esize2,
                                                 uint32_t p0, uint32_t p1, uint32_t p2, uint32_t p3) {
    const uint32_t pk[4] = {p0, p1, p2, p3};
#pragma unroll
    for (int j = 0; j < 8; j++) {
        if (esize2) reinterpret_cast<uint16_t *>(rowp)[x] = (uint16_t)(pk[j >> 1] >> (16 * (j & 1)));
        else rowp[x] = (uint8_t)(pk[j >> 2] >> (8 * (j & 3)));
        if (++x == w) { x = 0; rowp += pitch; }
    }
}
// kDecBatch consecutive samples; one or two vector stores when they stay inside the row and the address allows it
__device__ __forceinline__ void sink_put_batch(const SinkCfg &G, RasterPos &R, const int32_t (&a)[kDecBatch]) {
    static_assert(kDecBatch == 8, "packing below assumes 8 samples");
    const bool inside = R.x + kDecBatch <= R.w;
    if (G.intpath && (G.dtype == FRB_U16 || G.dtype == FRB_I16)) {
        uint32_t pk[4];
        bool tie = false;
#pragma unroll
        for (int j = 0; j < 4; j++) pk[j] = __byte_perm(sink_px(R, a[2 * j], tie), sink_px(R, a[2 * j + 1], tie), 0x5410);
        if (tie) {
            const uint4 r = sink_fix_ties(G.scale, G.rcp, R.imn, R.irange, R.kround, 1, a[0], a[1], a[2], a[3], a[4], a[5], a[6], a[7]);
            pk[0] = r.x; pk[1] = r.y; pk[2] = r.z; pk[3] = r.w;
        }
        if (inside) {
            uint16_t *p = reinterpret_cast<uint16_t *>(R.rowp) + R.x;
            const uintptr_t ad = reinterpret_cast<uintptr_t>(p);
            if ((ad & 15u) == 0) *reinterpret_cast<uint4 *>(p) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
            else if ((ad & 7u) == 0) { reinterpret_cast<uint2 *>(p)[0] = make_uint2(pk[0], pk[1]); reinterpret_cast<uint2 *>(p)[1] = make_uint2(pk[2], pk[3]); }
            else if ((ad & 3u) == 0) {
#pragma unroll
                for (int j = 0; j < 4; j++) reinterpret_cast<uint32_t *>(p)[j] = pk[j];
            } else {
#pragma unroll
                for (int j = 0; j < 4; j++) { p[2 * j] = (uint16_t)pk[j]; p[2 * j + 1] = (uint16_t)(pk[j] >> 16); }
            }
            R.x += kDecBatch;
            if (R.x == R.w) { R.x = 0; R.rowp += R.pitch; }
        } else {
            sink_store_straddle(R.rowp, R.x, R.w, R.pitch, 1, pk[0], pk[1], pk[2], pk[3]);
            sink_advance(R, kDecBatch);
        }
        return;
    }
    if (G.intpath && (G.dtype == FRB_U8 || G.dtype == FRB_I8)) {
        uint32_t pk[2] = {0, 0};
        bool tie = false;
#pragma unroll
        for (int j = 0; j < 8; j++) pk[j >> 2] |= (sink_px(R, a[j], tie) & 0xFFu) << (8 * (j & 3));
        if (tie) {
            const uint4 r = sink_fix_ties(G.scale, G.rcp, R.imn, R.irange, R.kround, 0, a[0], a[1], a[2], a[3], a[4], a[5], a[6], a[7]);
            pk[0] = r.x; pk[1] = r.y;
        }
        if (inside) {
            uint8_t *p = R.rowp + R.x;
            if ((reinterpret_cast<uintptr_t>(p) & 7u) == 0) *reinterpret_cast<uint2 *>(p) = make_uint2(pk[0], pk[1]);
            else {
#pragma unroll
                for (int j = 0; j < 8; j++) p[j] = (uint8_t)(pk[j >> 2] >> (8 * (j & 3)));
            }
            R.x += kDecBatch;
            if (R.x == R.w) { R.x = 0; R.rowp += R.pitch; }
        } else {
            sink_store_straddle(R.rowp, R.x, R.w, R.pitch, 0, pk[0], pk[1], 0u, 0u);
            sink_advance(R, kDecBatch);
        }
        return;
    }
    if (inside) {
        if (G.dtype == FRB_U16 || G.dtype == FRB_I16) {
            uint16_t *p = reinterpret_cast<uint16_t *>(R.rowp) + R.x;
#pragma unroll
            for (int j = 0; j < kDecBatch; j++) p[j] = (uint16_t)(int32_t)__double2ll_rn(sink_map(G, R, a[j]));
        } else if (G.dtype == FRB_U8 || G.dtype == FRB_I8) {
            uint8_t *p = R.rowp + R.x;
#pragma unroll
            for (int j = 0; j < kDecBatch; j++) p[j] = (uint8_t)(int32_t)__double2ll_rn(sink_map(G, R, a[j]));
        } else {
#pragma unroll
            for (int j = 0; j < kDecBatch; j++) store_denorm(R.rowp, G.dtype, R.x + j, sink_map(G, R, a[j]));
        }
        R.x += kDecBatch;
        if (R.x == R.w) { R.x = 0; R.rowp += R.pitch; }
    } else {
        FRB_SINK_SLOW(G, R, a);
    }
}

// ---- window sink: the tile sink clipped to a window -------------------------------------------------
__device__ __forceinline__ bool win_row_visible(const RasterPos &R) { return R.y - R.y0 < R.y1 - R.y0; }
__device__ __forceinline__ void win_put1(const SinkCfg &G, RasterPos &R, int32_t a) {
    if (win_row_visible(R) && R.x - R.x0 < R.x1 - R.x0) sink_store1(G, R, a);
    if (++R.x == R.w) { R.x = 0; R.y++; R.rowp += R.pitch; }
}
// A batch inside the row's visible span takes the tile sink's vector stores; a batch inside a row outside the window
// only moves the position; the rest (batches across a row end or a window edge) goes sample by sample.
__device__ __forceinline__ void win_put_batch(const SinkCfg &G, RasterPos &R, const int32_t (&a)[kDecBatch]) {
    const bool vis = win_row_visible(R);
    if (vis && R.x >= R.x0 && R.x + kDecBatch <= R.x1) {
        sink_put_batch(G, R, a);                 // inside the row: never straddles, wraps to x = 0 at the row end
        if (R.x == 0) R.y++;
    } else if (!vis && R.x + kDecBatch <= R.w) {
        R.x += kDecBatch;
        if (R.x == R.w) { R.x = 0; R.y++; R.rowp += R.pitch; }
    } else {
#pragma unroll 1
        for (int j = 0; j < kDecBatch; j++) win_put1(G, R, a[j]);
    }
}
template <int SINK>
__device__ __forceinline__ void sink_one(const SinkCfg &G, RasterPos &R, int32_t a) {
    if constexpr (SINK == kSinkWindow) win_put1(G, R, a); else sink_put1(G, R, a);
}

// FIXED / LPC subframe, part 1 (per lane, divergent): warm-up samples, predictor, residual coding header and the
// first partition's parameter.  Run BEFORE the warp picks its sample loop, so that the loop can use libFLAC's
// 32-bit rule with the subframe's ACTUAL coefficient precision (16-bit audio coded by libFLAC has precision <= 12
// and never needs 64-bit accumulation; assuming the maximum of 15 sent every LPC subframe down the 64-bit path).
template <int PMAX>
struct PredState {
    int32_t hist[PMAX];      // hist[PMAX-1] = newest warm-up sample
    int32_t cf[PMAX];        // cf[q] multiplies the sample q+1 back; 0 beyond the order
    int shift;
    uint32_t k, plen, esc, psize, part_left, raw_bits, i;
    bool escape, wide;
};
template <int PMAX, int SINK>
__device__ __forceinline__ void decode_prologue(SubCtx &S, bool active, PredState<PMAX> &P, const SinkCfg &G) {
    DecReader &br = S.br;
    const uint32_t n = S.n, order = S.order, wasted = S.wasted;
#pragma unroll
    for (int q = 0; q < PMAX; q++) { P.hist[q] = 0; P.cf[q] = 0; }
    P.shift = 0; P.k = 0; P.plen = 4; P.esc = 15; P.psize = 0; P.part_left = 0; P.raw_bits = 0; P.i = n;
    P.escape = false; P.wide = false;
    if (!active) return;
    for (uint32_t w = 0; w < order; w++) {
        const int32_t v = br.get_signed(S.sbps, &S.err);
#pragma unroll
        for (int q = 0; q < PMAX - 1; q++) P.hist[q] = P.hist[q + 1];
        P.hist[PMAX - 1] = v;
        const int32_t sv = shl_checked(v, wasted, S.err);
        if (SINK == kSinkAudio) S.dst[w] = sv; else sink_one<SINK>(G, S.rp, sv);
    }
    br.top_up();
    if (S.type == 3) {
        const uint32_t prec = br.get(4) + 1;
        const uint32_t sh = br.get(5);
        if (prec == 16 || (sh & 16)) S.err = true;
        P.shift = (int)sh;
#pragma unroll
        for (int q = 0; q < PMAX; q++) if ((uint32_t)q < order) { P.cf[q] = br.get_signed(prec); if ((q & 7) == 7) br.top_up(); }
        br.top_up();
        // libFLAC's rule: 32-bit arithmetic is exact when bps + precision + ilog2(order) <= 32
        P.wide = S.sbps + prec + (uint32_t)(31 - __clz(order | 1u)) > 32u || S.sbps + wasted > 32u;    // 33-bit subframes: range-checked loop
    } else {
        if (order >= 1) P.cf[0] = order == 1 ? 1 : order == 2 ? 2 : order == 3 ? 3 : 4;
        if (order >= 2) P.cf[1] = order == 2 ? -1 : order == 3 ? -3 : -6;
        if (order >= 3) P.cf[2] = order == 3 ? 1 : 4;
        if (order >= 4) P.cf[3] = -1;
        P.wide = S.sbps + order > 32u || S.sbps + wasted > 32u;
    }
    const uint32_t m = br.get(2);
    const uint32_t po = br.get(4);
    P.plen = m ? 5u : 4u; P.esc = m ? 31u : 15u;
    P.psize = n >> po;
    if (m > 1 || (po > 0 && (n & ((1u << po) - 1))) || P.psize < order) S.err = true;
    if (!S.err) {
        P.k = br.get(P.plen);
        P.escape = (P.k == P.esc);
        P.raw_bits = P.escape ? br.get(5) : 0;
        P.part_left = P.psize - order;
        P.i = order;
        while (P.part_left == 0 && P.i < n) {
            if (P.psize == 0) { S.err = true; break; }
            P.k = br.get(P.plen); P.escape = (P.k == P.esc); P.raw_bits = P.escape ? br.get(5) : 0; P.part_left = P.psize;
        }
        if (S.err) P.i = n;
    }
}

// Part 2.  Called by ALL lanes of the warp (lanes without a predictive subframe arrive with i == n): the sample loop
// re-converges the warp at every trip, and a trip is either one batch of kDecBatch Rice codes parsed without
// data-dependent branches (predicated word merges, see BitReader) followed by the predictor recursion from the
// register history, or a single sample through the generic path (escape-coded partitions, partition tails, codes
// longer than 32 bits).
template <int MAXORD, bool WIDE, int PMAX, int SINK>
__device__ __forceinline__ void decode_predictive(SubCtx &S, const PredState<PMAX> &P, const SinkCfg &G) {
    DecReader &br = S.br;
    const uint32_t n = S.n, wasted = S.wasted;
    int32_t *dst = S.dst;
    int32_t H[MAXORD + kDecBatch];
    int32_t cf[MAXORD];
#pragma unroll
    for (int q = 0; q < MAXORD; q++) { H[q] = P.hist[PMAX - MAXORD + q]; cf[q] = P.cf[q]; }
#pragma unroll
    for (int q = MAXORD; q < MAXORD + kDecBatch; q++) H[q] = 0;
    const int shift = P.shift;
    uint32_t k = P.k, part_left = P.part_left, raw_bits = P.raw_bits, i = P.i;
    const uint32_t plen = P.plen, esc = P.esc, psize = P.psize;
    bool escape = P.escape;
    // kDecBatch Rice codes with parameter kk, no data-dependent branch; returns the longest code (> 32: the values are
    // garbage and the caller rewinds the reader).
    // code = z zeros, a one, k low bits.  With f = bfind(window) = 31 - z: length (k + 32) - f, and window >> (f - k) holds
    // the stop bit at position k with nothing above it, i.e. 2^k + low bits, so
    // u = (z << k) + low = ((30 - f) << k) + (window >> (f - k)): shift, multiply-add, add
    auto parse_batch = [&](uint32_t kk, uint32_t (&uu)[kDecBatch]) -> uint32_t {
        const uint32_t kb = kk + 32, npow2k = 0u - (1u << kk), c30k = 30u << kk;
        uint32_t maxlen = 0;
#pragma unroll
        for (int j = 0; j < kDecBatch; j++) {
            const uint32_t win = br.window();
            const uint32_t f = bfind_u32(win);
            const uint32_t len = kb - f;
            maxlen = max(maxlen, len);
            uu[j] = f * npow2k + shr_clamped(win, f - kk) + c30k;
            br.advance_predicated(len);
        }
        return maxlen;
    };
    // predictor recursion over a parsed batch into H[MAXORD..]; output of the batch at sample index i
    // 64-bit instantiations: a reconstructed sample that does not fit int32 (a 33-bit side channel of full-range 32-bit audio;
    // also what damaged data can produce) marks the subframe as undecodable instead of wrapping silently
    uint32_t ovf = 0;
    auto reconstruct = [&](const uint32_t (&uu)[kDecBatch]) {
#pragma unroll
        for (int j = 0; j < kDecBatch; j++) {
            if constexpr (WIDE) {
                const long long v = (long long)unzigzag(uu[j]) + lpc_predict64<MAXORD>(cf, &H[MAXORD - 1 + j], shift);
                H[MAXORD + j] = (int32_t)v;
                const long long vs = v << wasted;                 // what is stored: must fit int32 as well
                ovf |= (uint32_t)((int32_t)(vs >> 32) ^ ((int32_t)vs >> 31));
            } else {
                H[MAXORD + j] = unzigzag(uu[j]) + lpc_predict<MAXORD, WIDE>(cf, &H[MAXORD - 1 + j], shift);
            }
        }
    };
    auto output_batch = [&]() {
        if (SINK != kSinkAudio) {
            int32_t o[kDecBatch];
#pragma unroll
            for (int j = 0; j < kDecBatch; j++) o[j] = (int32_t)((uint32_t)H[MAXORD + j] << wasted);
            if constexpr (SINK == kSinkWindow) win_put_batch(G, S.rp, o); else sink_put_batch(G, S.rp, o);
        } else if (S.aligned16) {
#pragma unroll
            for (int q = 0; q < kDecBatch / 4; q++)
                *reinterpret_cast<int4 *>(dst + i + 4 * q) =
                    make_int4((int32_t)((uint32_t)H[MAXORD + 4 * q] << wasted), (int32_t)((uint32_t)H[MAXORD + 4 * q + 1] << wasted),
                              (int32_t)((uint32_t)H[MAXORD + 4 * q + 2] << wasted), (int32_t)((uint32_t)H[MAXORD + 4 * q + 3] << wasted));
        } else {
#pragma unroll
            for (int j = 0; j < kDecBatch; j++) dst[i + j] = (int32_t)((uint32_t)H[MAXORD + j] << wasted);
        }
    };
    auto single_sample = [&]() {
        const int32_t r = escape ? br.get_signed(raw_bits) : unzigzag(br.rice_u(k));
        int32_t v;
        if constexpr (WIDE) {
            const long long v64 = (long long)r + lpc_predict64<MAXORD>(cf, &H[MAXORD - 1], shift);
            v = (int32_t)v64;
            const long long vs = v64 << wasted;
            ovf |= (uint32_t)((int32_t)(vs >> 32) ^ ((int32_t)vs >> 31));
        } else {
            v = r + lpc_predict<MAXORD, WIDE>(cf, &H[MAXORD - 1], shift);
        }
#pragma unroll
        for (int q = 0; q < MAXORD - 1; q++) H[q] = H[q + 1];
        H[MAXORD - 1] = v;
        if (SINK == kSinkAudio) dst[i] = (int32_t)((uint32_t)v << wasted); else sink_one<SINK>(G, S.rp, (int32_t)((uint32_t)v << wasted));
        part_left--; i++;
        if (br.overrun()) { S.err = true; i = n; }
    };
    // (Tried in round 2, not kept: running the reader ONE BATCH AHEAD -- a trip parses batch b+1 speculatively and
    // reconstructs batch b in the same basic block, so that the Rice chain and the predictor chain interleave.  Same-box
    // A/B: C3 3.02 vs 3.04 ms, C5 3.39 vs 3.26 ms: the extra parse-only trip at every partition start and the rewind
    // selects cost what the interleaving gains.)
    while (__any_sync(0xFFFFFFFFu, i < n)) {
        if (i >= n) continue;
        br.top_up();
        bool did = false;
        if (!escape && part_left >= (uint32_t)kDecBatch && (i & 3u) == 0) {       // (i & 3): keep the 16-byte stores aligned
            // ---- batch: kDecBatch codes, no data-dependent branch; redone sample by sample if one is longer than 32 bits ----
            const DecReader snap = br;
            uint32_t u[kDecBatch];
            if (parse_batch(k, u) <= 32) {
                reconstruct(u);
                output_batch();
#pragma unroll
                for (int q = 0; q < MAXORD; q++) H[q] = H[q + kDecBatch];
                part_left -= kDecBatch; i += kDecBatch;
                did = true;
            } else {
                br = snap;
            }
        }
        if (!did) single_sample();
        if (part_left == 0 && i < n) {
            k = br.get(plen); escape = (k == esc); raw_bits = escape ? br.get(5) : 0; part_left = psize;
        }
    }
    if (WIDE && ovf) S.err = true;
}

#ifndef FRB_DEC_MINB
#define FRB_DEC_MINB 4
#endif
// Fused skim + decode.  The first `n_skim_ctas` CTAs (lowest block indices, dispatched first) walk the frames and
// publish subframe offsets as they go; the remaining CTAs decode one subframe per thread in CHANNEL-MAJOR order
// (all subframes 0, then all subframes 1, ...), each waiting for its offset.  The walk of a frame reaches channel c
// after c/(C-1) of its run time, so the decode of channel c overlaps the walk of channels c+1.. instead of
// starting when the whole skim kernel has drained (5.0 -> see DESIGN.md section 4 for the measured step).  Forward
// progress: skim CTAs never wait, and they are resident before any waiting CTA is dispatched (the same in-order
// dispatch assumption as a decoupled look-back scan); a waiting thread gives up after kSpinLimit polls (status[5]).
constexpr uint32_t kSpinLimit = 1u << 22;
#ifdef FRB_DEC_TIMING
__device__ unsigned long long g_dec_dbg[16];
#endif
template <bool BIGORDER, int SINK>
__global__ void __launch_bounds__(kDecThreads, BIGORDER ? 1 : FRB_DEC_MINB)
k_decode_subframes(const uint8_t *__restrict__ bytes, const DecStreamDev *__restrict__ streams, uint32_t n_streams,
                   uint32_t channels, uint32_t bps, uint32_t blocksize, uint32_t total_frames,
                   const unsigned long long *__restrict__ frame_pos, uint32_t *__restrict__ sub_bitoff,
                   int32_t *__restrict__ audio, uint8_t *__restrict__ frame_chassign, uint32_t *__restrict__ status,
                   uint32_t n_skim_ctas, uint32_t skim_lanes, const SinkCfg sink, uint32_t indexed) {
    // indexed != 0: sub_bitoff is a READ-ONLY table the caller supplied (the stream's seek index, frb_encode_index): there is
    // no skim role and nothing to wait for; every decode thread checks the frame header itself
    __shared__ __align__(256) uint4 s_ring[kSkimRing * kDecThreads];
#ifdef FRB_DEC_TIMING
    unsigned long long t_start; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_start));
    if (threadIdx.x == 0) atomicMin(&g_dec_dbg[0], t_start);
#endif
    if (blockIdx.x < n_skim_ctas) {
        skim_role(s_ring, blockIdx.x, bytes, streams, n_streams, channels, bps, blocksize, total_frames, frame_pos, sub_bitoff,
                  frame_chassign, status, skim_lanes);
#ifdef FRB_DEC_TIMING
        unsigned long long t_end; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_end));
        if (threadIdx.x == 0) atomicMax(&g_dec_dbg[1], t_end);
#endif
        return;
    }
    const uint32_t s = (blockIdx.x - n_skim_ctas) * blockDim.x + threadIdx.x;
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t total_sub = total_frames * channels;
    bool alive = s < total_sub;
    // channel-major: a warp holds 32 consecutive frames of ONE channel (similar predictor orders, and their offsets
    // are published by one skim warp at about the same time)
    const uint32_t c = alive ? s / total_frames : 0, f = alive ? s - c * total_frames : 0;
    SubCtx S;
    S.err = false; S.type = 0; S.order = 0; S.n = 0; S.wasted = 0; S.sbps = bps; S.dst = audio; S.aligned16 = false;
    S.rp.rowp = sink.raster; S.rp.x = 0; S.rp.w = 1; S.rp.y = S.rp.y0 = S.rp.y1 = S.rp.x0 = S.rp.x1 = 0; S.rp.pitch = 0; S.rp.mn = 0.0; S.rp.range = 0.0; S.rp.imn = 0; S.rp.irange = 0; S.rp.kround = 0;
    S.br.gq = (const uint4 *)bytes; S.br.sbase = (uint32_t)__cvta_generic_to_shared(s_ring + threadIdx.x * kSkimRing);
    S.br.swz = (lane & 15u) << 4; S.br.sx = S.br.sbase ^ S.br.swz; S.br.cissue = 0; S.br.qlast = 0;
    S.br.woff = 12; S.br.A = S.br.B = S.br.Craw = 0; S.br.bp = 0;
    FrameLoc L; L.ok = false; L.start = L.end = 0; L.k = 0; L.n = 0;
    uint32_t hdr_bytes = 0;
    if (alive) {
        DecStreamDev st;
        L = locate_frame(streams, n_streams, blocksize, f, frame_pos, &st);
        if (!L.ok) { alive = false; if (c == 0 && !sub_bitoff) atomicAdd(&status[0], 1u); }
        else {
            uint32_t ch_assign = 0;
            uint64_t bit0;
            if (sub_bitoff && !indexed) {
                const uint32_t *slot = sub_bitoff + (size_t)f * channels + c;
                uint32_t off = ld_acquire_u32(slot), spins = 0;
                while (off == kNotReady) {
                    __nanosleep(200);
                    off = ld_acquire_u32(slot);
                    if (++spins > kSpinLimit) { atomicAdd(&status[5], 1u); off = 0; }
                }
                if (off == 0) alive = false;               // the skim pass already counted the error
                bit0 = L.start * 8 + off;
                ch_assign = frame_chassign[f];
            } else {
                FrameHdr h;
                if (!parse_frame_header(bytes + L.start, L.end - L.start, 0, bps, &h)) { alive = false; if (c == 0) atomicAdd(&status[2], 1u); }
                else { hdr_bytes = h.header_bytes; ch_assign = h.ch_assign; if (c == 0) frame_chassign[f] = (uint8_t)h.ch_assign; }
                bit0 = (L.start + hdr_bytes) * 8;
                if (indexed && alive && sub_bitoff) {
                    const uint32_t off = sub_bitoff[(size_t)f * channels + c];
                    // the index must agree with the stream: subframe 0 starts right behind the header, the others inside the frame
                    if (c == 0 ? off != hdr_bytes * 8 : (off <= hdr_bytes * 8 || (uint64_t)off >= (L.end - L.start) * 8)) { alive = false; atomicAdd(&status[2], 1u); }
                    bit0 = L.start * 8 + off;
                }
            }
            if (alive) {
                S.br.init(S.br.sbase, lane, bytes, bit0, L.end);
                S.n = L.n;
                const int64_t idx = st.audio_base + (int64_t)c * (int64_t)st.n_samples + (int64_t)L.k * blocksize;
                S.dst = audio + idx;
                S.aligned16 = ((reinterpret_cast<uintptr_t>(S.dst) & 15u) == 0);
                if (SINK == kSinkWindow) {
                    const frb_tile t = sink.tiles[L.stream];
                    if ((uint64_t)t.h * t.w != st.total_samples || t.w == 0) {
                        if (c == 0 && L.k == 0) atomicAdd(&status[6], 1u);
                        alive = false;
                    }
                    const uint64_t i0 = (uint64_t)(st.first_frame + L.k) * blocksize;
                    const uint32_t y = t.w ? (uint32_t)(i0 / t.w) : 0u;
                    // the window in tile coordinates, clipped to the tile
                    const int64_t wy = (int64_t)sink.win_row - t.row_off, wx = (int64_t)sink.win_col - t.col_off;
                    auto clip = [](int64_t v, uint32_t hi) -> uint32_t { return (uint32_t)(v < 0 ? 0 : v > (int64_t)hi ? (int64_t)hi : v); };
                    S.rp.y = y; S.rp.y0 = clip(wy, t.h); S.rp.y1 = clip(wy + sink.H, t.h);
                    S.rp.x0 = clip(wx, t.w); S.rp.x1 = clip(wx + sink.W, t.w);
                    S.rp.x = (uint32_t)(i0 - (uint64_t)y * t.w); S.rp.w = t.w; S.rp.pitch = sink.W * sink.esize;
                    // row y of the tile, column 0 (outside the window unless its rows and columns are: only ever offset)
                    S.rp.rowp = sink.raster + (((int64_t)c * sink.H + (int64_t)y - wy) * (int64_t)sink.W - wx) * (int64_t)sink.esize;
                    const double mn = sink.minmax[2 * L.stream];
                    const double range = __dsub_rn(sink.minmax[2 * L.stream + 1], mn);
                    if (sink.intpath) { S.rp.imn = (int32_t)mn - 1; S.rp.irange = (uint32_t)range; S.rp.kround = 32767u * S.rp.irange + 32767u + 65534u; }
                    else { S.rp.mn = mn; S.rp.range = range; }
                } else if (SINK == kSinkTile) {
                    const frb_tile t = sink.tiles[L.stream];
                    // the stream must be exactly this tile's pixels and the window must lie inside the raster (status[6])
                    if ((uint64_t)t.h * t.w != st.n_samples || t.w == 0 || (uint64_t)t.row_off + t.h > sink.H || (uint64_t)t.col_off + t.w > sink.W) {
                        if (c == 0 && L.k == 0) atomicAdd(&status[6], 1u);
                        alive = false;
                    }
                    const uint32_t i0 = L.k * blocksize, y = i0 / t.w;
                    S.rp.x = i0 - y * t.w; S.rp.w = t.w; S.rp.pitch = sink.W * sink.esize;
                    S.rp.rowp = sink.raster + (((size_t)c * sink.H + t.row_off + y) * sink.W + t.col_off) * sink.esize;
                    const double mn = sink.minmax[2 * L.stream];
                    const double range = __dsub_rn(sink.minmax[2 * L.stream + 1], mn);    // max-min unconditionally (:239)
                    if (sink.intpath) { S.rp.imn = (int32_t)mn - 1; S.rp.irange = (uint32_t)range; S.rp.kround = 32767u * S.rp.irange + 32767u + 65534u; }
                    else { S.rp.mn = mn; S.rp.range = range; }
                }
                if ((ch_assign == 8 && c == 1) || (ch_assign == 9 && c == 0) || (ch_assign == 10 && c == 1)) S.sbps++;
                const uint32_t hd = S.br.get(8);
                if (hd & 0x80) S.err = true;
                const uint32_t t = (hd >> 1) & 0x3F;
                if (hd & 1) S.wasted = S.br.unary() + 1;
                if (S.wasted >= S.sbps) { S.err = true; S.wasted = 0; }
                S.sbps -= S.wasted;
                if (t == 0) S.type = 0;
                else if (t == 1) S.type = 1;
                else if (t >= 8 && t <= 12) { S.type = 2; S.order = t - 8; }
                else if (t >= 32) { S.type = 3; S.order = t - 31; }
                else S.err = true;
                if (S.order > S.n) S.err = true;
            }
        }
    }
    const bool run = alive && !S.err;
    if (run) {
        if (S.type == 0) {
            const int32_t v = shl_checked(S.br.get_signed(S.sbps, &S.err), S.wasted, S.err);
            if (SINK == kSinkAudio) { for (uint32_t i = 0; i < S.n; i++) S.dst[i] = v; }
            else { for (uint32_t i = 0; i < S.n; i++) sink_one<SINK>(sink, S.rp, v); }
        } else if (S.type == 1) {
            for (uint32_t i = 0; i < S.n; i++) {
                if ((i & 3u) == 0) S.br.top_up();
                const int32_t v = shl_checked(S.br.get_signed(S.sbps, &S.err), S.wasted, S.err);
                if (SINK == kSinkAudio) S.dst[i] = v; else sink_one<SINK>(sink, S.rp, v);
            }
        } else if (!BIGORDER && S.order > 12) {
            S.err = true;
            atomicAdd(&status[4], 1u);
        }
    }
    {
        constexpr int PMAX = BIGORDER ? 32 : 12;
        const bool act = run && S.type >= 2 && (BIGORDER || S.order <= 12);
        PredState<PMAX> P;
        decode_prologue<PMAX, SINK>(S, act, P, sink);
        // warp-uniform sample loop (it is warp-synchronous): taps padded to the largest order in the warp, 64-bit MACs
        // only if a lane needs them
        const uint32_t cls = __reduce_max_sync(0xFFFFFFFFu, act ? S.order : 0u);
        const bool wide = __any_sync(0xFFFFFFFFu, act && P.wide);
        if (BIGORDER) decode_predictive<32, true, PMAX, SINK>(S, P, sink);
        else if (cls <= 4) { if (wide) decode_predictive<4, true, PMAX, SINK>(S, P, sink); else decode_predictive<4, false, PMAX, SINK>(S, P, sink); }
        else if (cls <= 8) { if (wide) decode_predictive<8, true, PMAX, SINK>(S, P, sink); else decode_predictive<8, false, PMAX, SINK>(S, P, sink); }
        else { if (wide) decode_predictive<12, true, PMAX, SINK>(S, P, sink); else decode_predictive<12, false, PMAX, SINK>(S, P, sink); }
    }
#ifdef FRB_DEC_TIMING
    {
        unsigned long long t_end; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_end));
        if (threadIdx.x == 0) { atomicMax(&g_dec_dbg[2], t_end); atomicMax(&g_dec_dbg[3 + (c & 7)], t_end); atomicMin(&g_dec_dbg[11], t_start); }
    }
#endif
    if (alive) {
        if (!S.err && c + 1 == channels) {
            // the last subframe must end (after byte padding) exactly 2 bytes before the next frame
            const uint64_t bits = S.br.bitpos() - L.start * 8;
            if (L.start + ((bits + 7) >> 3) + 2 != L.end) S.err = true;
        } else if (!S.err && indexed && sub_bitoff) {
            // indexed streams: a subframe must end exactly where the index says the next one starts
            if (S.br.bitpos() - L.start * 8 != (uint64_t)sub_bitoff[(size_t)f * channels + c + 1]) S.err = true;
        }
        if (S.err) atomicAdd(&status[2], 1u);
        else if (c + 1 == channels) atomicAdd(&status[3], 1u);
    }
}

#include "frb_crc16.cuh"   // warp-cooperative CRC-16 + k_crc16_frames
