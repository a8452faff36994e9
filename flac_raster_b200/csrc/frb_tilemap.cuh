// frb_tilemap.cuh -- per-tile sample mapping kernels (min/max, normalise, denormalise) for a planar
// (bands,H,W) raster resident in HBM.  Reference: normalization.py:149-187 and :222-249, applied per tile
// as cli.py:553-594 does.
//
// These three kernels are pure HBM streams (algorithmic bytes per sample: sizeof(T), sizeof(T)+4, 4+sizeof(T)).
// v1 (profiles/r01_launches_c3_v1.csv) spent 3.8 / 2.6 / 4.2 ms on C3 where the HBM floor is ~0.3 / 0.9 /
// 0.9 ms: a runtime dtype switch and an integer division per element.  v2 (typed, one CTA per row, one
// element per thread and iteration, table gathers) still took 2.3 / 2.7 / 4.9 ms
// (profiles/r01_launches_c3_v3.csv): with 2-4 bytes per load and a dependent loop there were far too few
// bytes in flight per SM to cover DRAM latency.  v3 (this file):
//   * one WARP per (band,row) of the tile; the row is walked in 16-byte vectors of the raster type (aligned
//     head/tail handled by single lanes), four independent vectors in flight per lane;
//   * the int32 audio side is accessed with 16-byte vectors as well whenever the row is 16-byte aligned
//     (always for the BASELINE shapes), else with scalar accesses;
//   * normalise, 8/16-bit sources: per-tile exact table over the tile's value range [min,max] (when it
//     spans fewer than kNormLutCap values), entry = normalize_one(value), so the fp64 pipe is idle;
//     everything else is computed directly with the reference's fp64 operation order.
#pragma once
#include "frb_normalize.cuh"

namespace frb {

constexpr uint32_t kNormLutCap = 16384;      // per-tile normalise table entries (int32)
constexpr int kMapThreads = 256;
constexpr int kMapWarps = kMapThreads / 32;

struct MapWorkspace {
    int32_t *norm_lut;       // n_tiles * kNormLutCap
};
static inline size_t map_ws_layout(uint32_t n_tiles, void *base, MapWorkspace *w) {
    size_t off = 0;
    uint8_t *b = (uint8_t *)base;
    if (w) w->norm_lut = (int32_t *)(b + off);
    off += (size_t)n_tiles * kNormLutCap * 4;
    return off + 256;
}

template <typename T> struct is_small_int { static constexpr bool value = false; };
template <> struct is_small_int<uint8_t> { static constexpr bool value = true; };
template <> struct is_small_int<int8_t> { static constexpr bool value = true; };
template <> struct is_small_int<uint16_t> { static constexpr bool value = true; };
template <> struct is_small_int<int16_t> { static constexpr bool value = true; };
template <typename T> struct is_fp { static constexpr bool value = false; };
template <> struct is_fp<float> { static constexpr bool value = true; };
template <> struct is_fp<double> { static constexpr bool value = true; };

// A group of G consecutive elements: the unit of the row walk.  G*sizeof(T) and G*4 are multiples of 16.
template <typename T> struct MapGroup {
    static constexpr int G = (16 / sizeof(T)) > 4 ? (16 / sizeof(T)) : 4;
    static constexpr int TV = G * sizeof(T) / 16;     // 16-byte vectors on the raster side
    static constexpr int AV = G * 4 / 16;             // 16-byte vectors on the int32 audio side
};

__device__ __forceinline__ uint4 ld_stream16(const void *p) { return __ldcs(reinterpret_cast<const uint4 *>(p)); }
__device__ __forceinline__ void st_stream16(void *p, uint4 v) { __stcs(reinterpret_cast<uint4 *>(p), v); }

template <typename T>
__device__ __forceinline__ void load_group(const T *p, T (&e)[MapGroup<T>::G]) {
    union { uint4 v[MapGroup<T>::TV]; T e[MapGroup<T>::G]; } u;
#pragma unroll
    for (int q = 0; q < MapGroup<T>::TV; q++) u.v[q] = ld_stream16(reinterpret_cast<const uint8_t *>(p) + 16 * q);
#pragma unroll
    for (int j = 0; j < MapGroup<T>::G; j++) e[j] = u.e[j];
}
// the same in two steps: the vectors as loaded (what a look-ahead buffer should hold: 4 registers per 16 bytes, whatever
// the element size), unpacked when they are used
template <typename T>
__device__ __forceinline__ void load_group_raw(const T *p, uint4 (&v)[MapGroup<T>::TV]) {
#pragma unroll
    for (int q = 0; q < MapGroup<T>::TV; q++) v[q] = ld_stream16(reinterpret_cast<const uint8_t *>(p) + 16 * q);
}
template <typename T>
__device__ __forceinline__ void unpack_group(const uint4 (&v)[MapGroup<T>::TV], T (&e)[MapGroup<T>::G]) {
    union { uint4 v[MapGroup<T>::TV]; T e[MapGroup<T>::G]; } u;
#pragma unroll
    for (int q = 0; q < MapGroup<T>::TV; q++) u.v[q] = v[q];
#pragma unroll
    for (int j = 0; j < MapGroup<T>::G; j++) e[j] = u.e[j];
}
template <typename T>
__device__ __forceinline__ void store_group(T *p, const T (&e)[MapGroup<T>::G]) {
    union { uint4 v[MapGroup<T>::TV]; T e[MapGroup<T>::G]; } u;
#pragma unroll
    for (int j = 0; j < MapGroup<T>::G; j++) u.e[j] = e[j];
#pragma unroll
    for (int q = 0; q < MapGroup<T>::TV; q++) st_stream16(reinterpret_cast<uint8_t *>(p) + 16 * q, u.v[q]);
}

// Row geometry shared by the three kernels: elements [0,head) and [tail0,w) are handled one per lane,
// groups g in [0,ngroups) start at element head + g*G (16-byte aligned on the raster side).
template <typename T>
struct RowSplit {
    uint32_t head, ngroups, tail0;
    __device__ __forceinline__ RowSplit(const T *row, uint32_t w) {
        constexpr uint32_t G = MapGroup<T>::G;
        uint32_t h = (uint32_t)(((16u - (uint32_t)(reinterpret_cast<uintptr_t>(row) & 15u)) & 15u) / sizeof(T));
        head = h < w ? h : w;
        ngroups = (w - head) / G;
        tail0 = head + ngroups * G;
    }
};

// ---------------------------------------------------------------- min/max
template <typename T>
__global__ void __launch_bounds__(kMapThreads)
k_minmax_tiles(const T *__restrict__ raster, uint32_t bands, uint32_t H, uint32_t W,
               const frb_tile *__restrict__ tiles, unsigned long long *keys, uint32_t parts) {
    constexpr int G = MapGroup<T>::G;
    // flattened grid: `parts` CTAs per tile (the tile index must not sit in gridDim.y, which stops at 65535)
    const uint32_t tile_i = blockIdx.x / parts, part = blockIdx.x - tile_i * parts;
    const frb_tile t = tiles[tile_i];
    const uint32_t rows = bands * t.h;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    bool any = false;
    T mn = T(0), mx = T(0);
    auto take = [&](T v) {
        if (is_fp<T>::value && v != v) return;
        if (!any) { mn = mx = v; any = true; }
        else { mn = v < mn ? v : mn; mx = v > mx ? v : mx; }
    };
    // 16-bit rasters: the vector body runs on packed halves (VIMNMX.U16x2 / .S16x2: one instruction per two pixels and
    // bound).  Element by element the kernel was ALU-bound (69 % ALU pipe at 51 % of the DRAM rate, 0.46 ms per C3 scene).
    constexpr bool PACK16 = sizeof(T) == 2 && is_small_int<T>::value;
    constexpr bool SGN = (T)(-1) < (T)0;
    uint32_t pmn = SGN ? 0x7FFF7FFFu : 0xFFFFFFFFu, pmx = SGN ? 0x80008000u : 0u;
    bool pany = false;
    auto take_vec = [&](const uint4 &v) {
        if (SGN) {
            pmn = __vmins2(__vmins2(pmn, v.x), __vmins2(v.y, __vmins2(v.z, v.w)));
            pmx = __vmaxs2(__vmaxs2(pmx, v.x), __vmaxs2(v.y, __vmaxs2(v.z, v.w)));
        } else {
            pmn = __vminu2(__vminu2(pmn, v.x), __vminu2(v.y, __vminu2(v.z, v.w)));
            pmx = __vmaxu2(__vmaxu2(pmx, v.x), __vmaxu2(v.y, __vmaxu2(v.z, v.w)));
        }
    };
    for (uint32_t ry = part * kMapWarps + warp; ry < rows; ry += parts * kMapWarps) {
        const uint32_t c = ry / t.h, y = ry - c * t.h;
        const T *src = raster + ((size_t)c * H + (t.row_off + y)) * W + t.col_off;
        const RowSplit<T> rs(src, t.w);
        if ((uint32_t)lane < rs.head) take(src[lane]);
        if (rs.tail0 + lane < t.w) take(src[rs.tail0 + lane]);
        const T *body = src + rs.head;
        uint32_t g = lane;
        if constexpr (PACK16) {
            if (g < rs.ngroups) pany = true;
            for (; g + 96 < rs.ngroups; g += 128) {
                const uint4 v0 = ld_stream16(body + (size_t)g * G), v1 = ld_stream16(body + (size_t)(g + 32) * G),
                            v2 = ld_stream16(body + (size_t)(g + 64) * G), v3 = ld_stream16(body + (size_t)(g + 96) * G);
                take_vec(v0); take_vec(v1); take_vec(v2); take_vec(v3);
            }
            for (; g < rs.ngroups; g += 32) take_vec(ld_stream16(body + (size_t)g * G));
        } else {
            for (; g + 96 < rs.ngroups; g += 128) {
                T e0[G], e1[G], e2[G], e3[G];
                load_group(body + (size_t)g * G, e0);
                load_group(body + (size_t)(g + 32) * G, e1);
                load_group(body + (size_t)(g + 64) * G, e2);
                load_group(body + (size_t)(g + 96) * G, e3);
#pragma unroll
                for (int j = 0; j < G; j++) { take(e0[j]); take(e1[j]); take(e2[j]); take(e3[j]); }
            }
            for (; g < rs.ngroups; g += 32) {
                T e0[G];
                load_group(body + (size_t)g * G, e0);
#pragma unroll
                for (int j = 0; j < G; j++) take(e0[j]);
            }
        }
    }
    if (PACK16 && pany) { take((T)(pmn & 0xFFFFu)); take((T)(pmn >> 16)); take((T)(pmx & 0xFFFFu)); take((T)(pmx >> 16)); }
    block_minmax_commit(any ? dkey((double)mn) : kKeyMinInit, any ? dkey((double)mx) : kKeyMaxInit, keys + 2 * (size_t)tile_i);
}

// ---------------------------------------------------------------- normalise
__global__ void __launch_bounds__(256)
k_build_norm_lut(const double *__restrict__ minmax, int bits, int32_t *__restrict__ lut, uint32_t parts) {
    const uint32_t tile_i = blockIdx.x / parts, part = blockIdx.x - tile_i * parts;
    // 16-bit audio: entries are stored as int16 in the same buffer (half the cache sectors per warp-wide gather)
    int16_t *lut16 = reinterpret_cast<int16_t *>(lut);
    const double mn = minmax[2 * tile_i], mx = minmax[2 * tile_i + 1];
    if (!(mx - mn < (double)kNormLutCap)) return;          // also false for NaN: those tiles use the direct path
    const double range = (mx <= mn) ? 1.0 : __dsub_rn(mx, mn);
    const double scale = scale_for_bits(bits);
    const uint32_t cnt = (uint32_t)(mx - mn) + 1;
    const size_t base = (size_t)tile_i * kNormLutCap;
    for (uint32_t j = part * blockDim.x + threadIdx.x; j < cnt; j += parts * blockDim.x) {
        const int32_t v = normalize_one(__dadd_rn(mn, (double)j), mn, range, scale);     // mn + j is exact (small integers)
        if (bits == 16) lut16[base + j] = (int16_t)v; else lut[base + j] = v;
    }
}

// A: element type of the planar audio (int32_t, or int16_t for 16-bit audio of 8/16-bit rasters: half the bytes written
// here and half the bytes both analysis kernels read back; G * sizeof(A) stays a multiple of 16 for those types)
// SLUT (int16 audio only): the CTA copies its tile's table into shared memory first (at most 32 KB) and gathers from
// there.  Round 2 measured the global-memory gathers at 1.40 ms per C3 scene for 3.9 GB of traffic (2.8 TB/s, 24
// instructions per sample, 64-bit address arithmetic and an L1 tag lookup per distinct line of every gather); round 1
// had rejected a shared-memory table because the int32 table of the time took 64 KB per CTA.
#ifndef FRB_NORM_MINB
#define FRB_NORM_MINB 4
#endif
template <typename T, typename A, bool SLUT = false>
__global__ void __launch_bounds__(kMapThreads, (sizeof(T) <= 2 && sizeof(A) == 2) ? FRB_NORM_MINB : 3)
k_normalize_tiles(const T *__restrict__ raster, uint32_t bands, uint32_t H, uint32_t W,
                  const frb_tile *__restrict__ tiles, const double *__restrict__ minmax, int bits,
                  A *__restrict__ audio, const int64_t *__restrict__ audio_base,
                  const int32_t *__restrict__ lut_all, uint32_t parts) {
    constexpr int G = MapGroup<T>::G, AV = G * (int)sizeof(A) / 16;
    static_assert(sizeof(A) == 4 || (G * sizeof(A)) % 16 == 0, "int16 audio needs 8 or 16 elements per group");
    static_assert(!SLUT || (sizeof(A) == 2 && is_small_int<T>::value), "shared-memory table: 8/16-bit rasters, int16 audio");
    extern __shared__ __align__(16) int16_t s_lut[];
    const uint32_t tile_i = blockIdx.x / parts, part = blockIdx.x - tile_i * parts;
    const frb_tile t = tiles[tile_i];
    const uint32_t n = t.h * t.w;
    const double mn = minmax[2 * tile_i], mx = minmax[2 * tile_i + 1];
    const double range = (mx <= mn) ? 1.0 : __dsub_rn(mx, mn);
    const double scale = scale_for_bits(bits);
    A *dst = audio + audio_base[tile_i];
    const uint32_t rows = bands * t.h;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool use_lut = is_small_int<T>::value && lut_all != nullptr && (mx - mn < (double)kNormLutCap);
    const int32_t vmin = use_lut ? (int32_t)mn : 0;
    // (staging the table in shared memory was tried: 64 KB per CTA costs more occupancy than the L1 gathers cost)
    const int32_t *lut = lut_all ? lut_all + (size_t)tile_i * kNormLutCap : nullptr;
    if (SLUT) {
        if (use_lut) {        // uniform over the CTA; whole 16-byte chunks (the tile's table region is kNormLutCap entries long)
            const uint32_t chunks = ((uint32_t)(mx - mn) + 1 + 7) / 8;
            const uint4 *g = reinterpret_cast<const uint4 *>(reinterpret_cast<const int16_t *>(lut_all) + (size_t)tile_i * kNormLutCap);
            for (uint32_t q = threadIdx.x; q < chunks; q += kMapThreads) reinterpret_cast<uint4 *>(s_lut)[q] = __ldg(g + q);
        }
        __syncthreads();
    }
    const int16_t *s_tab = s_lut - vmin;         // table indexed by the pixel value itself
    // the row walk is instantiated once per mapping, so the table path carries no per-sample test of `use_lut`
    // (with the test inside the mapping, every gather was followed by a branch around the inlined fp64 formula)
    auto walk = [&](auto map) {
        const uint32_t stride = parts * kMapWarps;
        // (band, row) of the current and of the next visited row, stepped without a division per row
        uint32_t cc = (part * kMapWarps + warp) / t.h, cy = (part * kMapWarps + warp) - cc * t.h, nc = cc, ny = cy;
        auto step = [&](uint32_t &c, uint32_t &y) { y += stride; while (y >= t.h) { y -= t.h; c++; } };
        step(nc, ny);
        auto row_src = [&](uint32_t c, uint32_t y) -> const T * { return raster + ((size_t)c * H + (t.row_off + y)) * W + t.col_off; };
        // The first 128 groups of a row (the whole row for tiles up to 1024 16-bit / 2048 8-bit pixels wide) are loaded one
        // row AHEAD: a warp alternated between waiting for its four loads and mapping them, so little was in flight while it
        // mapped (1.06 ms per C3 scene for 3.9 GB with the table already in shared memory).
        constexpr int TV = MapGroup<T>::TV;
        uint4 E[4][TV], En[4][TV];
        auto prefetch = [&](uint32_t c, uint32_t y, uint4 (&B)[4][TV]) {
            const T *src = row_src(c, y);
            const RowSplit<T> rs(src, t.w);
#pragma unroll
            for (int k = 0; k < 4; k++)
                if (lane + 32u * k < rs.ngroups) load_group_raw<T>(src + rs.head + (size_t)(lane + 32u * k) * G, B[k]);
        };
        // (only the int16-audio instantiations look ahead: the others are bound by their fp64 formula or by 4-byte audio
        // stores, and the two vector buffers cost them occupancy -- float32 74 -> 100 registers, C4's mapping 3.0 -> 5.0 ms)
        constexpr bool AHEAD = sizeof(A) == 2;
        uint32_t ry = part * kMapWarps + warp;
        if (AHEAD && ry < rows) prefetch(cc, cy, E);
        for (; ry < rows; ry += stride, cc = nc, cy = ny, step(nc, ny)) {
            if (AHEAD && ry + stride < rows) prefetch(nc, ny, En);
            const uint32_t c = cc, y = cy;
            const T *src = row_src(c, y);
            A *out = dst + (size_t)c * n + (size_t)y * t.w;
            const RowSplit<T> rs(src, t.w);
            if ((uint32_t)lane < rs.head) out[lane] = (A)map(src[lane]);
            if (rs.tail0 + lane < t.w) out[rs.tail0 + lane] = (A)map(src[rs.tail0 + lane]);
            const T *body = src + rs.head;
            A *obody = out + rs.head;
            const bool ovec = (reinterpret_cast<uintptr_t>(obody) & 15u) == 0;
            auto emit = [&](uint32_t g, const T (&e)[G]) {
                int32_t r[G];
#pragma unroll
                for (int j = 0; j < G; j++) r[j] = map(e[j]);
                A *o = obody + (size_t)g * G;
                if (ovec) {
                    if (sizeof(A) == 4) {
#pragma unroll
                        for (int q = 0; q < AV; q++)
                            st_stream16(o + 4 * q, make_uint4((uint32_t)r[4 * q], (uint32_t)r[4 * q + 1], (uint32_t)r[4 * q + 2], (uint32_t)r[4 * q + 3]));
                    } else {
                        auto pk = [&](int j) { return __byte_perm((uint32_t)r[j], (uint32_t)r[j + 1], 0x5410); };   // two int16 per word
#pragma unroll
                        for (int q = 0; q < AV; q++)
                            st_stream16(o + 8 * q, make_uint4(pk(8 * q), pk(8 * q + 2), pk(8 * q + 4), pk(8 * q + 6)));
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < G; j++) o[j] = (A)r[j];
                }
            };
            if (AHEAD) {
#pragma unroll
                for (int k = 0; k < 4; k++)
                    if (lane + 32u * k < rs.ngroups) {
                        T e[G];
                        unpack_group<T>(E[k], e);
                        emit(lane + 32u * k, e);
                    }
            }
            uint32_t g = lane + (AHEAD ? 128u : 0u);                                      // wider rows: the rest without look-ahead, four loads in flight
            for (; g + 96 < rs.ngroups; g += 128) {
                T e0[G], e1[G], e2[G], e3[G];
                load_group(body + (size_t)g * G, e0);
                load_group(body + (size_t)(g + 32) * G, e1);
                load_group(body + (size_t)(g + 64) * G, e2);
                load_group(body + (size_t)(g + 96) * G, e3);
                emit(g, e0); emit(g + 32, e1); emit(g + 64, e2); emit(g + 96, e3);
            }
            for (; g < rs.ngroups; g += 32) {
                T e0[G];
                load_group(body + (size_t)g * G, e0);
                emit(g, e0);
            }
            if (AHEAD) {
#pragma unroll
                for (int k = 0; k < 4; k++)
#pragma unroll
                    for (int q = 0; q < TV; q++) E[k][q] = En[k][q];
            }
        }
    };
    if (is_small_int<T>::value && use_lut) {
        if (SLUT) walk([&](T v) -> int32_t { return (int32_t)s_tab[(int32_t)v]; });
        else if (bits == 16) {
            const int16_t *tab = reinterpret_cast<const int16_t *>(lut_all) + (size_t)tile_i * kNormLutCap - vmin;
            walk([&](T v) -> int32_t { return (int32_t)__ldg(tab + (int32_t)v); });
        } else {
            const int32_t *tab = lut - vmin;
            walk([&](T v) -> int32_t { return __ldg(tab + (int32_t)v); });
        }
    } else {
        walk([&](T v) -> int32_t { return normalize_one((double)v, mn, range, scale); });
    }
}

// ---------------------------------------------------------------- denormalise
template <typename T> __device__ __forceinline__ T denorm_cast(double v) { return cast_round_out<T>(v); }
template <> __device__ __forceinline__ float denorm_cast<float>(double v) { return __double2float_rn(v); }
template <> __device__ __forceinline__ double denorm_cast<double>(double v) { return v; }

template <typename T>
__global__ void __launch_bounds__(kMapThreads)
k_denormalize_tiles(const int32_t *__restrict__ audio, const int64_t *__restrict__ audio_base,
                    const frb_tile *__restrict__ tiles, const double *__restrict__ minmax, double scale,
                    T *__restrict__ raster, uint32_t bands, uint32_t H, uint32_t W, uint32_t parts) {
    constexpr int G = MapGroup<T>::G, AV = MapGroup<T>::AV;
    const uint32_t tile_i = blockIdx.x / parts, part = blockIdx.x - tile_i * parts;
    const frb_tile t = tiles[tile_i];
    const uint32_t n = t.h * t.w;
    const double mn = minmax[2 * tile_i], mx = minmax[2 * tile_i + 1];
    const double range = __dsub_rn(mx, mn);                 // denormalize uses max-min unconditionally (:239)
    const int32_t *src = audio + audio_base[tile_i];
    const uint32_t rows = bands * t.h;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // the three scales the reference uses take the exact constant-division shortcut (see div_by_scale)
    const bool fast = scale == 32767.0 || scale == 8388607.0 || scale == 2147483647.0;
    const double rcp = __drcp_rn(scale);
    auto map = [&](int32_t a) -> T {
        return denorm_cast<T>(fast ? denormalize_one_fast((double)a, scale, rcp, mn, range) : denormalize_one((double)a, scale, mn, range));
    };
    for (uint32_t ry = part * kMapWarps + warp; ry < rows; ry += parts * kMapWarps) {
        const uint32_t c = ry / t.h, y = ry - c * t.h;
        T *out = raster + ((size_t)c * H + (t.row_off + y)) * W + t.col_off;
        const int32_t *in = src + (size_t)c * n + (size_t)y * t.w;
        const RowSplit<T> rs(out, t.w);
        if ((uint32_t)lane < rs.head) out[lane] = map(in[lane]);
        if (rs.tail0 + lane < t.w) out[rs.tail0 + lane] = map(in[rs.tail0 + lane]);
        T *obody = out + rs.head;
        const int32_t *ibody = in + rs.head;
        const bool ivec = (reinterpret_cast<uintptr_t>(ibody) & 15u) == 0;
        auto fetch = [&](uint32_t g, int32_t (&a)[G]) {
            const int32_t *p = ibody + (size_t)g * G;
            if (ivec) {
#pragma unroll
                for (int q = 0; q < AV; q++) {
                    const uint4 v = ld_stream16(p + 4 * q);
                    a[4 * q] = (int32_t)v.x; a[4 * q + 1] = (int32_t)v.y; a[4 * q + 2] = (int32_t)v.z; a[4 * q + 3] = (int32_t)v.w;
                }
            } else {
#pragma unroll
                for (int j = 0; j < G; j++) a[j] = __ldcs(p + j);
            }
        };
        auto emit = [&](uint32_t g, const int32_t (&a)[G]) {
            T e[G];
#pragma unroll
            for (int j = 0; j < G; j++) e[j] = map(a[j]);
            store_group(obody + (size_t)g * G, e);
        };
        uint32_t g = lane;
        for (; g + 32 < rs.ngroups; g += 64) {
            int32_t a0[G], a1[G];
            fetch(g, a0); fetch(g + 32, a1);
            emit(g, a0); emit(g + 32, a1);
        }
        for (; g < rs.ngroups; g += 32) {
            int32_t a0[G];
            fetch(g, a0);
            emit(g, a0);
        }
    }
}

// The window read's gather (frb_denormalize_window): audio of frame runs (frb_decode_window, dtype -1) -> the part of every
// tile that lies inside the window.  `parts` CTAs per tile, a warp per (band, visible row), a thread per group of G
// pixels; the same per-sample mapping as k_denormalize_tiles.
template <typename T>
__global__ void __launch_bounds__(kMapThreads)
k_denormalize_window(const int32_t *__restrict__ audio, const frb_window_stream *__restrict__ streams, uint32_t blocksize,
                     const frb_tile *__restrict__ tiles, const double *__restrict__ minmax, double scale, frb_tile win,
                     T *__restrict__ out_all, uint32_t bands, uint32_t parts) {
    constexpr int G = MapGroup<T>::G;
    const uint32_t tile_i = blockIdx.x / parts, part = blockIdx.x - tile_i * parts;
    const frb_tile t = tiles[tile_i];
    const frb_window_stream st = streams[tile_i];
    // visible rows / columns in tile coordinates
    const int64_t wy = (int64_t)win.row_off - t.row_off, wx = (int64_t)win.col_off - t.col_off;
    auto clip = [](int64_t v, uint32_t hi) -> uint32_t { return (uint32_t)(v < 0 ? 0 : v > (int64_t)hi ? (int64_t)hi : v); };
    const uint32_t y0 = clip(wy, t.h), y1 = clip(wy + win.h, t.h), x0 = clip(wx, t.w), x1 = clip(wx + win.w, t.w);
    if (y0 >= y1 || x0 >= x1) return;
    const uint64_t s0 = (uint64_t)st.first_frame * blocksize, s1 = (uint64_t)(st.first_frame + st.n_frames) * blocksize;
    const uint64_t run_n = (s1 < st.total_samples ? s1 : st.total_samples) - s0;
    const double mn = minmax[2 * tile_i], mx = minmax[2 * tile_i + 1];
    const double range = __dsub_rn(mx, mn);
    const bool fast = scale == 32767.0 || scale == 8388607.0 || scale == 2147483647.0;
    const double rcp = __drcp_rn(scale);
    auto map = [&](int32_t a) -> T {
        return denorm_cast<T>(fast ? denormalize_one_fast((double)a, scale, rcp, mn, range) : denormalize_one((double)a, scale, mn, range));
    };
    const uint32_t vh = y1 - y0, vw = x1 - x0, rows = bands * vh;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint32_t ry = part * kMapWarps + warp; ry < rows; ry += parts * kMapWarps) {
        const uint32_t c = ry / vh, y = y0 + (ry - c * vh);
        T *out = out_all + ((size_t)c * win.h + (size_t)((int64_t)y - wy)) * win.w + (size_t)((int64_t)x0 - wx);
        const int32_t *in = audio + st.audio_base + (int64_t)((size_t)c * run_n + ((uint64_t)y * t.w + x0 - s0));
        const RowSplit<T> rs(out, vw);
        if ((uint32_t)lane < rs.head) out[lane] = map(in[lane]);
        if (rs.tail0 + lane < vw) out[rs.tail0 + lane] = map(in[rs.tail0 + lane]);
        T *obody = out + rs.head;
        const int32_t *ibody = in + rs.head;
        for (uint32_t g = lane; g < rs.ngroups; g += 32) {
            T e[G];
#pragma unroll
            for (int j = 0; j < G; j++) e[j] = map(__ldcs(ibody + (size_t)g * G + j));
            store_group(obody + (size_t)g * G, e);
        }
    }
}

static inline uint32_t tile_grid_parts(uint32_t n_tiles, uint32_t max_rows) {
    // ~16 CTAs per SM in total, but never more CTAs per tile than it has (band,row) groups of kMapWarps
    uint32_t per_tile = (kNumSMs * 16 + n_tiles - 1) / n_tiles;
    const uint32_t cap = (max_rows + kMapWarps - 1) / kMapWarps;
    if (per_tile > cap) per_tile = cap;
    if (per_tile < 1) per_tile = 1;
    return per_tile;
}

#define FRB_DISPATCH_DTYPE(dtype, CALL)                                   \
    switch (dtype) {                                                      \
        case FRB_U8:  { using T = uint8_t;  CALL; } break;                \
        case FRB_I8:  { using T = int8_t;   CALL; } break;                \
        case FRB_U16: { using T = uint16_t; CALL; } break;                \
        case FRB_I16: { using T = int16_t;  CALL; } break;                \
        case FRB_U32: { using T = uint32_t; CALL; } break;                \
        case FRB_I32: { using T = int32_t;  CALL; } break;                \
        case FRB_F32: { using T = float;    CALL; } break;                \
        default:      { using T = double;   CALL; } break;                \
    }

}  // namespace frb

extern "C" int frb_sample_map_workspace_size(uint32_t n_tiles, size_t *bytes) {
    if (!bytes || !n_tiles) return FRB_ERR_INVALID_ARG;
    *bytes = frb::map_ws_layout(n_tiles, nullptr, nullptr);
    return FRB_OK;
}

extern "C" int frb_minmax_tiles(const void *d_raster, int dtype, uint32_t bands, uint32_t H, uint32_t W,
                                const frb_tile *d_tiles, uint32_t n_tiles, double *d_minmax, void *stream) {
    using namespace frb;
    if (!d_raster || !d_tiles || !d_minmax || dtype < 0 || dtype > FRB_F64 || !bands || !n_tiles) return FRB_ERR_INVALID_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    k_minmax_init<<<(n_tiles + 255) / 256, 256, 0, s>>>((unsigned long long *)d_minmax, n_tiles);
    FRB_LAUNCH_CHECK("k_minmax_init");
    const uint32_t parts = tile_grid_parts(n_tiles, bands * H), grid = parts * n_tiles;
    FRB_DISPATCH_DTYPE(dtype, (k_minmax_tiles<T><<<grid, kMapThreads, 0, s>>>((const T *)d_raster, bands, H, W, d_tiles, (unsigned long long *)d_minmax, parts)));
    FRB_LAUNCH_CHECK("k_minmax_tiles");
    k_minmax_finish<<<(n_tiles + 255) / 256, 256, 0, s>>>((unsigned long long *)d_minmax, n_tiles);
    FRB_LAUNCH_CHECK("k_minmax_finish");
    return FRB_OK;
}

extern "C" int frb_normalize_tiles(const void *d_raster, int dtype, uint32_t bands, uint32_t H, uint32_t W,
                                   const frb_tile *d_tiles, uint32_t n_tiles, const double *d_minmax,
                                   int bits_per_sample, int32_t *d_audio, const int64_t *d_audio_base,
                                   void *d_workspace, size_t workspace_bytes, void *stream) {
    using namespace frb;
    if (!d_raster || !d_tiles || !d_minmax || !d_audio || !d_audio_base || dtype < 0 || dtype > FRB_F64 || !bands || !n_tiles)
        return FRB_ERR_INVALID_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    const int32_t *lut = nullptr;
    if (d_workspace && dtype <= FRB_I16) {
        MapWorkspace w;
        if (map_ws_layout(n_tiles, d_workspace, &w) > workspace_bytes) return FRB_ERR_OVERFLOW;
        k_build_norm_lut<<<8 * n_tiles, 256, 0, s>>>(d_minmax, bits_per_sample, w.norm_lut, 8);
        FRB_LAUNCH_CHECK("k_build_norm_lut");
        lut = w.norm_lut;
    }
    const uint32_t parts = tile_grid_parts(n_tiles, bands * H), grid = parts * n_tiles;
    FRB_DISPATCH_DTYPE(dtype, (k_normalize_tiles<T, int32_t><<<grid, kMapThreads, 0, s>>>((const T *)d_raster, bands, H, W, d_tiles, d_minmax,
                                                                                                bits_per_sample, d_audio, d_audio_base, lut, parts)));
    FRB_LAUNCH_CHECK("k_normalize_tiles");
    return FRB_OK;
}

// The same mapping with int16 audio elements: 8/16-bit rasters at 16 bits per sample only (the tile path of the
// BASELINE configs C2, C3 and C5).  Consumed by frb_encode_analyse with FRB_ENC_AUDIO_I16 set in params.reserved.
extern "C" int frb_normalize_tiles_i16(const void *d_raster, int dtype, uint32_t bands, uint32_t H, uint32_t W,
                                       const frb_tile *d_tiles, uint32_t n_tiles, const double *d_minmax,
                                       int16_t *d_audio, const int64_t *d_audio_base,
                                       void *d_workspace, size_t workspace_bytes, void *stream) {
    using namespace frb;
    if (!d_raster || !d_tiles || !d_minmax || !d_audio || !d_audio_base || dtype < 0 || dtype > FRB_I16 || !bands || !n_tiles)
        return FRB_ERR_INVALID_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    const int32_t *lut = nullptr;
    if (d_workspace) {
        MapWorkspace w;
        if (map_ws_layout(n_tiles, d_workspace, &w) > workspace_bytes) return FRB_ERR_OVERFLOW;
        k_build_norm_lut<<<8 * n_tiles, 256, 0, s>>>(d_minmax, 16, w.norm_lut, 8);
        FRB_LAUNCH_CHECK("k_build_norm_lut");
        lut = w.norm_lut;
    }
    const uint32_t parts = tile_grid_parts(n_tiles, bands * H), grid = parts * n_tiles;
#define FRB_NORM16(T) do { if (lut) k_normalize_tiles<T, int16_t, true><<<grid, kMapThreads, kNormLutCap * 2, s>>>((const T *)d_raster, bands, H, W, d_tiles, d_minmax, 16, d_audio, d_audio_base, lut, parts); \
                           else k_normalize_tiles<T, int16_t, false><<<grid, kMapThreads, 0, s>>>((const T *)d_raster, bands, H, W, d_tiles, d_minmax, 16, d_audio, d_audio_base, lut, parts); } while (0)
    switch (dtype) {
        case FRB_U8: FRB_NORM16(uint8_t); break;
        case FRB_I8: FRB_NORM16(int8_t); break;
        case FRB_U16: FRB_NORM16(uint16_t); break;
        default: FRB_NORM16(int16_t); break;
    }
#undef FRB_NORM16
    FRB_LAUNCH_CHECK("k_normalize_tiles");
    return FRB_OK;
}

extern "C" int frb_denormalize_tiles(const int32_t *d_audio, const int64_t *d_audio_base,
                                     const frb_tile *d_tiles, uint32_t n_tiles, const double *d_minmax,
                                     double scale, void *d_raster, int dtype, uint32_t bands, uint32_t H,
                                     uint32_t W, void *d_workspace, size_t workspace_bytes, void *stream) {
    using namespace frb;
    (void)d_workspace; (void)workspace_bytes;       // the denormalise direction needs no tables
    if (!d_raster || !d_tiles || !d_minmax || !d_audio || !d_audio_base || dtype < 0 || dtype > FRB_F64 || !bands || !n_tiles)
        return FRB_ERR_INVALID_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    const uint32_t parts = tile_grid_parts(n_tiles, bands * H), grid = parts * n_tiles;
    FRB_DISPATCH_DTYPE(dtype, (k_denormalize_tiles<T><<<grid, kMapThreads, 0, s>>>(d_audio, d_audio_base, d_tiles, d_minmax, scale,
                                                                                  (T *)d_raster, bands, H, W, parts)));
    FRB_LAUNCH_CHECK("k_denormalize_tiles");
    return FRB_OK;
}
