// frb_host.cuh -- host-buffer entry points (the e2e path) and the libFLAC-shaped handle API.
//
// frb_host_encode / frb_host_decode are what the Python StreamEncoder /
// FileDecoder shims call through ctypes with numpy (host) buffers: H2D copy,
// kernels, D2H copy, all inside the call.  The frb_stream_encoder_* functions
// mirror the FLAC__stream_encoder_* calls pyflac's cffi layer makes
// (docs/sonos-pyflac.txt:2200-2212, :1994-1997, :2003-2014).
#pragma once
#include "frb_common.cuh"
#include <vector>
#include <string>
#include <string.h>

namespace frb {

// grow-only device / pinned scratch, one set per host thread
struct Scratch {
    void *ptr = nullptr; size_t cap = 0; bool pinned = false;
    int reserve(size_t bytes) {
        if (bytes <= cap) return FRB_OK;
        if (ptr) { if (pinned) cudaFreeHost(ptr); else cudaFree(ptr); ptr = nullptr; cap = 0; }
        size_t want = bytes + bytes / 8 + 4096;
        cudaError_t e = pinned ? cudaMallocHost(&ptr, want) : cudaMalloc(&ptr, want);
        if (e != cudaSuccess) return cuda_fail(e, pinned ? "cudaMallocHost" : "cudaMalloc");
        cap = want;
        return FRB_OK;
    }
};
struct HostCtx {
    Scratch d_in, d_audio, d_ws, d_out, d_misc;
    Scratch h_pin;
    cudaStream_t stream = nullptr;
    HostCtx() { h_pin.pinned = true; }
    int init() {
        if (!stream) FRB_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        return FRB_OK;
    }
};
static thread_local HostCtx t_ctx;

__global__ void __launch_bounds__(256)
k_deinterleave(const int32_t *__restrict__ in, int32_t *__restrict__ out, uint64_t n, uint32_t channels) {
    const uint64_t total = n * channels;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t s = i / channels; uint32_t c = (uint32_t)(i - s * channels);
        out[(uint64_t)c * n + s] = in[i];
    }
}
__global__ void __launch_bounds__(256)
k_interleave(const int32_t *__restrict__ in, int32_t *__restrict__ out, uint64_t n, uint32_t channels) {
    const uint64_t total = n * channels;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t s = i / channels; uint32_t c = (uint32_t)(i - s * channels);
        out[i] = in[(uint64_t)c * n + s];
    }
}

}  // namespace frb

extern "C" int frb_host_encode(const int32_t *interleaved, uint64_t n_samples, uint32_t channels,
                               uint32_t bps, uint32_t sample_rate, uint32_t level, uint32_t blocksize,
                               uint64_t first_frame_number,
                               uint8_t *out, size_t out_capacity, size_t *out_bytes,
                               uint32_t *frame_bytes, size_t frame_capacity, size_t *n_frames) {
    using namespace frb;
    if (!interleaved || !out || !out_bytes || n_samples == 0) return FRB_ERR_INVALID_ARG;
    if (first_frame_number != 0) return FRB_ERR_UNSUPPORTED;   // segments restart numbering per call (see handle API)
    frb_encode_params p = {1, channels, bps, blocksize, level, 0};
    if (!enc_params_ok(&p)) return FRB_ERR_INVALID_ARG;
    HostCtx &C = t_ctx;
    int rc = C.init();
    if (rc) return rc;
    const uint64_t total = n_samples * channels;
    const uint64_t frames = (n_samples + blocksize - 1) / blocksize;
    size_t ws_bytes = 0;
    if ((rc = frb_encode_workspace_size(&p, frames, &ws_bytes))) return rc;
    if ((rc = C.d_in.reserve(total * 4))) return rc;
    if ((rc = C.d_audio.reserve(total * 4))) return rc;
    if ((rc = C.d_ws.reserve(ws_bytes))) return rc;
    cudaStream_t s = C.stream;
    FRB_CUDA(cudaMemcpyAsync(C.d_in.ptr, interleaved, total * 4, cudaMemcpyHostToDevice, s));
    if (channels == 1) {
        FRB_CUDA(cudaMemcpyAsync(C.d_audio.ptr, C.d_in.ptr, total * 4, cudaMemcpyDeviceToDevice, s));
    } else {
        k_deinterleave<<<grid_for(total, 256 * 8, kNumSMs * 16), 256, 0, s>>>((const int32_t *)C.d_in.ptr, (int32_t *)C.d_audio.ptr, n_samples, channels);
        FRB_LAUNCH_CHECK("k_deinterleave");
    }
    uint64_t hn = n_samples; uint32_t hr = sample_rate; int64_t hb = 0; uint64_t total_bytes = 0;
    if ((rc = frb_encode_analyse(&p, (const int32_t *)C.d_audio.ptr, &hn, &hr, &hb, C.d_ws.ptr, C.d_ws.cap, nullptr, &total_bytes, s))) return rc;
    *out_bytes = (size_t)total_bytes;
    if (n_frames) *n_frames = (size_t)frames;
    if (total_bytes > out_capacity) return FRB_ERR_OVERFLOW;
    if ((rc = C.d_out.reserve(total_bytes + 16))) return rc;
    if ((rc = C.d_misc.reserve(frames * 4 + 64))) return rc;
    uint64_t off0 = 0;
    if ((rc = frb_encode_emit(&p, C.d_ws.ptr, C.d_ws.cap, &off0, (uint8_t *)C.d_out.ptr, C.d_out.cap, (uint32_t *)C.d_misc.ptr, s))) return rc;
    FRB_CUDA(cudaMemcpyAsync(out, C.d_out.ptr, total_bytes, cudaMemcpyDeviceToHost, s));
    if (frame_bytes) {
        size_t nf = frames < frame_capacity ? (size_t)frames : frame_capacity;
        FRB_CUDA(cudaMemcpyAsync(frame_bytes, C.d_misc.ptr, nf * 4, cudaMemcpyDeviceToHost, s));
    }
    FRB_CUDA(cudaStreamSynchronize(s));
    return FRB_OK;
}

namespace frb {
// planar != 0: out receives channel c's samples at out[c * n_samples ...] (the layout of the buffer[] pointers a
// FLAC__StreamDecoderWriteCallback gets); else interleaved (N, C)
static int host_decode_impl(const uint8_t *frames, size_t n_bytes, uint32_t channels, uint32_t bps,
                            uint32_t blocksize, uint32_t sample_rate, uint64_t n_samples_hint,
                            int32_t *interleaved_out, size_t out_capacity_samples,
                            uint64_t *n_samples_out, int planar) {
    if (!frames || !n_bytes || !n_samples_out) return FRB_ERR_INVALID_ARG;
    HostCtx &C = t_ctx;
    int rc = C.init();
    if (rc) return rc;
    cudaStream_t s = C.stream;
    if ((rc = C.d_in.reserve(n_bytes + 64))) return rc;
    FRB_CUDA(cudaMemsetAsync((uint8_t *)C.d_in.ptr + (n_bytes & ~(size_t)3), 0, 32, s));
    FRB_CUDA(cudaMemcpyAsync(C.d_in.ptr, frames, n_bytes, cudaMemcpyHostToDevice, s));
    uint64_t n_samples = n_samples_hint, n_frames = 0;
    if (n_samples == 0) {
        if ((rc = frb_probe_stream((const uint8_t *)C.d_in.ptr, 0, n_bytes, channels, bps, blocksize, sample_rate, &n_frames, &n_samples, s))) return rc;
    }
    n_frames = (n_samples + blocksize - 1) / blocksize;
    *n_samples_out = n_samples;
    if (!interleaved_out) return FRB_OK;                      // size query
    const uint64_t total = n_samples * channels;
    if (total > out_capacity_samples) return FRB_ERR_OVERFLOW;
    frb_decode_params p = {1, channels, bps, blocksize, 1, 12};
    size_t ws_bytes = 0;
    if ((rc = frb_decode_workspace_size(&p, n_frames, &ws_bytes))) return rc;
    if ((rc = C.d_ws.reserve(ws_bytes))) return rc;
    if ((rc = C.d_audio.reserve(total * 4))) return rc;
    if ((rc = C.d_out.reserve(total * 4))) return rc;
    if ((rc = C.d_misc.reserve(256))) return rc;
    frb_decode_stream st = {0, n_bytes, n_samples, 0, sample_rate, 0};
    uint32_t h_status[8];
    for (int attempt = 0; attempt < 2; attempt++) {
        if ((rc = frb_decode_batch(&p, &st, (const uint8_t *)C.d_in.ptr, n_frames, (int32_t *)C.d_audio.ptr, C.d_ws.ptr, C.d_ws.cap,
                                   (uint32_t *)C.d_misc.ptr, s))) return rc;
        FRB_CUDA(cudaMemcpyAsync(h_status, C.d_misc.ptr, sizeof h_status, cudaMemcpyDeviceToHost, s));
        FRB_CUDA(cudaStreamSynchronize(s));
        if (h_status[4] && attempt == 0) { p.reserved = 32; continue; }   // LPC order > 12: rerun the wide kernel
        break;
    }
    if (h_status[5]) return FRB_ERR_CUDA;                       // a decode thread gave up waiting for its subframe offset
    if (h_status[0] || h_status[2]) return FRB_ERR_BAD_STREAM;
    if (h_status[1]) return FRB_ERR_CRC;
    if (channels == 1 || planar) {
        FRB_CUDA(cudaMemcpyAsync(interleaved_out, C.d_audio.ptr, total * 4, cudaMemcpyDeviceToHost, s));
    } else {
        k_interleave<<<grid_for(total, 256 * 8, kNumSMs * 16), 256, 0, s>>>((const int32_t *)C.d_audio.ptr, (int32_t *)C.d_out.ptr, n_samples, channels);
        FRB_LAUNCH_CHECK("k_interleave");
        FRB_CUDA(cudaMemcpyAsync(interleaved_out, C.d_out.ptr, total * 4, cudaMemcpyDeviceToHost, s));
    }
    FRB_CUDA(cudaStreamSynchronize(s));
    return FRB_OK;
}
}  // namespace frb

extern "C" int frb_host_decode(const uint8_t *frames, size_t n_bytes, uint32_t channels, uint32_t bps,
                               uint32_t blocksize, uint32_t sample_rate, uint64_t n_samples_hint,
                               int32_t *interleaved_out, size_t out_capacity_samples,
                               uint64_t *n_samples_out) {
    return frb::host_decode_impl(frames, n_bytes, channels, bps, blocksize, sample_rate, n_samples_hint, interleaved_out,
                                 out_capacity_samples, n_samples_out, 0);
}

// ---------------------------------------------------------------- handle API
// State numbers follow FLAC__StreamEncoderState / FLAC__StreamDecoderState (docs/sonos-pyflac.txt:3079-3090, :2612-2625 of
// the cdef text) so a binding that prints get_state() keeps its meaning.
enum { FRB_ENC_OK = 0, FRB_ENC_UNINITIALIZED = 1, FRB_ENC_VERIFY_DECODER_ERROR = 3, FRB_ENC_VERIFY_MISMATCH = 4,
       FRB_ENC_CLIENT_ERROR = 5, FRB_ENC_IO_ERROR = 6, FRB_ENC_FRAMING_ERROR = 7, FRB_ENC_MEMORY_ERROR = 8 };

struct frb_stream_encoder {
    uint32_t channels = 2, bps = 16, sample_rate = 44100, level = 5, blocksize = 0;
    uint32_t verify = 0, streamable_subset = 1, limit_min_bitrate = 0;
    uint64_t total_estimate = 0;
    frb_encoder_write_cb cb = nullptr;
    frb_encoder_seek_cb seek_cb = nullptr;
    frb_encoder_tell_cb tell_cb = nullptr;
    frb_encoder_metadata_cb meta_cb = nullptr;
    void *client = nullptr;
    int state = FRB_ENC_UNINITIALIZED;
    std::vector<int32_t> pending;  // interleaved samples (the whole stream: the engine codes it as one batch in finish())
    std::vector<uint8_t> outbuf;
    std::vector<uint32_t> fsizes;
    std::vector<int32_t> verify_buf;
};

static const char kVendor[] = "flac-raster-b200 0.1 (sm_100a CUDA FLAC engine)";

static void frb_pack_streaminfo(uint8_t s[34], uint32_t blocksize, uint32_t min_frame, uint32_t max_frame, uint32_t rate,
                                uint32_t channels, uint32_t bps, uint64_t total) {
    memset(s, 0, 34);
    s[0] = (uint8_t)(blocksize >> 8); s[1] = (uint8_t)blocksize; s[2] = s[0]; s[3] = s[1];
    s[4] = (uint8_t)(min_frame >> 16); s[5] = (uint8_t)(min_frame >> 8); s[6] = (uint8_t)min_frame;
    s[7] = (uint8_t)(max_frame >> 16); s[8] = (uint8_t)(max_frame >> 8); s[9] = (uint8_t)max_frame;
    s[10] = (uint8_t)(rate >> 12); s[11] = (uint8_t)(rate >> 4);
    s[12] = (uint8_t)(((rate & 15) << 4) | ((channels - 1) << 1) | (((bps - 1) >> 4) & 1));
    s[13] = (uint8_t)((((bps - 1) & 15) << 4) | ((total >> 32) & 15));
    s[14] = (uint8_t)(total >> 24); s[15] = (uint8_t)(total >> 16); s[16] = (uint8_t)(total >> 8); s[17] = (uint8_t)total;
    // MD5 stays zero ("not computed", legal; the reference's files have it zero as well: SURVEY Q7)
}

extern "C" frb_stream_encoder *frb_stream_encoder_new(void) { return new (std::nothrow) frb_stream_encoder(); }
extern "C" void frb_stream_encoder_delete(frb_stream_encoder *e) { delete e; }
#define FRB_SETTER(name, field, type)                                                       \
    extern "C" int frb_stream_encoder_set_##name(frb_stream_encoder *e, type v) {            \
        if (!e || e->state != FRB_ENC_UNINITIALIZED) return 0;                              \
        e->field = v; return 1;                                                             \
    }
FRB_SETTER(channels, channels, uint32_t)
FRB_SETTER(bits_per_sample, bps, uint32_t)
FRB_SETTER(sample_rate, sample_rate, uint32_t)
FRB_SETTER(compression_level, level, uint32_t)
FRB_SETTER(blocksize, blocksize, uint32_t)
FRB_SETTER(total_samples_estimate, total_estimate, uint64_t)
FRB_SETTER(verify, verify, int)
FRB_SETTER(streamable_subset, streamable_subset, int)
FRB_SETTER(limit_min_bitrate, limit_min_bitrate, int)
#undef FRB_SETTER
extern "C" int frb_stream_encoder_get_state(const frb_stream_encoder *e) { return e ? e->state : FRB_ENC_MEMORY_ERROR; }
extern "C" int frb_stream_encoder_get_verify(const frb_stream_encoder *e) { return e ? (int)e->verify : 0; }

extern "C" int frb_stream_encoder_init_stream(frb_stream_encoder *e, frb_encoder_write_cb write_cb, frb_encoder_seek_cb seek_cb,
                                              frb_encoder_tell_cb tell_cb, frb_encoder_metadata_cb metadata_cb, void *client_data) {
    // return values follow FLAC__StreamEncoderInitStatus: 0 OK, 1 ENCODER_ERROR, 3 INVALID_CALLBACKS, 4 INVALID_NUMBER_OF_CHANNELS,
    // 5 INVALID_BITS_PER_SAMPLE, 6 INVALID_SAMPLE_RATE, 7 INVALID_BLOCK_SIZE, 11 NOT_STREAMABLE, 13 ALREADY_INITIALIZED
    if (!e) return 1;
    if (e->state != FRB_ENC_UNINITIALIZED) return 13;
    if (!write_cb || (seek_cb && !tell_cb)) return 3;
    if (e->channels < 1 || e->channels > FRB_MAX_CHANNELS) return 4;
    if (e->bps != 16 && e->bps != 32) return 5;                 // what pyflac can ask for (docs/sonos-pyflac.txt:1988-1991)
    if (e->sample_rate == 0 || e->sample_rate > 1048575u) return 6;
    if (e->level > 8) e->level = 8;
    // blocksize 0 (pyflac's default): libFLAC's init_stream picks 1152 when max_lpc_order == 0 (levels 0-2), 4096 otherwise
    if (e->blocksize == 0) e->blocksize = e->level <= 2 ? 1152 : 4096;
    if (e->blocksize < 16 || e->blocksize > FRB_MAX_BLOCKSIZE) return 7;
    // streamable subset (format.h rules quoted at docs/sonos-pyflac.txt:3498, :3527): <= 48 kHz caps the blocksize at 4608 and the
    // LPC order at 12 -- every preset of this engine satisfies both, so the flag only has to be accepted.
    // limit_min_bitrate (forces at least one non-constant subframe per frame in libFLAC 1.4) is not implemented.
    if (e->limit_min_bitrate) return 1;
    frb_encode_params p = {1, e->channels, e->bps, e->blocksize, e->level, 0};
    if (!frb::enc_params_ok(&p)) return 1;
    e->cb = write_cb; e->seek_cb = seek_cb; e->tell_cb = tell_cb; e->meta_cb = metadata_cb; e->client = client_data;
    // "fLaC" + STREAMINFO (unfinalised until finish(), and for good without a seek callback, like the reference's files:
    // SURVEY Q7) + VORBIS_COMMENT(vendor only)
    uint8_t hdr[4 + 4 + 34];
    memcpy(hdr, "fLaC", 4);
    hdr[4] = 0; hdr[5] = 0; hdr[6] = 0; hdr[7] = 34;
    frb_pack_streaminfo(hdr + 8, e->blocksize, 0, 0, e->sample_rate, e->channels, e->bps, 0);
    if (write_cb(e, hdr, 4, 0, 0, client_data)) { e->state = FRB_ENC_CLIENT_ERROR; return 1; }
    if (write_cb(e, hdr + 4, 38, 0, 0, client_data)) { e->state = FRB_ENC_CLIENT_ERROR; return 1; }
    const size_t vlen = sizeof(kVendor) - 1;
    std::vector<uint8_t> vc(4 + 4 + vlen + 4, 0);
    vc[0] = 0x84; vc[1] = (uint8_t)((8 + vlen) >> 16); vc[2] = (uint8_t)((8 + vlen) >> 8); vc[3] = (uint8_t)(8 + vlen);
    vc[4] = (uint8_t)vlen; vc[5] = (uint8_t)(vlen >> 8);
    memcpy(vc.data() + 8, kVendor, vlen);
    if (write_cb(e, vc.data(), vc.size(), 0, 0, client_data)) { e->state = FRB_ENC_CLIENT_ERROR; return 1; }
    e->state = FRB_ENC_OK;
    return 0;
}

// All samples are buffered until finish(): the engine encodes a whole stream as one batch (the
// reference makes exactly one process() call followed by finish(), converter.py:153-154).  Peak host memory is
// therefore the stream twice (caller's array + this copy) and the frame callbacks all fire inside finish().
extern "C" int frb_stream_encoder_process_interleaved(frb_stream_encoder *e, const int32_t *buffer, uint32_t samples) {
    if (!e || e->state != FRB_ENC_OK || (!buffer && samples)) return 0;
    try { e->pending.insert(e->pending.end(), buffer, buffer + (size_t)samples * e->channels); }
    catch (...) { e->state = FRB_ENC_MEMORY_ERROR; return 0; }
    return 1;
}

// planar form (FLAC__stream_encoder_process): buffer[c] points at `samples` samples of channel c
extern "C" int frb_stream_encoder_process(frb_stream_encoder *e, const int32_t *const buffer[], uint32_t samples) {
    if (!e || e->state != FRB_ENC_OK || (!buffer && samples)) return 0;
    try {
        const size_t base = e->pending.size();
        e->pending.resize(base + (size_t)samples * e->channels);
        for (uint32_t c = 0; c < e->channels; c++)
            for (uint32_t i = 0; i < samples; i++) e->pending[base + (size_t)i * e->channels + c] = buffer[c][i];
    } catch (...) { e->state = FRB_ENC_MEMORY_ERROR; return 0; }
    return 1;
}

extern "C" int frb_stream_encoder_finish(frb_stream_encoder *e) {
    if (!e) return 0;
    if (e->state != FRB_ENC_OK) { e->pending.clear(); e->state = FRB_ENC_UNINITIALIZED; return 0; }
    int ok = 1;
    const uint64_t n = e->pending.size() / e->channels;
    uint32_t min_frame = 0, max_frame = 0;
    if (n) {
        size_t cap = (size_t)n * e->channels * 5 + ((size_t)n / e->blocksize + 2) * 64 + 4096;
        e->outbuf.resize(cap);
        const size_t nf = (size_t)((n + e->blocksize - 1) / e->blocksize);
        e->fsizes.resize(nf);
        size_t ob = 0, got = 0;
        int rc = frb_host_encode(e->pending.data(), n, e->channels, e->bps, e->sample_rate, e->level, e->blocksize, 0,
                                 e->outbuf.data(), cap, &ob, e->fsizes.data(), nf, &got);
        if (rc != FRB_OK) { ok = 0; e->state = FRB_ENC_FRAMING_ERROR; }
        if (ok && e->verify) {
            // FLAC__stream_encoder_set_verify: decode what was just produced -- on the GPU decoder -- and compare
            e->verify_buf.resize((size_t)n * e->channels);
            uint64_t ns = 0;
            rc = frb_host_decode(e->outbuf.data(), ob, e->channels, e->bps, e->blocksize, e->sample_rate, n, e->verify_buf.data(),
                                 e->verify_buf.size(), &ns);
            if (rc != FRB_OK || ns != n) { ok = 0; e->state = FRB_ENC_VERIFY_DECODER_ERROR; }
            else if (memcmp(e->verify_buf.data(), e->pending.data(), (size_t)n * e->channels * 4) != 0) { ok = 0; e->state = FRB_ENC_VERIFY_MISMATCH; }
            e->verify_buf.clear(); e->verify_buf.shrink_to_fit();
        }
        if (ok) {
            size_t off = 0;
            min_frame = 0xFFFFFFFFu;
            for (size_t f = 0; f < nf; f++) {
                uint32_t bs = (f + 1 < nf) ? e->blocksize : (uint32_t)(n - (uint64_t)f * e->blocksize);
                if (e->cb(e, e->outbuf.data() + off, e->fsizes[f], bs, (uint32_t)f, e->client)) { ok = 0; e->state = FRB_ENC_CLIENT_ERROR; break; }
                off += e->fsizes[f];
                if (e->fsizes[f] < min_frame) min_frame = e->fsizes[f];
                if (e->fsizes[f] > max_frame) max_frame = e->fsizes[f];
            }
        }
    }
    if (ok && (e->seek_cb || e->meta_cb)) {
        // libFLAC finalises STREAMINFO (total samples, min/max frame size) when it can seek back, and reports it through
        // the metadata callback when one is given
        uint8_t body[34];
        frb_pack_streaminfo(body, e->blocksize, min_frame == 0xFFFFFFFFu ? 0 : min_frame, max_frame, e->sample_rate, e->channels, e->bps, n);
        if (e->seek_cb) {
            uint64_t end_pos = 0;
            if (e->tell_cb(e, &end_pos, e->client) || e->seek_cb(e, 8, e->client) || e->cb(e, body, 34, 0, 0, e->client) ||
                e->seek_cb(e, end_pos, e->client)) { ok = 0; e->state = FRB_ENC_CLIENT_ERROR; }
        }
        if (ok && e->meta_cb) {
            frb_stream_metadata md;
            memset(&md, 0, sizeof md);
            md.type = 0; md.is_last = 0; md.length = 34;
            md.stream_info.min_blocksize = md.stream_info.max_blocksize = e->blocksize;
            md.stream_info.min_framesize = min_frame == 0xFFFFFFFFu ? 0 : min_frame; md.stream_info.max_framesize = max_frame;
            md.stream_info.sample_rate = e->sample_rate; md.stream_info.channels = e->channels; md.stream_info.bits_per_sample = e->bps;
            md.stream_info.total_samples = n;
            e->meta_cb(e, &md, e->client);
        }
    }
    e->pending.clear(); e->pending.shrink_to_fit();
    if (ok) e->state = FRB_ENC_UNINITIALIZED;        // a failed finish keeps its error state for get_state(), as libFLAC does
    return ok;
}

// ---------------------------------------------------------------- decoder handle
enum { FRB_DEC_SEARCH_FOR_METADATA = 0, FRB_DEC_READ_METADATA = 1, FRB_DEC_SEARCH_FOR_FRAME_SYNC = 2, FRB_DEC_READ_FRAME = 3,
       FRB_DEC_END_OF_STREAM = 4, FRB_DEC_SEEK_ERROR = 6, FRB_DEC_ABORTED = 7, FRB_DEC_MEMORY_ERROR = 8, FRB_DEC_UNINITIALIZED = 9 };

struct frb_stream_decoder {
    int state = FRB_DEC_UNINITIALIZED;
    frb_decoder_write_cb write_cb = nullptr;
    frb_decoder_metadata_cb meta_cb = nullptr;
    frb_decoder_error_cb err_cb = nullptr;
    void *client = nullptr;
    std::vector<uint8_t> data;            // the whole stream (file contents / everything the read callback delivered)
    std::vector<int32_t> planar;          // decoded samples, channel-major
    frb_stream_metadata si;               // STREAMINFO once parsed
    bool have_si = false;
    uint64_t decoded_samples = 0;
};

extern "C" frb_stream_decoder *frb_stream_decoder_new(void) { return new (std::nothrow) frb_stream_decoder(); }
extern "C" void frb_stream_decoder_delete(frb_stream_decoder *d) { delete d; }
extern "C" int frb_stream_decoder_get_state(const frb_stream_decoder *d) { return d ? d->state : FRB_DEC_MEMORY_ERROR; }
extern "C" uint32_t frb_stream_decoder_get_channels(const frb_stream_decoder *d) { return d && d->have_si ? d->si.stream_info.channels : 0; }
extern "C" uint32_t frb_stream_decoder_get_bits_per_sample(const frb_stream_decoder *d) { return d && d->have_si ? d->si.stream_info.bits_per_sample : 0; }
extern "C" uint32_t frb_stream_decoder_get_sample_rate(const frb_stream_decoder *d) { return d && d->have_si ? d->si.stream_info.sample_rate : 0; }
extern "C" uint32_t frb_stream_decoder_get_blocksize(const frb_stream_decoder *d) { return d && d->have_si ? d->si.stream_info.max_blocksize : 0; }
extern "C" uint64_t frb_stream_decoder_get_total_samples(const frb_stream_decoder *d) { return d ? d->decoded_samples : 0; }

// FLAC__StreamDecoderInitStatus: 0 OK, 2 INVALID_CALLBACKS, 3 MEMORY_ALLOCATION_ERROR, 4 ERROR_OPENING_FILE, 5 ALREADY_INITIALIZED
extern "C" int frb_stream_decoder_init_stream(frb_stream_decoder *d, frb_decoder_read_cb read_cb, frb_decoder_seek_cb seek_cb,
                                              frb_decoder_tell_cb tell_cb, frb_decoder_length_cb length_cb, frb_decoder_eof_cb eof_cb,
                                              frb_decoder_write_cb write_cb, frb_decoder_metadata_cb metadata_cb,
                                              frb_decoder_error_cb error_cb, void *client_data) {
    (void)seek_cb; (void)tell_cb; (void)eof_cb;     // the engine never seeks: it pulls the whole stream, then decodes it as one batch
    if (!d) return 3;
    if (d->state != FRB_DEC_UNINITIALIZED) return 5;
    if (!read_cb || !write_cb || !error_cb) return 2;
    d->write_cb = write_cb; d->meta_cb = metadata_cb; d->err_cb = error_cb; d->client = client_data;
    d->data.clear(); d->have_si = false; d->decoded_samples = 0;
    try {
        uint64_t len = 0;
        if (length_cb && length_cb(d, &len, client_data) == 0 && len) d->data.reserve((size_t)len);
        std::vector<uint8_t> chunk(1 << 20);
        for (;;) {
            size_t nb = chunk.size();
            const int st = read_cb(d, chunk.data(), &nb, client_data);     // FLAC__StreamDecoderReadStatus: 0 continue, 1 end of stream, 2 abort
            if (st == 2) { d->state = FRB_DEC_ABORTED; return 0; }          // surfaces in process_*, as with libFLAC
            d->data.insert(d->data.end(), chunk.data(), chunk.data() + nb);
            if (st == 1 || nb == 0) break;
        }
    } catch (...) { return 3; }
    d->state = FRB_DEC_SEARCH_FOR_METADATA;
    return 0;
}

extern "C" int frb_stream_decoder_init_file(frb_stream_decoder *d, const char *filename, frb_decoder_write_cb write_cb,
                                            frb_decoder_metadata_cb metadata_cb, frb_decoder_error_cb error_cb, void *client_data) {
    if (!d) return 3;
    if (d->state != FRB_DEC_UNINITIALIZED) return 5;
    if (!write_cb || !error_cb) return 2;
    FILE *fh = filename ? fopen(filename, "rb") : nullptr;
    if (!fh) return 4;
    d->data.clear(); d->have_si = false; d->decoded_samples = 0;
    try {
        if (fseek(fh, 0, SEEK_END) == 0) { const long sz = ftell(fh); if (sz > 0) d->data.resize((size_t)sz); rewind(fh); }
        size_t got = d->data.empty() ? 0 : fread(d->data.data(), 1, d->data.size(), fh);
        d->data.resize(got);
    } catch (...) { fclose(fh); return 3; }
    fclose(fh);
    d->write_cb = write_cb; d->meta_cb = metadata_cb; d->err_cb = error_cb; d->client = client_data;
    d->state = FRB_DEC_SEARCH_FOR_METADATA;
    return 0;
}

namespace frb {
// metadata chain of the stream in d->data: STREAMINFO into d->si, returns the offset of the first frame (0 on error)
static size_t dec_parse_metadata(frb_stream_decoder *d) {
    const std::vector<uint8_t> &b = d->data;
    if (b.size() < 42 || memcmp(b.data(), "fLaC", 4) != 0) return 0;
    size_t pos = 4;
    bool last = false;
    while (!last) {
        if (pos + 4 > b.size()) return 0;
        last = (b[pos] & 0x80) != 0;
        const uint32_t type = b[pos] & 0x7F;
        const size_t len = ((size_t)b[pos + 1] << 16) | ((size_t)b[pos + 2] << 8) | b[pos + 3];
        pos += 4;
        if (pos + len > b.size() || type == 127) return 0;
        if (type == 0) {
            if (len < 34) return 0;
            const uint8_t *s = b.data() + pos;
            frb_stream_metadata &m = d->si;
            memset(&m, 0, sizeof m);
            m.type = 0; m.is_last = last ? 1 : 0; m.length = (uint32_t)len;
            m.stream_info.min_blocksize = ((uint32_t)s[0] << 8) | s[1];
            m.stream_info.max_blocksize = ((uint32_t)s[2] << 8) | s[3];
            m.stream_info.min_framesize = ((uint32_t)s[4] << 16) | ((uint32_t)s[5] << 8) | s[6];
            m.stream_info.max_framesize = ((uint32_t)s[7] << 16) | ((uint32_t)s[8] << 8) | s[9];
            m.stream_info.sample_rate = ((uint32_t)s[10] << 12) | ((uint32_t)s[11] << 4) | (s[12] >> 4);
            m.stream_info.channels = ((s[12] >> 1) & 7) + 1;
            m.stream_info.bits_per_sample = (((uint32_t)(s[12] & 1) << 4) | (s[13] >> 4)) + 1;
            m.stream_info.total_samples = ((uint64_t)(s[13] & 15) << 32) | ((uint64_t)s[14] << 24) | ((uint64_t)s[15] << 16) | ((uint64_t)s[16] << 8) | s[17];
            memcpy(m.stream_info.md5sum, s + 18, 16);
            d->have_si = true;
        }
        pos += len;
    }
    return d->have_si ? pos : 0;
}
}  // namespace frb

extern "C" int frb_stream_decoder_process_until_end_of_metadata(frb_stream_decoder *d) {
    if (!d || d->state == FRB_DEC_UNINITIALIZED || d->state == FRB_DEC_ABORTED) return 0;
    if (d->state != FRB_DEC_SEARCH_FOR_METADATA) return 1;
    if (!frb::dec_parse_metadata(d)) { d->err_cb(d, 0 /* LOST_SYNC */, d->client); d->state = FRB_DEC_END_OF_STREAM; return 1; }
    if (d->meta_cb) d->meta_cb(d, &d->si, d->client);           // libFLAC's default: respond to STREAMINFO only
    d->state = FRB_DEC_SEARCH_FOR_FRAME_SYNC;
    return 1;
}

extern "C" int frb_stream_decoder_process_until_end_of_stream(frb_stream_decoder *d) {
    using namespace frb;
    if (!d || d->state == FRB_DEC_UNINITIALIZED || d->state == FRB_DEC_ABORTED) return 0;
    if (d->state == FRB_DEC_SEARCH_FOR_METADATA && !frb_stream_decoder_process_until_end_of_metadata(d)) return 0;
    if (d->state != FRB_DEC_SEARCH_FOR_FRAME_SYNC) return d->state == FRB_DEC_END_OF_STREAM ? 1 : 0;
    const size_t first = dec_parse_metadata(d);
    const auto &si = d->si.stream_info;
    if (si.min_blocksize != si.max_blocksize && si.total_samples > si.max_blocksize) {       // variable-blocksize stream
        d->err_cb(d, 3 /* UNPARSEABLE_STREAM */, d->client); d->state = FRB_DEC_ABORTED; return 0;
    }
    // a legacy --spatial file is several complete streams back to back (spatial_encoder.py:155-258): this one ends where
    // the next "fLaC" + STREAMINFO block header begins
    size_t end = d->data.size();
    {
        static const uint8_t m0[8] = {'f', 'L', 'a', 'C', 0x00, 0x00, 0x00, 0x22}, m1[8] = {'f', 'L', 'a', 'C', 0x80, 0x00, 0x00, 0x22};
        for (size_t q = first; q + 8 <= d->data.size(); q++) {
            const uint8_t *p = (const uint8_t *)memchr(d->data.data() + q, 'f', d->data.size() - 7 - q);
            if (!p) break;
            q = (size_t)(p - d->data.data());
            if (memcmp(p, m0, 8) == 0 || memcmp(p, m1, 8) == 0) { end = q; break; }
        }
    }
    if (end <= first) { d->state = FRB_DEC_END_OF_STREAM; return 1; }                      // metadata only
    uint64_t n = si.total_samples, ns = 0;
    int rc = FRB_OK;
    if (n == 0) rc = host_decode_impl(d->data.data() + first, end - first, si.channels, si.bits_per_sample, si.max_blocksize, si.sample_rate,
                                      0, nullptr, 0, &n, 1);                                 // reference files: total_samples == 0 (SURVEY Q7)
    if (rc == FRB_OK) {
        try { d->planar.resize((size_t)n * si.channels); } catch (...) { d->state = FRB_DEC_MEMORY_ERROR; return 0; }
        rc = host_decode_impl(d->data.data() + first, end - first, si.channels, si.bits_per_sample, si.max_blocksize, si.sample_rate, n,
                              d->planar.data(), d->planar.size(), &ns, 1);
    }
    if (rc != FRB_OK) {
        // FLAC__StreamDecoderErrorStatus: 0 LOST_SYNC, 1 BAD_HEADER, 2 FRAME_CRC_MISMATCH, 3 UNPARSEABLE_STREAM
        d->err_cb(d, rc == FRB_ERR_CRC ? 2 : rc == FRB_ERR_BAD_STREAM ? 0 : 3, d->client);
        d->state = FRB_DEC_ABORTED;
        return 0;
    }
    const uint32_t bs = si.max_blocksize;
    const uint64_t nf = (n + bs - 1) / bs;
    const int32_t *chan[FRB_MAX_CHANNELS];
    for (uint64_t f = 0; f < nf; f++) {
        frb_frame fr;
        memset(&fr, 0, sizeof fr);
        fr.header.blocksize = (f + 1 < nf) ? bs : (uint32_t)(n - f * bs);
        fr.header.sample_rate = si.sample_rate; fr.header.channels = si.channels; fr.header.bits_per_sample = si.bits_per_sample;
        fr.header.channel_assignment = 0;                      // samples are handed out after inter-channel restoration
        fr.header.number_type = 0; fr.header.number.frame_number = (uint32_t)f;
        for (uint32_t c = 0; c < si.channels; c++) chan[c] = d->planar.data() + (size_t)c * n + (size_t)f * bs;
        d->state = FRB_DEC_READ_FRAME;
        if (d->write_cb(d, &fr, chan, d->client)) { d->state = FRB_DEC_ABORTED; return 0; }
        d->decoded_samples += fr.header.blocksize;
    }
    d->state = FRB_DEC_END_OF_STREAM;
    return 1;
}

extern "C" int frb_stream_decoder_finish(frb_stream_decoder *d) {
    if (!d) return 0;
    const int ok = d->state != FRB_DEC_UNINITIALIZED;
    d->data.clear(); d->data.shrink_to_fit(); d->planar.clear(); d->planar.shrink_to_fit();
    d->state = FRB_DEC_UNINITIALIZED;
    return ok;            // (MD5 checking is off by default in libFLAC and not offered here: finish never reports a mismatch)
}
