/*
 * flacraster_b200.h -- C ABI of libflacraster_b200.so (sm_100a CUDA FLAC engine).
 *
 * Drop-in boundary for flac-raster's one data-parallel hot path: raster
 * samples -> FLAC frames -> raster samples.  Every entry point replaces a
 * reference interface, cited as (file:line) into yharby/flac-raster:
 *
 *   sample mapping      normalization.py:126-202 (normalize_to_audio)
 *                       normalization.py:205-253 (denormalize_from_audio)
 *   codec (encode)      pyflac.StreamEncoder.process/finish at converter.py:139-154,
 *                       spatial_encoder.py:291-304; FFI crossed today:
 *                       FLAC__stream_encoder_process_interleaved
 *                       (docs/sonos-pyflac.txt:1994-1997, cdef :3206-3263)
 *   codec (decode)      pyflac.FileDecoder.process at converter.py:181-182, cli.py:479-480;
 *                       FFI: FLAC__stream_decoder_process_until_end_of_stream
 *                       (docs/sonos-pyflac.txt:1621, cdef :2826-2935)
 *   tile loop           cli.py:553-622 (_create_streaming_flac), cli.py:297-315 (extract)
 *
 * Conventions: plain C types only; every function returns an int status
 * (FRB_OK == 0), never throws, never allocates device memory behind the
 * caller's back in the *device* API (section 2/3/4: caller passes workspaces;
 * sizes come from the *_workspace_* queries).  `stream` is a cudaStream_t
 * passed as void*.  Device-API calls are asynchronous on `stream` unless
 * documented otherwise.  The host API (section 5) owns its device buffers and
 * synchronises before returning.
 */
#ifndef FLACRASTER_B200_H
#define FLACRASTER_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---------------------------------------------------------------- status */
enum {
    FRB_OK = 0,
    FRB_ERR_INVALID_ARG = 1,
    FRB_ERR_CUDA = 2,
    FRB_ERR_UNSUPPORTED = 3,     /* e.g. variable-blocksize streams, blocksize > 4096 on encode */
    FRB_ERR_BAD_STREAM = 4,      /* malformed FLAC input */
    FRB_ERR_CRC = 5,             /* frame CRC-16 / header CRC-8 mismatch */
    FRB_ERR_OVERFLOW = 6,        /* caller buffer too small */
    FRB_ERR_NO_DEVICE = 7
};

/* sample dtype codes (numpy dtype of the raster, normalization.py:7-15) */
enum {
    FRB_U8 = 0, FRB_I8 = 1, FRB_U16 = 2, FRB_I16 = 3,
    FRB_U32 = 4, FRB_I32 = 5, FRB_F32 = 6, FRB_F64 = 7
};

#define FRB_MAX_CHANNELS 8
#define FRB_MAX_BLOCKSIZE 4096      /* reference always uses 4096 (converter.py:143) */

/* --------------------------------------------------------- 1. misc/info */
int frb_version(void);                      /* 100*major + minor */
const char *frb_error_string(int status);
const char *frb_last_cuda_error(void);      /* text of the last CUDA failure on this thread */
int frb_device_count(int *count);
/* number of kernel launches issued by this library since load (bench gpu_launches) */
uint64_t frb_launch_count(void);
/* Host self-test (no GPU): CRC-16 (poly 0x8005, init 0; RFC 9639 9.3, the frame footer libFLAC writes and checks) of bytes
 * [a, e) of `bytes`, computed by the SAME per-lane code the kernels run (table-free fold form, frb_crc16.cuh), the lanes of a
 * thread group one after the other.  group: 32 (a warp per frame, rows of 30 chunks) or 128 (rows of 120 chunks).  `bytes`
 * 16-byte aligned and readable up to the 16-byte boundary after e. */
int frb_selftest_crc16(const uint8_t *bytes, uint64_t a, uint64_t e, int group, uint32_t *crc);

/* Optional per-kernel timing: when enabled the library brackets its dominant kernels with
 * cudaEvents on the caller's stream.  which: 0 k_enc_code (Rice search + packing, the dominant
 * encode kernel), 1 k_decode_subframes, 2 k_emit_frames, 3 k_sync_scan, 4 k_enc_stats,
 * 5 k_skim_subframes, 6 whole subframe analysis (stats + fixed + model + code + tail frames).
 * frb_profile_last_ms synchronises on the end event. */
int frb_profile_enable(int on);
int frb_profile_last_ms(int which, float *ms);

/* ------------------------------------------------ 2. sample mapping (device)
 * A "tile" is a window of a planar (bands, H, W) raster resident on the
 * device; tile t covers rows [row_off, row_off+h) x cols [col_off, col_off+w).
 * Its audio is `bands` planar channels of n = h*w samples (row-major), the
 * planar equivalent of the reference's interleaved (H*W, bands) array
 * (converter.py:99-110): channel c, sample i == pixel i of band c.
 * Audio is int32 on the device (int16 on the 16-bit tile path, see frb_normalize_tiles_i16): tile t, channel c,
 * sample i lives at audio[audio_base[t] + c*n_t + i].
 */
typedef struct frb_tile {
    uint32_t row_off, col_off, h, w;
} frb_tile;

/* nanmin/nanmax over all bands of each tile (normalization.py:149-153).
 * d_minmax: 2*n_tiles doubles {min,max}.  All-NaN tiles give NaN. */
int frb_minmax_tiles(const void *d_raster, int dtype, uint32_t bands, uint32_t H, uint32_t W,
                     const frb_tile *d_tiles, uint32_t n_tiles, double *d_minmax, void *stream);

/* normalize_to_audio (normalization.py:156-187) for every tile, fp64, same
 * operation order as numpy, truncating cast.  bits_per_sample: 16 -> scale
 * 32767, 24 -> 8388607, else 2147483647.  d_audio_base: n_tiles int64. */
int frb_normalize_tiles(const void *d_raster, int dtype, uint32_t bands, uint32_t H, uint32_t W,
                        const frb_tile *d_tiles, uint32_t n_tiles, const double *d_minmax,
                        int bits_per_sample, int32_t *d_audio, const int64_t *d_audio_base,
                        void *d_workspace, size_t workspace_bytes, void *stream);

/* The same mapping with int16 audio elements (same indices, half the bytes): 8/16-bit rasters at 16 bits per
 * sample only.  frb_encode_analyse reads such a buffer when FRB_ENC_AUDIO_I16 is set in frb_encode_params.reserved.
 * Round 1 moved every sample as int32 (3.8 GB written + 2 x 3.9 GB read back per C3 scene). */
int frb_normalize_tiles_i16(const void *d_raster, int dtype, uint32_t bands, uint32_t H, uint32_t W,
                            const frb_tile *d_tiles, uint32_t n_tiles, const double *d_minmax,
                            int16_t *d_audio, const int64_t *d_audio_base,
                            void *d_workspace, size_t workspace_bytes, void *stream);

/* Optional device workspace for frb_normalize_tiles / frb_denormalize_tiles: exact lookup tables that
 * replace the per-sample fp64 divisions (entries are computed with the same operations, so results
 * are unchanged).  Pass NULL/0 to compute every sample directly. */
int frb_sample_map_workspace_size(uint32_t n_tiles, size_t *bytes);

/* denormalize_from_audio (normalization.py:222-249), integer path
 * (audio/scale, fp64), np.round for integer dtypes, scattered back into the
 * planar raster windows.  scale is the divisor (32767, 8388607, ...). */
int frb_denormalize_tiles(const int32_t *d_audio, const int64_t *d_audio_base,
                          const frb_tile *d_tiles, uint32_t n_tiles, const double *d_minmax,
                          double scale, void *d_raster, int dtype, uint32_t bands, uint32_t H,
                          uint32_t W, void *d_workspace, size_t workspace_bytes, void *stream);

/* Self test of the constant-divisor shortcut used by frb_denormalize_tiles: counts the integers a in [lo, hi]
 * for which the shortcut's a/scale differs from the correctly rounded IEEE quotient (expected: 0).
 * Synchronises on `stream`. */
int frb_selftest_division(double scale, int64_t lo, int64_t hi, uint64_t *h_mismatches, void *stream);

/* Flat elementwise forms used by the drop-in normalize_to_audio /
 * denormalize_from_audio functions: n elements, any layout, one (min,max).
 * out16 != 0 writes int16 (16-bit path), else int32. */
int frb_minmax_flat(const void *d_src, int dtype, uint64_t n, double *d_minmax, void *stream);
int frb_normalize_flat(const void *d_src, int dtype, uint64_t n, double data_min, double data_max,
                       int bits_per_sample, void *d_out, int out16, void *stream);
/* audio_kind: 0 int16, 1 int32, 2 float64 (pyflac's WAV round trip, SURVEY Q3) */
int frb_denormalize_flat(const void *d_audio, int audio_kind, uint64_t n, double data_min,
                         double data_max, double scale, void *d_out, int dtype, void *stream);

/* --------------------------------------------------- 3. encode (device)
 * Batch of independent FLAC streams ("tiles"), all with the same channel
 * count, bits per sample (16 or 32) and blocksize; per-stream length and
 * sample rate.  Replaces one StreamEncoder.process/finish pair per tile
 * (converter.py:139-154).  compression_level 0..8 follows libFLAC's preset
 * table (docs/sonos-pyflac.txt:6926-6934).
 */
typedef struct frb_encode_params {
    uint32_t n_streams;
    uint32_t channels;          /* 1..8 */
    uint32_t bps;               /* 16 or 32 (what pyflac derives, docs/sonos-pyflac.txt:1988-1991) */
    uint32_t blocksize;         /* 16..4096 */
    uint32_t level;             /* 0..8 */
    uint32_t reserved;          /* flags: FRB_ENC_AUDIO_I16, FRB_ENC_RANGE_30 */
} frb_encode_params;
/* d_audio of frb_encode_analyse holds int16 elements (bps must be 16; written by frb_normalize_tiles_i16) */
#define FRB_ENC_AUDIO_I16 1u
/* every sample of a 32-bps stream is below 2^30 in magnitude (24-bit audio in a 32-bps stream, what the reference makes of
 * float32 / 32-bit rasters): two-channel streams then get libFLAC's mid/side search with its 33-bit side subframes, as 16-bps
 * streams always do; without the flag they are coded as independent channels.  A sample that breaks the promise makes
 * frb_encode_emit return FRB_ERR_INVALID_ARG. */
#define FRB_ENC_RANGE_30 2u

/* Bytes of device workspace needed by frb_encode_analyse/emit for
 * `total_frames` frames (sum over streams of ceil(n/blocksize)). */
int frb_encode_workspace_size(const frb_encode_params *p, uint64_t total_frames, size_t *bytes);

/* Pass 1: analyse + entropy-code every subframe into fixed slots of the
 * workspace; compute per-frame byte sizes, per-stream payload sizes and the
 * exclusive scans.  Host arrays (n_streams each): h_n_samples (per channel),
 * h_sample_rate, h_audio_base (int64 index into d_audio).
 * d_stream_bytes (device, n_streams uint64, optional) receives each stream's
 * frame payload size; h_stream_bytes (host, n_streams uint64, optional) is
 * filled after an internal stream synchronise when non-NULL. */
int frb_encode_analyse(const frb_encode_params *p, const void *d_audio /* int32, or int16 with FRB_ENC_AUDIO_I16 */,
                       const uint64_t *h_n_samples, const uint32_t *h_sample_rate,
                       const int64_t *h_audio_base, void *d_workspace, size_t workspace_bytes,
                       uint64_t *d_stream_bytes, uint64_t *h_stream_bytes, void *stream);

/* Pass 2: assemble frames (header, CRC-8, bit-concatenated subframes,
 * padding, CRC-16) into d_out.  Stream s's frames are written contiguously
 * starting at d_out + h_out_offset[s] (host array, bytes; the caller leaves
 * room for metadata blocks in front of each stream).  h_out_offset == NULL:
 * the streams are packed back to back in stream order (exclusive scan of the
 * sizes frb_encode_analyse computed, done on the device: no host round trip
 * between the two passes; out_capacity must cover the sum).  d_frame_bytes
 * (optional, total_frames uint32) receives every frame's size in stream order. */
int frb_encode_emit(const frb_encode_params *p, void *d_workspace, size_t workspace_bytes,
                    const uint64_t *h_out_offset, uint8_t *d_out, size_t out_capacity,
                    uint32_t *d_frame_bytes, void *stream);

/* Seek index of the streams the last frb_encode_analyse on this workspace coded (optional, any time after it):
 * d_frame_bytes[total_frames] = byte size of every frame in stream order, d_sub_bitoff[total_frames * channels] = bit
 * offset of every subframe from the first byte of its frame (entry 0 of a frame = its header's length in bits).
 * Subframes of a FLAC frame are bit-packed back to back, so without this a decoder has to walk every Rice code of
 * subframes 0..C-2 just to find where the next one starts; a decoder that is handed the index (frb_decode_*_indexed)
 * skips that walk and the sync-code scan.  The Python layer stores it per tile in a FLAC APPLICATION block ("frbI"),
 * which other decoders ignore.  Either pointer may be NULL. */
int frb_encode_index(const frb_encode_params *p, void *d_workspace, size_t workspace_bytes,
                     uint32_t *d_frame_bytes, uint32_t *d_sub_bitoff, void *stream);

/* --------------------------------------------------- 4. decode (device)
 * Batch of FLAC streams whose bytes are resident on the device.  The host
 * has parsed the metadata blocks (STREAMINFO) and passes, per stream, the
 * byte range holding audio frames.  Reference-made streams carry no seek
 * table and a zeroed STREAMINFO total (SURVEY Q7), so frames are located by
 * a parallel sync-code + CRC-8 scan.  Fixed-blocksize streams only (all the
 * reference produces).  Replaces FileDecoder.process (converter.py:181-182).
 */
typedef struct frb_decode_stream {
    uint64_t byte_offset;       /* first audio frame, offset into d_bytes */
    uint64_t byte_length;       /* bytes of audio frames */
    uint64_t n_samples;         /* expected samples per channel */
    int64_t  audio_base;        /* index into d_audio for channel 0 sample 0 */
    uint32_t sample_rate;
    uint32_t frame_base;        /* exclusive scan of ceil(n_samples/blocksize) */
} frb_decode_stream;

typedef struct frb_decode_params {
    uint32_t n_streams;
    uint32_t channels;
    uint32_t bps;
    uint32_t blocksize;         /* STREAMINFO max blocksize */
    uint32_t verify_crc16;      /* bit 0: check every frame's CRC-16 (libFLAC always does); bit 1: run the subframe-offset
                                   walk of multi-channel streams as a launch of its own instead of inside the decode launch
                                   (no assumption about the order in which CTAs become resident; slower) */
    uint32_t reserved;
} frb_decode_params;

int frb_decode_workspace_size(const frb_decode_params *p, uint64_t total_frames, size_t *bytes);

/* d_bytes must be readable 16 bytes past the last stream's end.
 * d_audio: int32 planar, same layout as section 2.  d_status: 8 uint32
 * {frames_missing, crc16_errors, parse_errors, frames_decoded, lpc_order_above_12 (rerun with
 * reserved = 32), offset_wait_timeouts, tiles_rejected (frb_decode_tiles: h*w != n_samples or window
 * outside the raster; nothing is written for them), 0}.  Multi-channel streams: the subframe offsets of a frame
 * are found and consumed inside ONE launch (skim CTAs publish, decode threads acquire). */
int frb_decode_batch(const frb_decode_params *p, const frb_decode_stream *h_streams,
                     const uint8_t *d_bytes, uint64_t total_frames, int32_t *d_audio,
                     void *d_workspace, size_t workspace_bytes, uint32_t *d_status, void *stream);

/* Fused decode + denormalise (the tile fetch of cli.py:297-315 followed by denormalize_from_audio,
 * normalization.py:222-249, in one launch): stream i holds tile d_tiles[i] of a (bands,H,W) raster of
 * `dtype` (frb_dtype), bands == p->channels, n_samples == h*w; every decode thread writes its samples
 * straight into the tile's window of d_raster, so the int32 audio never goes through HBM.  d_minmax:
 * {data_min,data_max} per tile; scale: 32767 / 8388607 / 2147483647 (normalization.py:222-232).
 * Two-channel streams (possible mid/side frames) return FRB_ERR_UNSUPPORTED: use frb_decode_batch +
 * frb_denormalize_tiles.  Same workspace, status words and slack rule as frb_decode_batch. */
int frb_decode_tiles(const frb_decode_params *p, const frb_decode_stream *h_streams,
                     const uint8_t *d_bytes, uint64_t total_frames,
                     const frb_tile *d_tiles, const double *d_minmax, double scale,
                     void *d_raster, int dtype, uint32_t bands, uint32_t H, uint32_t W,
                     void *d_workspace, size_t workspace_bytes, uint32_t *d_status, void *stream);

/* The same two calls for streams that come with a seek index (frb_encode_index): no sync scan, no walk for subframe
 * starts -- every subframe of the batch is decoded independently from the first instruction.  The index is verified
 * against the streams while decoding (frame sizes must add up to byte_length, every header must parse, every subframe
 * must end where the next one is said to begin, CRC-16): a wrong index shows up in the status words like a damaged
 * stream, and the caller then repeats the call without it. */
int frb_decode_batch_indexed(const frb_decode_params *p, const frb_decode_stream *h_streams,
                             const uint8_t *d_bytes, uint64_t total_frames,
                             const uint32_t *d_frame_bytes, const uint32_t *d_sub_bitoff, int32_t *d_audio,
                             void *d_workspace, size_t workspace_bytes, uint32_t *d_status, void *stream);
int frb_decode_tiles_indexed(const frb_decode_params *p, const frb_decode_stream *h_streams,
                             const uint8_t *d_bytes, uint64_t total_frames,
                             const uint32_t *d_frame_bytes, const uint32_t *d_sub_bitoff,
                             const frb_tile *d_tiles, const double *d_minmax, double scale,
                             void *d_raster, int dtype, uint32_t bands, uint32_t H, uint32_t W,
                             void *d_workspace, size_t workspace_bytes, uint32_t *d_status, void *stream);

/* Windowed read: a pixel window of a raster whose tiles are FLAC streams, decoding only the frames that cover it.
 * The sample order of a tile is row-major, so the samples of tile t that fall inside the window lie between its first
 * and its last visible pixel: a run of consecutive frames [first_frame, first_frame + n_frames) per stream.  A run is
 * decoded as a stream of its own (the indexed path never compares a frame's coded number with its position; the scan
 * path uses the coded numbers to find the run's frames and the frame behind it).
 *   byte_offset / byte_length: indexed path (d_frame_bytes != NULL): the bytes of the run's frames only; scan path: the
 *                              bytes of ALL the stream's frames (the scan finds the run's frames by number)
 *   total_samples:             samples per channel of the whole stream (h*w of its tile)
 *   audio_base:                dtype -1 only: index into d_out of the run's channel 0, first sample; the run's samples
 *                              per channel are min(n_frames * blocksize, total_samples - first_frame * blocksize)
 *   frame_base:                exclusive scan of n_frames (the run's frames in d_frame_bytes / d_sub_bitoff) */
typedef struct frb_window_stream {
    uint64_t byte_offset;
    uint64_t byte_length;
    uint64_t total_samples;
    int64_t  audio_base;
    uint32_t sample_rate;
    uint32_t frame_base;
    uint32_t first_frame;
    uint32_t n_frames;
} frb_window_stream;

/* Decodes the frame runs of h_streams and writes the pixels of stream i (tile d_tiles[i], image coordinates) that lie
 * inside `window` (image coordinates; row_off, col_off, h, w) to d_out, a (bands, window.h, window.w) array of `dtype`:
 * pixel (y, x) of the image lands at d_out[c, y - window.row_off, x - window.col_off].  Pixels of a run outside the window
 * are decoded (the frames have to be) but not stored.  The values are bit-identical to frb_decode_tiles (same integer
 * form, same fp64 tie path).  Tiles may overlap the window partly or not at all.
 * d_frame_bytes (total_frames entries: the runs' frame sizes, run after run) and d_sub_bitoff (total_frames * channels)
 * select the indexed path; both NULL select the scan path.  total_frames = sum of n_frames.
 * dtype -1: no pixels, d_out receives the runs' int32 planar audio at audio_base (two-channel streams, whose frames may
 * be mid/side coded, and the dtypes whose mapping runs faster as a kernel of its own): then frb_denormalize_window.
 * Otherwise two-channel streams return FRB_ERR_UNSUPPORTED.
 * Workspace: frb_decode_workspace_size(p, total_frames).  Status words as frb_decode_batch; frames_decoded counts the run
 * frames, tiles_rejected counts streams whose tile does not hold total_samples pixels.  Only the decoded frames are
 * validated: a damaged frame outside the runs is not seen. */
int frb_decode_window(const frb_decode_params *p, const frb_window_stream *h_streams,
                      const uint8_t *d_bytes, uint64_t total_frames,
                      const uint32_t *d_frame_bytes, const uint32_t *d_sub_bitoff,
                      const frb_tile *d_tiles, const double *d_minmax, double scale, frb_tile window,
                      void *d_out, int dtype, void *d_workspace, size_t workspace_bytes, uint32_t *d_status, void *stream);

/* The pixels of the window from the int32 audio frb_decode_window wrote with dtype -1 (same mapping as
 * frb_denormalize_tiles).  d_streams: the stream table of that call copied to the device; d_out as frb_decode_window. */
int frb_denormalize_window(const int32_t *d_audio, const frb_window_stream *d_streams, uint32_t n_tiles, uint32_t blocksize,
                           const frb_tile *d_tiles, const double *d_minmax, double scale, frb_tile window,
                           void *d_out, int dtype, uint32_t bands, void *stream);

/* Frame discovery for a stream of unknown length (FileDecoder on a file
 * whose STREAMINFO total_samples is 0 and no tags are known).  Synchronous.
 * Returns the number of frames and the total samples per channel. */
int frb_probe_stream(const uint8_t *d_bytes, uint64_t byte_offset, uint64_t byte_length,
                     uint32_t channels, uint32_t bps, uint32_t blocksize, uint32_t sample_rate,
                     uint64_t *n_frames, uint64_t *n_samples, void *stream);

/* Test aid: occupies the device with `ctas` thread blocks of 128 threads that each hold `smem_bytes` of shared memory and
 * spin for `ns` nanoseconds (asynchronous on `stream`).  Used to run the decode launch under SM contention. */
int frb_debug_spin(uint32_t ctas, uint32_t smem_bytes, uint64_t ns, void *stream);

/* Small host <-> device transfers for the tables and read-backs around the batch calls (tile tables, min/max,
 * status words).  They go through pinned staging and a copy kernel instead of cudaMemcpyAsync, so that they do not
 * queue behind the bulk H2D/D2H transfers of a host pipeline on the copy engines.  frb_small_upload is asynchronous
 * on `stream` (h_src may be reused on return); frb_small_download returns once h_dst holds the data (it
 * synchronises `stream`).  Device pointers must be 4-byte aligned; above 2 MiB both fall back to cudaMemcpyAsync. */
int frb_small_upload(void *d_dst, const void *h_src, size_t bytes, void *stream);
int frb_small_download(void *h_dst, const void *d_src, size_t bytes, void *stream);

/* ------------------------------------------------------ 5. host API
 * One-shot calls on HOST buffers (the e2e path: H2D, kernels, D2H inside).
 * frb_host_encode takes the interleaved int32 buffer pyflac passes to
 * FLAC__stream_encoder_process_interleaved and returns the frame payload
 * (no metadata blocks) plus per-frame sizes; frb_host_decode takes the frame
 * bytes of one stream and returns interleaved int32 samples
 * (the layout of FLAC__StreamDecoderWriteCallback after column_stack,
 * docs/sonos-pyflac.txt:1809-1854).
 */
int frb_host_encode(const int32_t *interleaved, uint64_t n_samples, uint32_t channels,
                    uint32_t bps, uint32_t sample_rate, uint32_t level, uint32_t blocksize,
                    uint64_t first_frame_number,
                    uint8_t *out, size_t out_capacity, size_t *out_bytes,
                    uint32_t *frame_bytes, size_t frame_capacity, size_t *n_frames);

int frb_host_decode(const uint8_t *frames, size_t n_bytes, uint32_t channels, uint32_t bps,
                    uint32_t blocksize, uint32_t sample_rate, uint64_t n_samples_hint,
                    int32_t *interleaved_out, size_t out_capacity_samples,
                    uint64_t *n_samples_out);

/* --------------------------------------------- 5b. tile files (host, no GPU work)
 * Metadata walk over n standalone tile FLAC files that sit in one host buffer (file i = base[offsets[i] .. +sizes[i])):
 * what SpatialFLACStreamer needs per tile before the batched GPU decode -- where the frames start, STREAMINFO, the
 * GEOSPATIAL_* numbers the reference parses from the VORBIS tags (converter.py:356-377) and the seek index block.
 * Returns FRB_ERR_BAD_STREAM if any file is not a FLAC stream (its entry has first_frame_offset == 0). */
typedef struct frb_tile_header {
    uint32_t first_frame_offset;        /* 0: not a parseable FLAC file */
    uint32_t sample_rate, channels, bps, min_blocksize, max_blocksize;
    uint32_t width, height, count;      /* GEOSPATIAL_WIDTH / HEIGHT / COUNT (0 when absent) */
    int32_t dtype;                      /* FRB_U8..FRB_F64 from GEOSPATIAL_DTYPE, -1 when absent / unknown */
    uint32_t flags;                     /* bit 0: GEOSPATIAL_CRS present, bit 1: nodata is a number, bit 2: seek index block present */
    uint32_t index_offset, index_len;   /* "frbI" APPLICATION data (behind the 4-byte id), offset from the start of the file */
    uint64_t total_samples;
    double data_min, data_max, nodata;  /* NaN when absent */
} frb_tile_header;
int frb_parse_tile_headers(const uint8_t *base, const uint64_t *offsets, const uint64_t *sizes, uint32_t n,
                           frb_tile_header *out);
/* Concatenates the tiles' seek indices in payload order for frb_decode_*_indexed (frame_bytes_out: sum(frames_per_tile)
 * entries, sub_bitoff_out: that times channels; NULL allowed for one channel).  FRB_ERR_BAD_STREAM if a tile has no
 * index or one that does not match (channels, blocksize, frame count): decode without an index then. */
int frb_gather_seek_index(const uint8_t *base, const uint64_t *offsets, const frb_tile_header *hdrs, uint32_t n,
                          uint32_t channels, uint32_t blocksize, const uint32_t *frames_per_tile,
                          uint32_t *frame_bytes_out, uint32_t *sub_bitoff_out);

/* ------------------------------------------ 6. libFLAC-shaped handle API
 * The exact calls pyflac's cffi layer makes, so a binding written against FLAC__stream_encoder_* /
 * FLAC__stream_decoder_* (cdef at docs/sonos-pyflac.txt:3206-3263 and :2826-2935) can be retargeted by renaming
 * FLAC__ -> frb_.  Same argument order and meaning, FLAC__bool-style returns (1 = success) for the
 * set/process/finish calls, FLAC__Stream{En,De}coderInitStatus numbers for the init calls and
 * FLAC__Stream{En,De}coderState numbers for get_state.  Handles are not thread-safe; callbacks run on
 * the calling thread; callback buffers are borrowed for the duration of the callback (pyflac copies them,
 * docs/sonos-pyflac.txt:2325, :1840-1841).
 *
 * Difference in timing, not in content: the engine codes a stream as ONE GPU batch, so the encoder
 * buffers every process*() call and delivers all frame callbacks inside finish() (peak host memory:
 * the stream twice), and the decoder pulls the whole stream before the first write callback.  The
 * reference makes one process() call followed by finish() (converter.py:153-154) and decodes whole
 * files (converter.py:181-182), so it cannot observe the difference. */

/* ---- metadata / frame views handed to callbacks: the leading members of FLAC__StreamMetadata (with its
 * stream_info arm, docs/sonos-pyflac.txt:2698-2708, :2799-2813) and of FLAC__Frame (:2598-2610, :2679-2683) */
typedef struct frb_stream_info {
    uint32_t min_blocksize, max_blocksize;
    uint32_t min_framesize, max_framesize;
    uint32_t sample_rate, channels, bits_per_sample;
    uint64_t total_samples;
    uint8_t md5sum[16];
} frb_stream_info;
typedef struct frb_stream_metadata {
    int type;                   /* 0 = STREAMINFO (the only block the callbacks report, libFLAC's default) */
    int is_last;
    uint32_t length;
    frb_stream_info stream_info;
} frb_stream_metadata;

typedef struct frb_frame_header {
    uint32_t blocksize;
    uint32_t sample_rate;
    uint32_t channels;
    int channel_assignment;     /* always 0 (independent): buffer[] holds the restored channels */
    uint32_t bits_per_sample;
    int number_type;            /* 0 = frame number (fixed-blocksize streams) */
    union { uint32_t frame_number; uint64_t sample_number; } number;
    uint8_t crc;
} frb_frame_header;
typedef struct frb_frame {
    frb_frame_header header;    /* FLAC__Frame continues with subframes[8] and the footer; pyflac reads the header only
                                   (docs/sonos-pyflac.txt:1823-1846) */
} frb_frame;

/* ---- encoder (FLAC__stream_encoder_*, docs/sonos-pyflac.txt:3206-3263; used at :2186-2212, :1994-1997, :2003-2014) */
typedef struct frb_stream_encoder frb_stream_encoder;
/* FLAC__StreamEncoderWriteCallback (:3192): returns 0 on success.  samples == 0 marks a metadata chunk */
typedef int (*frb_encoder_write_cb)(const frb_stream_encoder *enc, const uint8_t *buffer,
                                    size_t bytes, uint32_t samples, uint32_t current_frame,
                                    void *client_data);
/* FLAC__StreamEncoderSeekCallback / TellCallback / MetadataCallback (:3193-3195): 0 = OK */
typedef int (*frb_encoder_seek_cb)(const frb_stream_encoder *enc, uint64_t absolute_byte_offset, void *client_data);
typedef int (*frb_encoder_tell_cb)(const frb_stream_encoder *enc, uint64_t *absolute_byte_offset, void *client_data);
typedef void (*frb_encoder_metadata_cb)(const frb_stream_encoder *enc, const frb_stream_metadata *metadata, void *client_data);

frb_stream_encoder *frb_stream_encoder_new(void);
void frb_stream_encoder_delete(frb_stream_encoder *enc);
int frb_stream_encoder_set_verify(frb_stream_encoder *enc, int value);       /* finish() decodes its own frames on the GPU and compares */
int frb_stream_encoder_set_channels(frb_stream_encoder *enc, uint32_t v);
int frb_stream_encoder_set_bits_per_sample(frb_stream_encoder *enc, uint32_t v);
int frb_stream_encoder_set_sample_rate(frb_stream_encoder *enc, uint32_t v);
int frb_stream_encoder_set_compression_level(frb_stream_encoder *enc, uint32_t v);
int frb_stream_encoder_set_blocksize(frb_stream_encoder *enc, uint32_t v);
int frb_stream_encoder_set_total_samples_estimate(frb_stream_encoder *enc, uint64_t v);
int frb_stream_encoder_set_streamable_subset(frb_stream_encoder *enc, int value);   /* every preset is subset-conformant: accepted */
int frb_stream_encoder_set_limit_min_bitrate(frb_stream_encoder *enc, int value);   /* 1 is refused by init_stream (not implemented) */
int frb_stream_encoder_get_verify(const frb_stream_encoder *enc);
/* FLAC__StreamEncoderState: 0 OK, 1 UNINITIALIZED, 3 VERIFY_DECODER_ERROR, 4 VERIFY_MISMATCH_IN_AUDIO_DATA, 5 CLIENT_ERROR,
 * 7 FRAMING_ERROR, 8 MEMORY_ALLOCATION_ERROR */
int frb_stream_encoder_get_state(const frb_stream_encoder *enc);
/* Emits "fLaC" + STREAMINFO + VORBIS_COMMENT(vendor) through write_cb (samples == 0).  seek_cb, tell_cb and
 * metadata_cb may be NULL (the reference passes none, converter.py:139-144: STREAMINFO then stays unfinalised,
 * SURVEY Q7); with seek_cb + tell_cb finish() seeks to byte 8 and rewrites the STREAMINFO body with the total samples
 * and min/max frame sizes (MD5 stays zero).  Returns a FLAC__StreamEncoderInitStatus (0 = OK). */
int frb_stream_encoder_init_stream(frb_stream_encoder *enc, frb_encoder_write_cb write_cb,
                                   frb_encoder_seek_cb seek_cb, frb_encoder_tell_cb tell_cb,
                                   frb_encoder_metadata_cb metadata_cb, void *client_data);
/* return 1 (true) on success like FLAC__bool */
int frb_stream_encoder_process_interleaved(frb_stream_encoder *enc, const int32_t *buffer,
                                           uint32_t samples);
int frb_stream_encoder_process(frb_stream_encoder *enc, const int32_t *const buffer[], uint32_t samples);
int frb_stream_encoder_finish(frb_stream_encoder *enc);

/* ---- decoder (FLAC__stream_decoder_*, cdef docs/sonos-pyflac.txt:2826-2935; used by pyflac.FileDecoder at :1584-1629
 * and by its write callback at :1809-1854) */
typedef struct frb_stream_decoder frb_stream_decoder;
/* FLAC__StreamDecoderWriteCallback (:2825): one call per frame, buffer[c] = header.blocksize samples of channel c
 * (16-bit samples sign-extended in int32, like libFLAC).  Return 0 to continue, non-zero to abort. */
typedef int (*frb_decoder_write_cb)(const frb_stream_decoder *dec, const frb_frame *frame,
                                    const int32_t *const buffer[], void *client_data);
typedef void (*frb_decoder_metadata_cb)(const frb_stream_decoder *dec, const frb_stream_metadata *metadata, void *client_data);
/* status: FLAC__StreamDecoderErrorStatus (0 LOST_SYNC, 1 BAD_HEADER, 2 FRAME_CRC_MISMATCH, 3 UNPARSEABLE_STREAM) */
typedef void (*frb_decoder_error_cb)(const frb_stream_decoder *dec, int status, void *client_data);
/* FLAC__StreamDecoderReadCallback (:2820): fill buffer[0..*bytes), set *bytes; return 0 continue, 1 end of stream, 2 abort */
typedef int (*frb_decoder_read_cb)(const frb_stream_decoder *dec, uint8_t buffer[], size_t *bytes, void *client_data);
typedef int (*frb_decoder_seek_cb)(const frb_stream_decoder *dec, uint64_t absolute_byte_offset, void *client_data);
typedef int (*frb_decoder_tell_cb)(const frb_stream_decoder *dec, uint64_t *absolute_byte_offset, void *client_data);
typedef int (*frb_decoder_length_cb)(const frb_stream_decoder *dec, uint64_t *stream_length, void *client_data);
typedef int (*frb_decoder_eof_cb)(const frb_stream_decoder *dec, void *client_data);

frb_stream_decoder *frb_stream_decoder_new(void);
void frb_stream_decoder_delete(frb_stream_decoder *dec);
/* FLAC__StreamDecoderInitStatus: 0 OK, 2 INVALID_CALLBACKS, 3 MEMORY_ALLOCATION_ERROR, 4 ERROR_OPENING_FILE,
 * 5 ALREADY_INITIALIZED.  seek/tell/length/eof callbacks may be NULL (the engine never seeks). */
int frb_stream_decoder_init_stream(frb_stream_decoder *dec, frb_decoder_read_cb read_cb, frb_decoder_seek_cb seek_cb,
                                   frb_decoder_tell_cb tell_cb, frb_decoder_length_cb length_cb, frb_decoder_eof_cb eof_cb,
                                   frb_decoder_write_cb write_cb, frb_decoder_metadata_cb metadata_cb,
                                   frb_decoder_error_cb error_cb, void *client_data);
int frb_stream_decoder_init_file(frb_stream_decoder *dec, const char *filename, frb_decoder_write_cb write_cb,
                                 frb_decoder_metadata_cb metadata_cb, frb_decoder_error_cb error_cb, void *client_data);
int frb_stream_decoder_process_until_end_of_metadata(frb_stream_decoder *dec);
/* whole stream: metadata callback (STREAMINFO), GPU decode, one write callback per frame.  A file holding several
 * concatenated streams (legacy --spatial layout) yields the first one.  Returns 1 on success. */
int frb_stream_decoder_process_until_end_of_stream(frb_stream_decoder *dec);
int frb_stream_decoder_finish(frb_stream_decoder *dec);
/* FLAC__StreamDecoderState: 0 SEARCH_FOR_METADATA, 2 SEARCH_FOR_FRAME_SYNC, 3 READ_FRAME, 4 END_OF_STREAM, 7 ABORTED,
 * 8 MEMORY_ALLOCATION_ERROR, 9 UNINITIALIZED */
int frb_stream_decoder_get_state(const frb_stream_decoder *dec);
uint32_t frb_stream_decoder_get_channels(const frb_stream_decoder *dec);
uint32_t frb_stream_decoder_get_bits_per_sample(const frb_stream_decoder *dec);
uint32_t frb_stream_decoder_get_sample_rate(const frb_stream_decoder *dec);
uint32_t frb_stream_decoder_get_blocksize(const frb_stream_decoder *dec);
uint64_t frb_stream_decoder_get_total_samples(const frb_stream_decoder *dec);   /* samples handed to the write callback so far */

#ifdef __cplusplus
}
#endif
#endif /* FLACRASTER_B200_H */
