/*
 * include/vdl2gpu.h — C-ABI of libvdl2gpu.so: the B200 (sm_100a) implementation of dumpvdl2's
 * per-channel DSP hot path (reference src/demod.c + src/decode.c burst part + src/chebyshev.c +
 * src/rs.c + src/libfec + the src/bitstream.c helpers).
 *
 * Plain C: pointers and sizes only, no CUDA or torch types (a cudaStream_t travels as void*).
 * Every entry point returns 0 on success or a negative VDL2GPU_E* code; the library never calls
 * exit().  There is NO CPU fallback: without a CUDA device every call that needs one fails with
 * VDL2GPU_ENODEV.
 *
 * Two front doors (INTEGRATION.md shows the reference-side binding for both):
 *
 *  (1) batch API (this file): one context = one IQ stream fanned out to N channels, or many streams
 *      (n_streams, vdl2gpu_create_streams) each with its own channels.  It replaces, as a
 *      unit, what the reference spreads over
 *        process_buf_uchar/process_buf_short   (src/demod.c:339-365)    -> vdl2gpu_submit
 *        N x process_samples threads + barriers (src/demod.c:288-337)   -> kernels K0-K3 on a stream
 *        decode_vdl2_burst -> avlc_decoder_queue_push (src/decode.c:165-194,196-384) -> vdl2gpu_poll/flush callback
 *
 *  (2) drop-in symbols (include/vdl2_dropin.h): the exact names/signatures of src/dumpvdl2.h:371-389 so
 *      that the unmodified front-ends and main() of the reference link against this library.
 */
#ifndef VDL2GPU_H
#define VDL2GPU_H
#include <stddef.h>
#include <stdint.h>
#include <sys/time.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VDL2GPU_ABI_VERSION 2

/* error codes */
enum {
	VDL2GPU_OK = 0,
	VDL2GPU_EINVAL = -1,      /* bad argument */
	VDL2GPU_ENODEV = -2,      /* no usable CUDA device / extension not usable */
	VDL2GPU_ECUDA = -3,       /* CUDA runtime error (vdl2gpu_last_error() has the text) */
	VDL2GPU_ENOMEM = -4,
	VDL2GPU_ETOOBIG = -5,     /* chunk larger than max_chunk_bytes */
	VDL2GPU_EOVERFLOW = -6    /* an internal device queue overflowed; bursts were dropped (see stats) */
};

/* sample formats: reference enum sample_formats (src/dumpvdl2.h:319) */
enum { VDL2GPU_FMT_U8 = 0, VDL2GPU_FMT_S16_LE = 1 };

/* config flags */
enum {
	VDL2GPU_FLAG_TRACE = 1u << 0,        /* record sync/header/burst events (debug, parity tests) */
	VDL2GPU_FLAG_KEEP_DEC = 1u << 1,     /* keep the decimated samples of the last chunk readable (parity tests) */
	VDL2GPU_FLAG_K1_SCALAR = 1u << 2,    /* use the plain per-sample K1 kernel instead of the pipelined one */
	VDL2GPU_FLAG_NO_OVERLAP = 1u << 3,   /* one stream: do not run K0/K1 of chunk c+1 beside K2/K3 of chunk c (profiling) */
	VDL2GPU_FLAG_NO_GRAPH = 1u << 4      /* launch every kernel individually instead of replaying the per-chunk CUDA graphs */
};

typedef struct {
	uint32_t sample_rate;        /* Hz; must equal 105000 * oversample (src/dumpvdl2.c:1073) */
	uint32_t oversample;         /* src/dumpvdl2.h:348 */
	uint32_t sample_fmt;         /* VDL2GPU_FMT_* */
	uint32_t centerfreq;         /* Hz */
	uint32_t n_channels;
	const uint32_t *freqs;       /* n_channels channel frequencies, Hz (src/demod.c:379-392) */
	float max_ppm;               /* Config.max_ppm (src/demod.c:192); 0 = off */
	uint32_t max_chunk_bytes;    /* largest len ever passed to submit; 0 = 1 MiB */
	int32_t device;              /* CUDA device ordinal; -1 = current device */
	uint32_t flags;              /* VDL2GPU_FLAG_* */
	uint32_t n_inflight;         /* chunks in flight before submit blocks (back-pressure); 0 = 4 */
	uint32_t n_streams;          /* independent IQ streams (0 = 1).  With S > 1 the n_channels = S x C channels are split
	                              * stream-major: channels [s*C, (s+1)*C) demodulate stream s; C must be a multiple of 32,
	                              * or 1 (one stream per channel: every channel reads its own IQ buffer, as every
	                              * channel thread of the reference does, src/demod.c:302-310) */
	uint32_t reserved[4];
} vdl2gpu_config;

/* One AVLC frame with the metadata the reference attaches in decode_frame (src/decode.c:173-194,
 * struct vdl2_msg_metadata src/output-common.h:31-43).  `data` is valid only during the callback. */
typedef struct {
	uint32_t channel;            /* index into freqs[] */
	uint32_t freq;
	uint32_t burst_seq;          /* per-channel count of bursts that reached the data stage */
	int32_t idx;                 /* frame number within the burst (metadata->idx) */
	const uint8_t *data;         /* frame octets, FCS included, flags excluded */
	uint32_t len;
	uint32_t synd_weight;
	uint32_t datalen_octets;
	int32_t num_fec_corrections;
	float frame_pwr_dbfs, nf_pwr_dbfs, ppm_error;
	float frame_pwr, mag_nf;     /* the raw values the two dBFS figures derive from */
	uint64_t sync_dec_index;     /* decimated-sample index at which preamble sync was declared */
	struct timeval burst_timestamp; /* chunk arrival time + sample offset (the reference calls gettimeofday at sync) */
	uint16_t fcs_residue;        /* crc16 over the frame; 0xF0B8 = good (src/avlc.c:40,177-179) */
	uint16_t fcs_ok;             /* len >= 11 && residue good */
} vdl2gpu_frame;

typedef void (*vdl2gpu_frame_cb)(const vdl2gpu_frame *frame, void *user);

/* per-context counters; names follow the reference's statsd counters (src/statsd.c:33-64) */
typedef struct {
	uint64_t chunks_submitted, chunks_completed;
	uint64_t iq_samples;                 /* complex samples accepted */
	uint64_t dec_samples;                /* decimated samples produced per channel */
	uint64_t demod_sync_good;            /* demod.sync.good */
	uint64_t decoder_crc_good;           /* decoder.crc.good (header syndrome 0) */
	uint64_t bursts;                     /* bursts that reached DEC_DATA */
	uint64_t burst_errors;               /* bursts dropped in DEC_DATA (any decoder.errors.*) */
	uint64_t blocks_processed, blocks_fec_ok;
	uint64_t msg_good;                   /* decoder.msg.good = frames pushed */
	uint64_t fcs_good, fcs_bad;          /* avlc.frames.good / avlc.errors.bad_fcs (len >= 11 only) */
	uint64_t pool_overflows;             /* bursts lost because the device burst pool was exhausted (must be 0) */
	uint64_t out_overflows;              /* bursts lost because the output region was exhausted (must be 0) */
	uint64_t kernel_launches;            /* kernels launched by this context so far */
	uint64_t out_bytes;                  /* burst-record bytes K3 wrote to host memory (device->host traffic) */
	uint64_t graph_launches;             /* CUDA graph replays (3 per chunk of the nominal shape; 0 with VDL2GPU_FLAG_NO_GRAPH) */
	uint64_t reserved[2];
} vdl2gpu_stats;

/* trace event (VDL2GPU_FLAG_TRACE): same layout as the oracle's vo_event */
typedef struct {
	uint32_t channel, kind;      /* kind: 1 sync, 2 header, 3 burst */
	uint64_t dec_index;
	int32_t i[8];
	float f[8];
} vdl2gpu_event;

typedef struct vdl2gpu_ctx vdl2gpu_ctx;

/* Receiver farm: n_streams IQ streams, each from its own receiver with its own centre frequency, each carrying any number
 * of channels (0 allowed).  cfg->freqs lists the channels stream-major (stream 0's first), so channel k demodulates the
 * stream it falls into by the running sum of channels_per_stream.  Everything after create works as with
 * cfg->n_streams = S: submit / submit_device take S buffers of `len` bytes back to back, frames carry the channel index
 * into cfg->freqs and its frequency.  Rules: cfg->n_streams is 0 or n_streams; counts sum to cfg->n_channels; every
 * channel lies less than sample_rate / 2 from its stream's centre; oversample 10, 13 or 20; VDL2GPU_FMT_U8 or
 * VDL2GPU_FMT_S16_LE; no VDL2GPU_FLAG_K1_SCALAR.  A layout that breaks one returns VDL2GPU_EINVAL before any device
 * call. */
typedef struct {
	uint32_t n_streams;
	const uint32_t *channels_per_stream; /* n_streams counts (0 allowed), sum == cfg->n_channels */
	const uint32_t *centerfreqs;         /* n_streams centre frequencies in Hz; NULL = cfg->centerfreq for every stream */
} vdl2gpu_stream_layout;

/* ---- life cycle ---- */
int vdl2gpu_abi_version(void);
int vdl2gpu_device_count(void);
int vdl2gpu_create(const vdl2gpu_config *cfg, vdl2gpu_ctx **out);
int vdl2gpu_create_streams(const vdl2gpu_config *cfg, const vdl2gpu_stream_layout *layout, vdl2gpu_ctx **out);
int vdl2gpu_destroy(vdl2gpu_ctx *ctx);
const char *vdl2gpu_strerror(int code);
const char *vdl2gpu_last_error(void);

/* ---- data path ---- */
/* == process_buf_uchar / process_buf_short (src/demod.c:339-365): `iq` is interleaved I,Q, `len` is in BYTES,
 * the caller may reuse `iq` as soon as the call returns.  Asynchronous: copies into a pinned staging ring,
 * enqueues H2D + kernels.  Blocks only when n_inflight chunks are pending (the reference's back-pressure).
 * With n_streams = S > 1, `iq` holds S buffers of `len` bytes back to back (stream 0 first) and `len` is the size of ONE. */
int vdl2gpu_submit(vdl2gpu_ctx *ctx, const void *iq, uint32_t len);
/* Ingest adaptor for front-ends that deliver I and Q as separate int16 arrays (SDRplay: src/sdrplay.c:72-134,
 * src/sdrplay3.c): n_pairs values each; replaces the host-side interleave + process_buf_short.  The context must
 * have been created with VDL2GPU_FMT_S16_LE. */
int vdl2gpu_submit_planar_s16(vdl2gpu_ctx *ctx, const int16_t *xi, const int16_t *xq, uint32_t n_pairs);
/* Same, but `dev_iq` already lives in this GPU's memory (e.g. the receive buffer of an NCCL broadcast).
 * `producer_stream` (cudaStream_t, may be NULL = legacy default stream) is the stream on which the buffer
 * was produced; the library orders its work after it.  The buffer may be overwritten once
 * vdl2gpu_wait_input_consumed() has been enqueued on the stream that overwrites it. */
int vdl2gpu_submit_device(vdl2gpu_ctx *ctx, const void *dev_iq, uint32_t len, void *producer_stream);
int vdl2gpu_wait_input_consumed(vdl2gpu_ctx *ctx, void *stream);
/* Make `stream` (cudaStream_t) wait for all device work enqueued by this context so far (for timing with
 * events recorded on the caller's stream, and for ordering consumers of device-side results). */
int vdl2gpu_stream_wait(vdl2gpu_ctx *ctx, void *stream);
/* Deliver the frames of every chunk that has finished, in (chunk, channel, burst, idx) order.  Returns the
 * number of frames delivered or a negative error.  cb may be NULL (frames are dropped, counters kept). */
int vdl2gpu_poll(vdl2gpu_ctx *ctx, vdl2gpu_frame_cb cb, void *user);
/* Chunks submitted whose frames have not been harvested yet (0 right after a poll = everything delivered). */
int vdl2gpu_chunks_in_flight(vdl2gpu_ctx *ctx);
/* Block until everything submitted so far has been processed, then deliver like poll. */
int vdl2gpu_flush(vdl2gpu_ctx *ctx, vdl2gpu_frame_cb cb, void *user);
int vdl2gpu_get_stats(vdl2gpu_ctx *ctx, vdl2gpu_stats *out);
/* per-channel counters, 9 x uint64 per channel in the order: sync_good, hdr_crc_good, bursts, burst_err,
 * blocks_processed, blocks_fec_ok, msg_good, fcs_good, fcs_bad.  Implies a flush of device work. */
int vdl2gpu_get_channel_counters(vdl2gpu_ctx *ctx, uint64_t *out, uint32_t n_channels);

/* ---- multi-GPU ingest (one process per GPU; global channel k is demodulated on GPU k mod N, the reference's
 * channel threads share nothing but the read-only sample buffer: src/dumpvdl2.c:117-135, src/demod.c:50,300-301).
 * Rank 0 owns the IQ source; vdl2gpu_mg_* fans every step's chunks out into a double-buffered receive area on every
 * rank and feeds the rank's context from it (vdl2gpu_submit_device), either with ncclBroadcast (libnccl is dlopen()ed)
 * or, with no kernel at all, with copy-engine peer copies into CUDA-IPC-mapped buffers ordered by stream memory
 * operations.  The caller carries the small opaque blobs between the processes (MPI, sockets, ...).  Typical sequence:
 *
 *     uint8_t id[VDL2GPU_MG_ID_BYTES];              // NCCL mode only
 *     if(rank == 0) vdl2gpu_mg_unique_id(id, sizeof id);   bcast(id);
 *     vdl2gpu_mg_create(ctx, rank, world, mode, id, step_bytes, &mg);
 *     // copy-engine mode only:  vdl2gpu_mg_export(mg, blob, n);  allgather(blob -> all);  vdl2gpu_mg_import(mg, all, world * n);
 *     half = vdl2gpu_mg_stage(mg, pieces, sizes, n_pieces, host?, step_bytes);          // step 0
 *     for(;;) {
 *         next = vdl2gpu_mg_stage(mg, ...);          // step s+1 travels while step s is demodulated
 *         vdl2gpu_mg_submit(mg, half, chunks_per_step, chunk_bytes);
 *         vdl2gpu_poll(ctx, frame_cb, user);
 *         half = next;
 *     }
 * ---- */
enum { VDL2GPU_MG_NCCL = 0, VDL2GPU_MG_COPY_ENGINE = 1 };
#define VDL2GPU_MG_ID_BYTES 128
typedef struct vdl2gpu_mg vdl2gpu_mg;
int vdl2gpu_mg_unique_id(uint8_t *id, size_t cap);      /* rank 0: ncclGetUniqueId */
int vdl2gpu_mg_create(vdl2gpu_ctx *ctx, int rank, int world, int mode, const uint8_t *nccl_id /* NULL in copy-engine mode */,
		uint32_t stage_bytes /* bytes of one step, at most */, vdl2gpu_mg **out);
size_t vdl2gpu_mg_blob_bytes(void);
int vdl2gpu_mg_export(vdl2gpu_mg *mg, uint8_t *blob, size_t cap);
int vdl2gpu_mg_import(vdl2gpu_mg *mg, const uint8_t *all_blobs, size_t bytes);
/* rank 0: the pieces (device pointers, or pinned host pointers with src_is_host) that make up the step, `total` bytes;
 * other ranks: n_src = 0, same total.  Returns the half (0/1) for vdl2gpu_mg_submit or a negative error.  Asynchronous. */
int vdl2gpu_mg_stage(vdl2gpu_mg *mg, const void *const *src, const uint32_t *src_bytes, uint32_t n_src, int src_is_host, uint32_t total);
int vdl2gpu_mg_submit(vdl2gpu_mg *mg, int half, uint32_t n_chunks, uint32_t chunk_bytes);
int vdl2gpu_mg_mode(vdl2gpu_mg *mg);
int vdl2gpu_mg_destroy(vdl2gpu_mg *mg);

/* One frame in the reference's raw-frame archive format (2-octet big-endian record length + proto3
 * dumpvdl2.raw_avlc_frame, proto/dumpvdl2.proto:25-48, as written by src/fmtr-binary.c + src/output-file.c:181-189):
 * records written back to back replay through an unmodified `dumpvdl2 --raw-frames-file`.
 * Returns the record size in octets, or a negative error.  Host-only helper (no device work). */
int vdl2gpu_serialize_raw_frame(const vdl2gpu_frame *frame, const char *station_id, uint8_t *out, size_t cap);

/* ---- introspection for parity tests / profiling ---- */
/* tables the kernels use, computed by the library's own host code (restating src/demod.c:349-377,367-370,84-96) */
int vdl2gpu_get_tables(vdl2gpu_ctx *ctx, float levels[256], float sin_lut[257], float cos_lut[257],
		float A[3], float B[3], float lr_X[16], float *lr_denom, float pr_phase[16]);
/* decimated samples of the most recent chunk (VDL2GPU_FLAG_KEEP_DEC): out[n_dec][n_channels][2] floats.
 * *n_dec receives the count; cap_floats is the capacity of out.  Synchronises. */
int vdl2gpu_read_dec(vdl2gpu_ctx *ctx, float *out, size_t cap_floats, uint32_t *n_dec);
/* drain trace events (VDL2GPU_FLAG_TRACE).  Synchronises.  Returns the number copied (0: none left).  The device buffer
 * holds 2^20 events and restarts whenever it has been drained; if it filled up in between, the stored events are
 * delivered first and the following call returns VDL2GPU_EOVERFLOW once (the count of lost events in vdl2gpu_last_error). */
int vdl2gpu_read_events(vdl2gpu_ctx *ctx, vdl2gpu_event *out, uint32_t cap);
/* device time (ms) spent in each kernel for the chunks completed so far, measured with CUDA events on
 * the library's streams when timing was enabled with vdl2gpu_enable_timing(ctx, 1).
 * Order: K0, K1, K2a, K2 (+history copy), K3 (+finish).  A receiver farm has no K0 (0 launches). */
int vdl2gpu_enable_timing(vdl2gpu_ctx *ctx, int on);
int vdl2gpu_get_kernel_ms(vdl2gpu_ctx *ctx, double ms[5], uint64_t launches[5]);
/* stage boundaries of the timed chunks harvested so far, 8 floats per chunk: chunk number, then ms since
 * vdl2gpu_enable_timing(ctx, 1) of: front (K0+K1) start, K1 end, K2a start, K2a end, K2 start, K2|K3, K3 end (with graph
 * replay K3 counts into K2).  Returns the number of rows copied. */
int vdl2gpu_get_timeline(vdl2gpu_ctx *ctx, float *out, uint32_t cap_rows);
/* diagnostic (context created with VDL2GPU_BLOCK_TRACE=1 in the environment): where and when every block of K1 / K2 ran,
 * 6 x uint64 per record {kernel (1 K1, 2 K2), block, SM id, 0, start ns, end ns}.  Synchronises. */
int vdl2gpu_debug_block_trace(vdl2gpu_ctx *ctx, uint64_t *out, uint32_t cap_records);

/* ---- raw launch stubs (extern "C", plain pointers; used by the micro-parity tests and by hosts that
 *      manage device memory themselves).  All pointers are DEVICE pointers unless stated otherwise; `stream` is a
 *      cudaStream_t.  The launch stubs only enqueue kernels: no allocation, no synchronisation.
 *      (vdl2gpu_launch_rs_verify builds its GF tables on the first call on a device.) ---- */
/* K0: raw cu8/cs16 -> float samples {re, im} per complex sample, the reference's sbuf (src/demod.c:339-365:
 * process_buf_uchar / process_buf_short).  levels256 = the 256-entry table of process_buf_uchar_init
 * (src/demod.c:349-354), only read for VDL2GPU_FMT_U8. */
int vdl2gpu_launch_convert(const void *raw, uint32_t n_pairs, uint32_t sample_fmt, const float *levels256,
		float *samples_out /* [n_pairs][2] */, void *stream);
/* K4: FCS residue of n frames stored back to back (src/crc.c:21-64 as used at src/avlc.c:177) */
int vdl2gpu_launch_fcs_crc16(const uint8_t *frames, const uint32_t *offsets, const uint32_t *lens,
		uint32_t n_frames, uint16_t *residues_out, void *stream);
/* RS(255,249) errors-and-erasures decode of n blocks in place (src/rs.c:32-49); fec_octets[i] in {0,2,4,6} */
int vdl2gpu_launch_rs_verify(uint8_t *blocks /* [n][255] */, const int32_t *fec_octets, uint32_t n_blocks,
		int32_t *ret_out, void *stream);

/* K2a: phase_out[i] = (float)atan2((double)im, (double)re) and mag_out[i] = hypotf(re, im) of n_elems decimated
 * samples dec[n_elems][2] (src/demod.c:232,238,256).  exact_libm = 0: the short double-precision evaluation with a
 * Ziv rounding test the pipeline uses; 1: the general libdevice atan2 for every element.  Same floats either way. */
int vdl2gpu_launch_phase_mag(const float *dec, uint32_t n_elems, float *phase_out, float *mag_out, int exact_libm, void *stream);

/* ---- stage stubs: the three per-channel stages one at a time, on device memory the caller owns.
 * A vdl2gpu_stage is the device-resident state of n_channels vdl2_channel_t's (src/dumpvdl2.h:321-352) plus the
 * read-only tables, laid out inside ONE block of device memory that the caller allocates (256-byte aligned,
 * vdl2gpu_stage_device_bytes() bytes).  vdl2gpu_stage_create fills it (synchronous copies, no allocation); the three
 * launch stubs below then only enqueue kernels on `stream`.  Decimated samples travel between K1 and K2 in a caller
 * buffer dec[n_dec][row_stride][2] floats, row_stride = vdl2gpu_stage_row_stride(n_channels) (channels padded to 32).
 * Config fields used: sample_rate, oversample, centerfreq, n_channels, freqs, max_ppm, flags (TRACE, K1_SCALAR). ---- */
typedef struct vdl2gpu_stage vdl2gpu_stage;
size_t vdl2gpu_stage_device_bytes(uint32_t n_channels, uint32_t max_dec, uint32_t flags);
uint32_t vdl2gpu_stage_row_stride(uint32_t n_channels);
int vdl2gpu_stage_create(const vdl2gpu_config *cfg, uint32_t max_dec /* decimated samples per launch, at most */,
		void *device_mem, size_t device_bytes, vdl2gpu_stage **out);
int vdl2gpu_stage_destroy(vdl2gpu_stage *stage);
/* device address of the stage's cu8 level table, for vdl2gpu_launch_convert */
int vdl2gpu_stage_levels(vdl2gpu_stage *stage, const float **levels256_dev);
/* K1: NCO mix + 2-pole Chebyshev IIR + decimation == the sample loop of process_samples (src/demod.c:288-337, with
 * sincosf_lut :58-72, multiply :200-203, chebyshev_lpf_2pole :74-79) for every channel.  Filter, NCO and decimation
 * state persist in the stage across calls.  *n_dec_out (host) receives the number of rows written to dec_out. */
int vdl2gpu_launch_mix_iir_decimate(vdl2gpu_stage *stage, const float *samples /* [n_pairs][2] */, uint32_t n_pairs,
		float *dec_out /* [n_dec][row_stride][2] */, uint32_t *n_dec_out, void *stream);
/* K2a + K2: demod() (src/demod.c:222-286: phase ring, got_sync :105-198, D8PSK slicing) and the header part of
 * decode_vdl2_burst (src/decode.c:198-258) over n_dec decimated samples of every channel; completed bursts are
 * queued inside the stage for vdl2gpu_launch_burst_fec. */
int vdl2gpu_launch_sync_slice(vdl2gpu_stage *stage, const float *dec /* [n_dec][row_stride][2] */, uint32_t n_dec, void *stream);
/* K3 (+K4): the data part of decode_vdl2_burst (src/decode.c:259-380: descramble, de-interleave, RS, HDLC unstuff)
 * and the FCS residue of every frame, for all queued bursts.  `region` (device memory, or mapped pinned host memory;
 * 16-byte aligned) receives a 32-byte header followed by the burst records; copy it to the host and hand it to
 * vdl2gpu_parse_records. */
int vdl2gpu_launch_burst_fec(vdl2gpu_stage *stage, uint8_t *region, uint32_t region_bytes, void *stream);
/* HOST helper: records of one region -> frames in (channel, burst, idx) order through cb (`data` valid during the
 * callback).  decimated_rate = sample_rate / oversample.  Returns the number of frames or a negative error. */
int vdl2gpu_parse_records(const uint8_t *region_host, uint32_t region_bytes, uint32_t decimated_rate,
		vdl2gpu_frame_cb cb, void *user);
/* trace events of the stage (VDL2GPU_FLAG_TRACE).  Synchronises the device. */
int vdl2gpu_stage_read_events(vdl2gpu_stage *stage, vdl2gpu_event *out, uint32_t cap);

#ifdef __cplusplus
}
#endif
#endif
