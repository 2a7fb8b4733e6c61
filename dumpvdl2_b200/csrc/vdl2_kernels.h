/* vdl2_kernels.h — kernel parameter blocks and launch prototypes (internal to libvdl2gpu.so). */
#ifndef VDL2_KERNELS_H
#define VDL2_KERNELS_H
#include <stdint.h>
#include <cuda_runtime.h>
#include "vdl2_types.h"

/* Per-chunk values that change from one chunk to the next.  The host writes one of these into pinned memory and the
 * first node of the chunk's CUDA graph copies it to the device, so the captured kernel nodes never need new
 * parameters: kernels given a non-NULL `ca` take these fields from it instead of from their parameter block. */
typedef struct {
	const void *raw;             /* K0 input (device pointer) */
	uint64_t dec_base;           /* absolute index of the chunk's first decimated sample */
	uint32_t n_pairs;            /* complex samples per stream in this chunk */
	uint32_t cnt0;               /* decimation counter on entry */
	uint32_t n_dec;              /* decimated samples this chunk produces */
	uint32_t prev_n_dec;         /* ... and the previous chunk produced (its last 160 phase rows are this chunk's history) */
} vdl2_chunk_args;

/* optional per-block scheduling trace (VDL2GPU_BLOCK_TRACE=1): every block of K1 and K2 appends one record */
typedef struct {
	uint32_t kernel;             /* 1 = K1, 2 = K2 */
	uint32_t block;
	uint32_t smid;
	uint32_t pad;
	uint64_t t_start, t_end;     /* %globaltimer, ns */
} vdl2_block_rec;
typedef struct {
	uint32_t n, cap;
	vdl2_block_rec rec[1];
} vdl2_block_trace;

typedef struct {
	const float2 *samples;       /* K0 output: {re, im} per complex sample; stream s at samples + s * stream_stride */
	uint32_t n_pairs;
	uint32_t oversample;
	uint32_t cnt0;               /* decimation counter on entry (src/demod.c:289,322), same for all channels */
	uint32_t n_ch, n_chp;        /* channels; per-channel array stride = channel SLOTS (n_chp >= n_ch, multiple of 32) */
	uint32_t lanes;              /* channels per warp (1..32) for the first `full_warps` warps, lanes - 1 for the others: the
	                              * channels are dealt out evenly so that the warps of the channel kernels cover every SM
	                              * sub-partition and all live equally long (see create_impl in vdl2_host.cu) */
	uint32_t full_warps;
	float2 *dec;                 /* [n_dec][n_chp] */
	uint32_t *state;             /* [K1_NFIELDS][n_chp] */
	const float4 *lut;           /* 257 x {cos, sin, dcos*2^-16, dsin*2^-16} */
	float a0, a1, a2, b1, b2;
	float one, neg_one, two;     /* run-time 1.0f / -1.0f / 2.0f (see k1_mix_iir_decimate_packed) */
	uint32_t ch_per_stream;      /* independent-streams mode: channels [s*C, (s+1)*C) read stream s; 0 = one stream for all;
	                              * 1 = one stream per channel: `samples` is float2[n_pairs][stream_stride], time-major across streams */
	uint32_t stream_stride;      /* float2 elements between consecutive streams in `samples` (ch_per_stream == 1: per sample row) */
	const vdl2_chunk_args *ca;   /* NULL, or device pointer overriding n_pairs / cnt0 */
	vdl2_block_trace *trace_blocks;
	/* fused phase pass (vdl2_k1_fuses_phase): K1 also writes fl32(atan2(im, re)) of every decimated sample to
	 * phase[(160 + m) * n_chp + slot] and first copies the 160 history rows from phase_prev[(prev_n_dec + i) * n_chp + slot];
	 * NULL = decimated samples only (a K2a launch produces the phase plane) */
	float *phase;
	const float *phase_prev;
	uint32_t prev_n_dec;         /* overridden by ca->prev_n_dec */
} vdl2_k1_params;

/* receiver farm (vdl2gpu_create_streams): many raw streams, each with its own channels; K1 reads the raw bytes itself */
typedef struct {
	const void *raw;             /* stream s at raw + s * n_pairs * bpp bytes (overridden by ca->raw) */
	const uint32_t *list;        /* [blocks][1 + K1F_BLOCK]: per 128-slot block the number of streams its channels read, then
	                              * those streams in ascending order */
	const uint32_t *col;         /* [n_chp]: a slot's index into its block's stream list */
	const float *levels;         /* cu8 level table (src/demod.c:349-354) */
	uint32_t fmt;                /* VDL2GPU_FMT_U8 / VDL2GPU_FMT_S16_LE */
	uint32_t groups;             /* decimation groups per staged tile */
	uint32_t max_list;           /* largest stream list of any block (the row length of the staged tile) */
	uint32_t smem_bytes;         /* dynamic shared memory of a block, vdl2_k1_farm_smem_bytes */
} vdl2_k1_farm;
#define K1F_BLOCK 128

typedef struct {
	const float2 *dec;
	float *phase;                /* [160 + n_dec][n_chp]: rows 0..159 = last 160 phases of the previous chunks */
	float *mag;                  /* [n_dec][n_chp] */
	float *hist_tmp;             /* [160][n_chp] scratch for the history shift of short chunks */
	uint32_t n_dec;
	uint32_t n_ch, n_chp;
	uint32_t lanes, full_warps;  /* channel slot mapping, as in vdl2_k1_params */
	uint64_t dec_base;           /* absolute index of dec[0] */
	uint32_t *state;             /* [K2_NFIELDS][n_chp] */
	float *ring;                 /* [160][n_chp] */
	const vdl2_tables *tables;
	float max_ppm;
	uint32_t s27;
	vdl2_burst_slot *pool;
	int32_t *free_list;
	uint32_t *ready;
	vdl2_queue_ctl *ctl;
	void *events;
	uint32_t event_cap;
	uint32_t trace;
	uint32_t variant;            /* walk variant, see vdl2_launch_k2 */
	uint32_t k2a_mode;           /* 0: libdevice atan2 for every sample; 1: vdl2_phase_fast with the Ziv fall-back */
	const vdl2_chunk_args *ca;   /* NULL, or device pointer overriding n_dec / dec_base */
	vdl2_block_trace *trace_blocks;
} vdl2_k2_params;

/* K2a in its resident form (k2a_phase_mag_warps): warp w computes phase and magnitude of slots [32 w, 32 w + 32) for every
 * decimated sample of the chunk and first carries the last 160 phase rows of the previous chunk's plane over */
typedef struct {
	const float2 *dec;           /* [n_dec][n_chp] */
	float *phase;                /* this chunk's plane [160 + n_dec][n_chp] */
	float *mag;                  /* [n_dec][n_chp], or NULL: the walk (variant 5) takes the magnitudes from the samples itself */
	const float *phase_prev;     /* the previous chunk's plane (the other of the two) */
	uint32_t n_dec, prev_n_dec;
	uint32_t n_ch, n_chp, lanes, full_warps;
	uint32_t mode;               /* 0 libdevice atan2 / IEEE sqrt for every sample, 1 the Ziv-guarded short forms */
	uint32_t split;              /* time slices per chunk: the grid is `split` x (one block per 128 slots) */
	const vdl2_chunk_args *ca;
} vdl2_k2a_params;

typedef struct {
	vdl2_burst_slot *pool;
	int32_t *free_list;
	const uint32_t *ready;
	vdl2_queue_ctl *ctl;
	const vdl2_tables *tables;
	uint8_t *out;                /* device address of the mapped pinned output region (header + records) */
	uint32_t out_cap;            /* bytes available for records */
	uint32_t n_chp;
	uint32_t *counters;          /* [VDL2_NUM_COUNTERS][n_chp] */
} vdl2_k3_params;

#ifdef __cplusplus
extern "C" {
#endif
/* once per device (thread-safe): the shared-memory carve-out every kernel of the chain asks for */
int vdl2_kernels_init_device(int device);
/* n_streams streams of n_pairs samples each: raw stream s at raw + s * raw_stride bytes, output at out2 + s * out_stride float2 */
int vdl2_launch_k0(const void *raw, uint32_t n_pairs, uint32_t fmt, const float *levels, float *out2, uint32_t n_streams,
		uint32_t raw_stride, uint32_t out_stride, const vdl2_chunk_args *ca, cudaStream_t st);
/* one stream per channel: raw[s][i] -> out2[i][out_stride] float2, time-major across streams */
int vdl2_launch_k0_lanes(const void *raw, uint32_t n_pairs, uint32_t fmt, const float *levels, float *out2, uint32_t n_streams,
		uint32_t raw_stride, uint32_t out_stride, uint32_t lanes, uint32_t full_warps, const vdl2_chunk_args *ca, cudaStream_t st);
int vdl2_launch_k1(const vdl2_k1_params *p, int force_scalar, int variant, cudaStream_t st);
/* receiver farm: shared-memory layout of k1_mix_iir_decimate_farm for these shapes (f->groups, f->smem_bytes are set);
 * returns 0 or cudaErrorInvalidValue when even one group per tile does not fit the block's budget */
int vdl2_k1_farm_layout(uint32_t oversample, uint32_t fmt, uint32_t max_list, vdl2_k1_farm *f);
int vdl2_launch_k1_farm(const vdl2_k1_params *p, const vdl2_k1_farm *f, cudaStream_t st);
/* whether vdl2_launch_k1 with these arguments runs a kernel that honours p->phase (the pipelined packed kernel with
 * 128-channel blocks); everything else leaves the phase plane to K2a */
int vdl2_k1_fuses_phase(uint32_t oversample, uint32_t ch_per_stream, int force_scalar, int variant);
int vdl2_launch_copy_hist(const vdl2_k2_params *p, cudaStream_t st);
int vdl2_launch_k2a(const vdl2_k2_params *p, cudaStream_t st);
int vdl2_launch_k2a_warps(const vdl2_k2a_params *p, cudaStream_t st);
int vdl2_launch_k2(const vdl2_k2_params *p, cudaStream_t st);
int vdl2_launch_k3(const vdl2_k3_params *p, uint32_t grid, cudaStream_t st);
int vdl2_launch_k4(const uint8_t *frames, const uint32_t *offsets, const uint32_t *lens, uint32_t n, uint16_t *out, cudaStream_t st);
int vdl2_launch_rs(uint8_t *blocks, const int32_t *fec_octets, uint32_t n, int32_t *ret, const vdl2_tables *tables, cudaStream_t st);
#ifdef __cplusplus
}
#endif
#endif
