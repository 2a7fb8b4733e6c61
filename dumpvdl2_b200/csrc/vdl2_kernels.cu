/*
 * vdl2_kernels.cu — sm_100a kernels of libvdl2gpu.so and their extern "C" launch stubs.
 *
 *   K0  k0_convert            raw cu8/cs16 -> float samples        src/demod.c:339-365
 *   K1  k1_mix_iir_decimate   NCO mix + 2-pole IIR + decimate      src/demod.c:58-79,200-203,288-337
 *   K2a k2a_phase_mag         atan2 / hypot of every decimated sample  src/demod.c:232,238,256
 *   K2  k2_sync_slice         preamble sync, D8PSK slicing, header src/demod.c:105-198,222-286; src/decode.c:198-258
 *   K3  k3_burst_fec          descramble, de-interleave, RS, HDLC  src/decode.c:259-380; src/rs.c; src/libfec; src/bitstream.c
 *   K4  (inside K3)           AVLC FCS residue per frame           src/crc.c:21-64
 *
 * Unit of parallelism: K0, K2a element; K1/K2 one thread per VDL2 channel (32 channels per warp, the sample
 * stream is broadcast to the warp from shared memory); K3 one thread block per burst.
 * No tensor cores: there is no dense contraction on this path.  Built with -fmad=false; all float
 * arithmetic additionally goes through explicit round-to-nearest intrinsics / PTX.
 */
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include <mutex>
#include <type_traits>
#include "vdl2_core.cuh"
#include "vdl2_fastmath.cuh"
#include "vdl2_kernels.h"

/* block scheduling trace: where and when a block ran (diagnostic, off unless the context was created with VDL2GPU_BLOCK_TRACE=1) */
__device__ __forceinline__ uint64_t vdl2_globaltimer() { uint64_t t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
__device__ __forceinline__ uint32_t vdl2_smid() { uint32_t s; asm volatile("mov.u32 %0, %%smid;" : "=r"(s)); return s; }
__device__ __forceinline__ int vdl2_trace_begin(vdl2_block_trace *t, uint32_t kernel) {
	if(t == nullptr) return -1;
	const uint32_t k = atomicAdd(&t->n, 1u);
	if(k >= t->cap) return -1;
	t->rec[k].kernel = kernel; t->rec[k].block = blockIdx.x; t->rec[k].smid = vdl2_smid(); t->rec[k].t_start = vdl2_globaltimer(); t->rec[k].t_end = 0;
	return (int)k;
}
__device__ __forceinline__ void vdl2_trace_end(vdl2_block_trace *t, int k) { if(k >= 0) t->rec[k].t_end = vdl2_globaltimer(); }

/* slot (index into every per-channel array) -> public channel number and activity: a warp holds `lanes` channels in its
 * first `lanes` lanes */
__device__ __forceinline__ bool vdl2_slot_channel(uint32_t slot, uint32_t lanes, uint32_t full_warps, uint32_t n_ch, uint32_t &chan) {
	const uint32_t lane = slot & 31u, w = slot >> 5;
	const uint32_t mine = w < full_warps ? lanes : lanes - 1u;                 /* channels of this warp */
	chan = (w < full_warps ? w * lanes : full_warps * lanes + (w - full_warps) * (lanes - 1u)) + lane;
	return lane < mine && chan < n_ch;
}

/* ------------------------------------------------------------------------------------------------
 * K0: sample conversion.  Output: float2 {re, im} per complex sample (src/demod.c:339-365).
 * ---------------------------------------------------------------------------------------------- */
/* one interleaved complex sample -> {re, im}; every kernel that reads raw input converts through these two */
__device__ __forceinline__ float2 vdl2_iq_u8(uchar2 v, const float *__restrict__ levels) {      /* src/demod.c:343-345, table :349-354 */
	return make_float2(__ldg(&levels[v.x]), __ldg(&levels[v.y]));
}
__device__ __forceinline__ float2 vdl2_iq_s16(short2 v) {                                        /* src/demod.c:361-363 */
	return make_float2(__fdiv_rn((float)v.x, 32768.0f), __fdiv_rn((float)v.y, 32768.0f));
}

__global__ void __launch_bounds__(256) k0_convert(const uint8_t *__restrict__ raw0, uint32_t n_pairs_p, uint32_t fmt,
		const float *__restrict__ levels, float2 *__restrict__ out0, uint32_t raw_stride, uint32_t out_stride,
		const vdl2_chunk_args *__restrict__ ca) {
	const uint32_t n_pairs = ca ? ca->n_pairs : n_pairs_p;
	const uint8_t *raw = (ca ? static_cast<const uint8_t *>(ca->raw) : raw0) + (size_t)blockIdx.y * raw_stride;   /* stream blockIdx.y */
	float2 *out = out0 + (size_t)blockIdx.y * out_stride;
	uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= n_pairs) return;
	float2 v;
	if(fmt == 0) {
		v = vdl2_iq_u8(reinterpret_cast<const uchar2 *>(raw)[i], levels);
	} else if(fmt == 1) {
		v = vdl2_iq_s16(reinterpret_cast<const short2 *>(raw)[i]);
	} else {
		/* planar cs16: n_pairs I values followed by n_pairs Q values, the shape the SDRplay APIs deliver
		 * (src/sdrplay.c:72, src/sdrplay3.c callbacks); same arithmetic as the interleaved case, the
		 * host-side interleave loop of src/sdrplay.c:95-121 is not needed */
		const short *pl = reinterpret_cast<const short *>(raw);
		v.x = __fdiv_rn((float)pl[i], 32768.0f);
		v.y = __fdiv_rn((float)pl[n_pairs + i], 32768.0f);
	}
	out[i] = v;
}

/* K0 for the one-stream-per-channel layout: raw[s][i] -> out[i][s] float2 {re, im}, i.e. TIME-major across streams, so
 * that the 32 lanes of a K1 warp (32 different streams) read 256 contiguous bytes per sample.  32x32 tile through
 * shared memory: reads run along the samples of a stream, writes along the streams of a sample. */
__global__ void __launch_bounds__(1024) k0_convert_lanes(const uint8_t *__restrict__ raw0, uint32_t n_pairs_p, uint32_t fmt,
		const float *__restrict__ levels, float2 *__restrict__ out, uint32_t n_streams, uint32_t raw_stride, uint32_t out_stride,
		uint32_t lanes, uint32_t full_warps, const vdl2_chunk_args *__restrict__ ca) {
	__shared__ float2 tile[32][33];
	const uint32_t n_pairs = ca ? ca->n_pairs : n_pairs_p;
	const uint8_t *raw = ca ? static_cast<const uint8_t *>(ca->raw) : raw0;
	const uint32_t tx = threadIdx.x, ty = threadIdx.y;
	const uint32_t i_in = blockIdx.x * 32u + tx;
	uint32_t s_in;                                    /* stream = channel that lives in column (slot) blockIdx.y * 32 + ty */
	const bool have = vdl2_slot_channel(blockIdx.y * 32u + ty, lanes, full_warps, n_streams, s_in);
	float2 v = make_float2(0.f, 0.f);
	if(have && i_in < n_pairs) {
		const uint8_t *r = raw + (size_t)s_in * raw_stride;
		if(fmt == 0) v = vdl2_iq_u8(reinterpret_cast<const uchar2 *>(r)[i_in], levels);
		else v = vdl2_iq_s16(reinterpret_cast<const short2 *>(r)[i_in]);
	}
	tile[ty][tx] = v;
	__syncthreads();
	const uint32_t i_out = blockIdx.x * 32u + ty, s_out = blockIdx.y * 32u + tx;
	if(i_out < n_pairs && s_out < out_stride) out[(size_t)i_out * out_stride + s_out] = tile[tx][ty];
}

/* ------------------------------------------------------------------------------------------------
 * K1, plain per-sample form (reference for the pipelined kernel; selected by VDL2GPU_FLAG_K1_SCALAR
 * and for oversample values without a specialisation).
 * ---------------------------------------------------------------------------------------------- */
#define K1_TILE 1024

__device__ __forceinline__ void k1_load_state(const vdl2_k1_params &p, uint32_t ch, float &xr1, float &xr2, float &xi1,
		float &xi2, float &yr1, float &yr2, float &yi1, float &yi2, uint32_t &phi, uint32_t &dphi) {
	const uint32_t *st = p.state;
	const uint32_t s = p.n_chp;
	xr1 = __uint_as_float(st[K1_XR1 * s + ch]); xr2 = __uint_as_float(st[K1_XR2 * s + ch]);
	xi1 = __uint_as_float(st[K1_XI1 * s + ch]); xi2 = __uint_as_float(st[K1_XI2 * s + ch]);
	yr1 = __uint_as_float(st[K1_YR1 * s + ch]); yr2 = __uint_as_float(st[K1_YR2 * s + ch]);
	yi1 = __uint_as_float(st[K1_YI1 * s + ch]); yi2 = __uint_as_float(st[K1_YI2 * s + ch]);
	phi = st[K1_PHI * s + ch]; dphi = st[K1_DPHI * s + ch];
}

__device__ __forceinline__ void k1_store_state(const vdl2_k1_params &p, uint32_t ch, float xr1, float xr2, float xi1,
		float xi2, float yr1, float yr2, float yi1, float yi2, uint32_t phi) {
	uint32_t *st = p.state;
	const uint32_t s = p.n_chp;
	st[K1_XR1 * s + ch] = __float_as_uint(xr1); st[K1_XR2 * s + ch] = __float_as_uint(xr2);
	st[K1_XI1 * s + ch] = __float_as_uint(xi1); st[K1_XI2 * s + ch] = __float_as_uint(xi2);
	st[K1_YR1 * s + ch] = __float_as_uint(yr1); st[K1_YR2 * s + ch] = __float_as_uint(yr2);
	st[K1_YI1 * s + ch] = __float_as_uint(yi1); st[K1_YI2 * s + ch] = __float_as_uint(yi2);
	st[K1_PHI * s + ch] = phi & 0xFFFFFFu;
}

/* independent-streams mode: all channels of a block belong to stream (first channel / ch_per_stream); a block never
 * straddles two streams because ch_per_stream is a multiple of the block size (checked by the launcher) */
__device__ __forceinline__ const float2 *k1_stream_of(const vdl2_k1_params &p, uint32_t first_ch) {
	return p.ch_per_stream ? p.samples + (size_t)(first_ch / p.ch_per_stream) * p.stream_stride : p.samples;
}

template<int BLOCK>
__global__ void __launch_bounds__(BLOCK) k1_mix_iir_decimate_scalar(vdl2_k1_params p) {
	__shared__ float4 s_lut[257];
	__shared__ float2 s_tile[K1_TILE];
	const uint32_t tid = threadIdx.x;
	const uint32_t ch = blockIdx.x * BLOCK + tid;
	uint32_t chan;
	const bool active = vdl2_slot_channel(ch, p.lanes, p.full_warps, p.n_ch, chan);
	const uint32_t n_pairs = p.ca ? p.ca->n_pairs : p.n_pairs, cnt0 = p.ca ? p.ca->cnt0 : p.cnt0;
	const float2 *samples = k1_stream_of(p, blockIdx.x * BLOCK);
	for(uint32_t i = tid; i < 257; i += BLOCK) s_lut[i] = p.lut[i];
	float xr1 = 0, xr2 = 0, xi1 = 0, xi2 = 0, yr1 = 0, yr2 = 0, yi1 = 0, yi2 = 0;
	uint32_t phi = 0, dphi = 0;
	if(active) k1_load_state(p, ch, xr1, xr2, xi1, xi2, yr1, yr2, yi1, yi2, phi, dphi);
	uint32_t cnt = cnt0, m = 0;
	const float a0 = p.a0, a1 = p.a1, a2 = p.a2, b1 = p.b1, b2 = p.b2;
	for(uint32_t base = 0; base < n_pairs; base += K1_TILE) {
		const uint32_t n = min((uint32_t)K1_TILE, n_pairs - base);
		__syncthreads();
		for(uint32_t i = tid; i < n; i += BLOCK) s_tile[i] = samples[base + i];
		__syncthreads();
		if(!active) continue;
		for(uint32_t k = 0; k < n; k++) {
			const float2 s = s_tile[k];
			/* NCO: src/demod.c:58-72 (table entry = {cos, sin, dcos*2^-16, dsin*2^-16}) */
			const float4 e = s_lut[(phi >> 16) & 0xFFu];
			const float fr = (float)(phi & 0xFFFFu);
			const float cs = __fadd_rn(e.x, __fmul_rn(e.z, fr));
			const float sn = __fadd_rn(e.y, __fmul_rn(e.w, fr));
			phi += dphi;
			/* complex multiply: src/demod.c:200-203 */
			const float re = __fsub_rn(__fmul_rn(s.x, cs), __fmul_rn(s.y, sn));
			const float im = __fadd_rn(__fmul_rn(s.y, cs), __fmul_rn(s.x, sn));
			/* biquad, evaluation order of src/demod.c:74-79 */
			float r = __fmul_rn(a0, re);
			r = __fadd_rn(r, __fadd_rn(__fmul_rn(a1, xr1), __fmul_rn(a2, xr2)));
			r = __fadd_rn(r, __fadd_rn(__fmul_rn(b1, yr1), __fmul_rn(b2, yr2)));
			float q = __fmul_rn(a0, im);
			q = __fadd_rn(q, __fadd_rn(__fmul_rn(a1, xi1), __fmul_rn(a2, xi2)));
			q = __fadd_rn(q, __fadd_rn(__fmul_rn(b1, yi1), __fmul_rn(b2, yi2)));
			xr2 = xr1; xr1 = re; yr2 = yr1; yr1 = r;
			xi2 = xi1; xi1 = im; yi2 = yi1; yi1 = q;
			if(++cnt == p.oversample) {                   /* src/demod.c:322-328 */
				cnt = 0;
				p.dec[(size_t)m * p.n_chp + ch] = make_float2(r, q);
				m++;
			}
		}
	}
	if(active) k1_store_state(p, ch, xr1, xr2, xi1, xi2, yr1, yr2, yi1, yi2, phi);
}

/* ------------------------------------------------------------------------------------------------
 * K1, pipelined form.  I and Q ride in the two halves of one f32x2 register pair (FMUL2/FFMA2 on
 * sm_100a): the two biquads of src/demod.c:319-320 become one instruction stream.  ptxas contracts
 * mul.rn.f32x2 + add.rn.f32x2 into FFMA2 even with --fmad=false, which would change the rounding,
 * so every addition is issued as fma(x, ONE, y) with ONE a run-time 1.0f the optimiser cannot see
 * through: x*1+y rounds exactly like x+y and a product feeding it cannot be fused any further.
 * The loop over one decimation group (OS samples) is fully unrolled so that the NCO/mix work of later
 * samples fills the issue slots left by the serial y[n-1] -> y[n] recurrence.
 * ---------------------------------------------------------------------------------------------- */
typedef unsigned long long u64;
__device__ __forceinline__ u64 f2_mul(u64 a, u64 b) { u64 r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ u64 f2_fma(u64 a, u64 b, u64 c) { u64 r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
__device__ __forceinline__ u64 f2_pack(float lo, float hi) { u64 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
#pragma nv_diag_suppress 550      /* the unused half of an unpacked pair */
__device__ __forceinline__ float f2_lo(u64 v) { float a, b; asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); return a; }
__device__ __forceinline__ float f2_hi(u64 v) { float a, b; asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); return b; }
#pragma nv_diag_default 550
__device__ __forceinline__ float f1_fma(float a, float b, float c) { float r; asm("fma.rn.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c)); return r; }

struct k1_packed_consts { u64 ONE, SGN, A0, A1, A2, B1, B2, TWO; float one, neg_one; };

/* mixer, src/demod.c:200-203: with P = (re, im) * cos and Q = (re, im) * sin (two packed products by a broadcast scalar)
 *   x0 = (P.re - Q.im, P.im + Q.re) = (re*cos - im*sin, im*cos + re*sin),
 * each product and each sum rounded once, as in the reference; the two sums are scalar fma(q, -+1, p) so that the
 * sample never needs a swapped copy. */
__device__ __forceinline__ u64 k1_mix(const float2 s, const u64 CS, const k1_packed_consts &c) {
	const float cs = f2_lo(CS), sn = f2_hi(CS);
	const u64 S2 = f2_pack(s.x, s.y);
	const u64 P = f2_mul(S2, f2_pack(cs, cs)), Q = f2_mul(S2, f2_pack(sn, sn));
	return f2_pack(f1_fma(f2_hi(Q), c.neg_one, f2_lo(P)), f1_fma(f2_lo(Q), c.one, f2_hi(P)));
}

/* one input sample through NCO, mixer and filter; returns the filtered (I,Q) pair */
__device__ __forceinline__ u64 k1_packed_step(const float2 s, const float4 e, uint32_t &phi, const uint32_t dphi,
		u64 &x1, u64 &x2, u64 &y1, u64 &y2, const k1_packed_consts &c) {
	const float fr = (float)(phi & 0xFFFFu);
	phi += dphi;
	const u64 CS = f2_fma(f2_mul(f2_pack(e.z, e.w), f2_pack(fr, fr)), c.ONE, f2_pack(e.x, e.y));   /* (cos, sin) */
	const u64 x0 = k1_mix(s, CS, c);
	const u64 t = f2_fma(f2_mul(c.A1, x1), c.ONE, f2_mul(c.A2, x2));
	const u64 r = f2_fma(f2_mul(c.A0, x0), c.ONE, t);
	const u64 u = f2_fma(f2_mul(c.B1, y1), c.ONE, f2_mul(c.B2, y2));
	const u64 y0 = f2_fma(r, c.ONE, u);
	x2 = x1; x1 = x0; y2 = y1; y1 = y0;
	return y0;
}

/* TMA (bulk asynchronous copy) staging of the sample stream: one elected lane asks the copy engine for the next
 * tile (cp.async.bulk global -> shared, completion counted in bytes on an mbarrier) while the block works on the
 * current one; two tiles in flight hide the L2 round trip completely.  SASS: UBLKCP + SYNCS. */
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
	asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tma_load_tile(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
	asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
	asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
			:: "r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
	asm volatile("{\n\t.reg .pred p;\n\tWAIT_%=:\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t@p bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}"
			:: "r"(smem_u32(bar)), "r"(parity) : "memory");
}

#define K1P_TILE_GROUPS(OS) ((640 / (OS)) & ~1)  /* <= 640 samples = 5 KB of float2 per tile; an even number of groups keeps every
                                                  * tile an even number of samples = a multiple of 16 bytes for the bulk copy */

/* BLOCK = 128: the four warps of an SM's four sub-partitions share one block, i.e. one copy of the sample tiles and of
 * the NCO table.  The table is then kept EIGHT times (33 KB), copy c holding entry i at float4 index 8 i + c, and lane l
 * reads copy l mod 8: the eight lanes of a quarter-warp always hit eight different 16-byte bank groups, so the look-up
 * is conflict-free whatever the 32 phases are (4 wavefronts per LDS.128, the minimum for 512 bytes).  With a single
 * copy, 32 unrelated phases cost ~10 wavefronts per look-up and the four warps of an SM saturate its shared-memory
 * pipe (measured: 6.6 ms instead of 5.1 ms per launch once the channels of a warp sit on different frequencies).
 * BLOCK = 32 keeps one warp per block and a single table copy; the launcher uses it when a 128-channel block would
 * straddle two streams in independent-streams mode. */
/* NCO table look-up of the hot loops: byte offset of entry (phase >> 16) & 0xFF in this lane's copy of the table, formed
 * as ((phase >> 9) & 0x7F80) | lane_bytes (NLUT = 8: 128 bytes per entry, the copy in bits 4..6) resp. (phase >> 12) & 0xFF0
 * (single copy) - one shift and one three-input logic operation, the table's shared-memory address folded into the load.
 * Written via indices the compiler spent a second logic operation and an address add on it. */
template<int NLUT>
__device__ __forceinline__ float4 k1_lut_entry(const float4 *s_lut, uint32_t phase, uint32_t lane_bytes) {
	const uint32_t off = NLUT == 8 ? (((phase >> 9) & 0x7F80u) | lane_bytes) : ((phase >> 12) & 0xFF0u);
	return *reinterpret_cast<const float4 *>(reinterpret_cast<const unsigned char *>(s_lut) + off);
}

/* break-point table of vdl2_phase_fast: constant memory, copied to shared memory by the kernels that use it */
__constant__ double c_atan_tab[VDL2_ATAN_TABLE_DOUBLES] = VDL2_ATAN_TABLE_INIT;

/* PH (fused phase pass, opt-in: VDL2GPU_FUSE_PHASE=1): the thread also produces the phase of every decimated sample it
 * writes.  In the tile loop the atan2 of group g-1's output is written out as straight-line code at the top of group g's
 * unrolled body (vdl2_phase_fast_nb: ~20 FP64 operations and their conversions, no branch) so that it can be scheduled
 * into the group's FP32 filter recurrence; the Ziv fall-back (about one sample in a million) and the store come at the
 * end of the body.  Measured: 6.4 instead of 5.0 ms per launch, more than the separate K2a pass costs (DESIGN.md section 4). */
__device__ __forceinline__ float k1_phase_exact(float re, float im, const double *tab) {
	int slow;
	float f = vdl2_phase_fast_nb(re, im, tab, &slow);
	if(slow) f = vdl2_phase_of(re, im);
	return f;
}

template<int OS, int BLOCK, int BATCH, bool SYM, bool PH = false>
__global__ void __launch_bounds__(BLOCK) k1_mix_iir_decimate_packed(vdl2_k1_params p) {
	constexpr int TG = K1P_TILE_GROUPS(OS);
	constexpr int NLUT = BLOCK >= 128 ? 8 : 1;                    /* table copies */
	static_assert(!PH || (BATCH != 0 && BLOCK >= VDL2_ATAN_TABLE_DOUBLES), "fused phase pass: pipelined kernel only");
	__shared__ double s_atan[PH ? VDL2_ATAN_TABLE_DOUBLES : 1];
	__shared__ float4 s_lut[257 * NLUT];
	__shared__ __align__(128) float2 s_tiles[2][TG * OS + 2];
	__shared__ __align__(8) uint64_t s_bar[2];
	const uint32_t tid = threadIdx.x;
	const int trace_k = tid == 0 ? vdl2_trace_begin(p.trace_blocks, 1) : -1;
	const uint32_t ch = blockIdx.x * BLOCK + tid;
	uint32_t chan;
	const bool active = vdl2_slot_channel(ch, p.lanes, p.full_warps, p.n_ch, chan);
	const uint32_t n_pairs = p.ca ? p.ca->n_pairs : p.n_pairs, cnt0 = p.ca ? p.ca->cnt0 : p.cnt0;
	const float2 *samples = k1_stream_of(p, blockIdx.x * BLOCK);
	for(uint32_t i = tid; i < 257 * NLUT; i += BLOCK) s_lut[i] = p.lut[i / NLUT];
	const float4 *lut = s_lut + (NLUT > 1 ? (tid & (NLUT - 1)) : 0);       /* this lane's copy; entry i at lut[i * NLUT] */
	const uint32_t lane_bytes = NLUT > 1 ? (tid & (NLUT - 1)) * 16u : 0u;
	if(tid == 0) { mbar_init(&s_bar[0], 1); mbar_init(&s_bar[1], 1); mbar_fence_init(); }
	if(PH && tid < VDL2_ATAN_TABLE_DOUBLES) s_atan[tid] = c_atan_tab[tid];
	float *phase = nullptr;                                   /* this slot's column, row 0 = first sample of the chunk */
	if(PH && active) {
		/* history prefix: the last 160 phase rows of the previous chunk (src/demod.c:105-198 looks 150 samples back) */
		const uint32_t prev_n_dec = p.ca ? p.ca->prev_n_dec : p.prev_n_dec;
		const float *src = p.phase_prev + (size_t)prev_n_dec * p.n_chp + ch;
		float *dst = p.phase + ch;
#pragma unroll 8
		for(uint32_t i = 0; i < VDL2_SYNC_BUFLEN; i++) dst[(size_t)i * p.n_chp] = src[(size_t)i * p.n_chp];
		phase = p.phase + (size_t)VDL2_SYNC_BUFLEN * p.n_chp + ch;
	}
	float xr1 = 0, xr2 = 0, xi1 = 0, xi2 = 0, yr1 = 0, yr2 = 0, yi1 = 0, yi2 = 0;
	uint32_t phi = 0, dphi = 0;
	if(active) k1_load_state(p, ch, xr1, xr2, xi1, xi2, yr1, yr2, yi1, yi2, phi, dphi);
	u64 x1 = f2_pack(xr1, xi1), x2 = f2_pack(xr2, xi2), y1 = f2_pack(yr1, yi1), y2 = f2_pack(yr2, yi2);
	k1_packed_consts c;
	c.ONE = f2_pack(p.one, p.one); c.SGN = f2_pack(p.neg_one, p.one);
	c.A0 = f2_pack(p.a0, p.a0); c.A1 = f2_pack(p.a1, p.a1); c.A2 = f2_pack(p.a2, p.a2);
	c.B1 = f2_pack(p.b1, p.b1); c.B2 = f2_pack(p.b2, p.b2); c.TWO = f2_pack(p.two, p.two);
	c.one = p.one; c.neg_one = p.neg_one;
	/* SYM: the feed-forward taps of this filter design are {A0, 2*A0, A0} (checked on the host).  A1*x[n-1] and
	 * A2*x[n-2] are then exactly 2*(A0*x[n-1]) and A0*x[n-2], products the previous two steps already formed
	 * (doubling is exact; no operand can be subnormal here, see DESIGN.md), so two multiplies per sample go away:
	 * t = fma(P1, 2, P2) rounds once, exactly like A1*x1 + A2*x2. */
	u64 P1 = f2_mul(c.A0, x1), P2 = f2_mul(c.A0, x2);
	__syncthreads();

	uint32_t cnt = cnt0, m = 0, pos = 0;
	/* head: samples up to the first decimation-group boundary, straight from global memory */
	const uint32_t head = min(n_pairs, (OS - cnt0 % OS) % OS);
	if(active) {
		for(; pos < head; pos++) {
			u64 y0 = k1_packed_step(samples[pos], lut[((phi >> 16) & 0xFFu) * NLUT], phi, dphi, x1, x2, y1, y2, c);
			if(++cnt == OS) {
				cnt = 0;
				p.dec[(size_t)m * p.n_chp + ch] = make_float2(f2_lo(y0), f2_hi(y0));
				if(PH) phase[(size_t)m * p.n_chp] = k1_phase_exact(f2_lo(y0), f2_hi(y0), s_atan);
				m++;
			}
		}
	}
	/* same bookkeeping for every lane, active or not */
	pos = head;
	m = (cnt0 + head) / OS;
	cnt = (cnt0 + head) % OS;
	P1 = f2_mul(c.A0, x1); P2 = f2_mul(c.A0, x2);            /* after the head samples */
	/* body: whole groups, staged through shared memory tile by tile */
	const uint32_t n_groups = (n_pairs - pos) / OS;
	const uint32_t n_tiles = (n_groups + TG - 1) / TG;
	/* The bulk copy wants 16-byte aligned addresses and sizes, a sample is 8 bytes: when the first body sample sits on an
	 * odd element (odd decimation phase on entry), every tile is fetched from one sample earlier and read from element 1
	 * on (`mis`); an odd trailing sample of the last tile is copied by hand.  Tile t lands in buffer t & 1, its mbarrier
	 * phase is (t >> 1) & 1. */
	const uint32_t mis = (uint32_t)((reinterpret_cast<uintptr_t>(samples + pos) >> 3) & 1u);
	auto request_tile = [&](uint32_t t, uint32_t buf) {              /* thread 0 only */
		const uint32_t n = min((uint32_t)TG, n_groups - t * TG) * OS + mis;
		const float2 *src = samples + head + (size_t)t * TG * OS - mis;
		tma_load_tile(s_tiles[buf], src, (n & ~1u) * (uint32_t)sizeof(float2), &s_bar[buf]);
		if(n & 1u) s_tiles[buf][n - 1] = src[n - 1];
	};
	if(tid == 0)
		for(uint32_t t = 0; t < 2 && t < n_tiles; t++) request_tile(t, t);
	__syncthreads();
	/* the tile loop, compiled twice: with the tile known to start on element 0 the compiler fetches two samples per
	 * LDS.128; the misaligned case (odd decimation phase on entry) reads from element 1 with 64-bit loads */
	u64 yprev = f2_pack(1.0f, 0.0f);                              /* output of the previous group, its phase still owed */
	bool owed = false;
	auto tile_loop = [&](auto MIS) {
	for(uint32_t g0 = 0, tile = 0; g0 < n_groups; g0 += TG, tile++) {
		const uint32_t ng = min((uint32_t)TG, n_groups - g0);
		const float2 *s_tile = s_tiles[tile & 1u] + decltype(MIS)::value;
		mbar_wait(&s_bar[tile & 1u], (tile >> 1) & 1u);
		if(active) {
			for(uint32_t g = 0; g < ng; g++) {
				const float2 *sp = &s_tile[g * OS];
				u64 y0 = 0;
				float ph_prev = 0.0f;
				int ph_slow = 0;
				if(PH) ph_prev = vdl2_phase_fast_nb(f2_lo(yprev), f2_hi(yprev), s_atan, &ph_slow);
				if(BATCH == 0) {
#pragma unroll
					for(int k = 0; k < OS; k++)
						y0 = k1_packed_step(sp[k], lut[((phi >> 16) & 0xFFu) * NLUT], phi, dphi, x1, x2, y1, y2, c);
				} else {
					/* software pipeline written out over the unrolled group: loads run LA samples ahead of the
					 * mixer, the mixer MA samples ahead of the filter recurrence */
					constexpr int LA = BATCH, MA = BATCH / 2;
					float2 S[OS];
					float4 E[OS];
					float FR[OS];
					u64 X0[OS];
#pragma unroll
					for(int k = -LA; k < OS; k++) {
						const int kl = k + LA, km = k + MA;
						if(kl < OS) {
							const uint32_t ph = phi + (uint32_t)kl * dphi;
							E[kl] = k1_lut_entry<NLUT>(s_lut, ph, lane_bytes);
							FR[kl] = (float)(ph & 0xFFFFu);
							S[kl] = sp[kl];
						}
						if(km >= 0 && km < OS) {
							const u64 CS = f2_fma(f2_mul(f2_pack(E[km].z, E[km].w), f2_pack(FR[km], FR[km])), c.ONE, f2_pack(E[km].x, E[km].y));
							X0[km] = k1_mix(S[km], CS, c);
						}
						if(k >= 0) {
							const u64 x0 = X0[k];
							u64 r;
							if(SYM) {
								const u64 P0 = f2_mul(c.A0, x0);
								r = f2_fma(P0, c.ONE, f2_fma(P1, c.TWO, P2));
								P2 = P1; P1 = P0;
							} else {
								const u64 t = f2_fma(f2_mul(c.A1, x1), c.ONE, f2_mul(c.A2, x2));
								r = f2_fma(f2_mul(c.A0, x0), c.ONE, t);
							}
							const u64 u = f2_fma(f2_mul(c.B1, y1), c.ONE, f2_mul(c.B2, y2));
							y0 = f2_fma(r, c.ONE, u);
							x2 = x1; x1 = x0; y2 = y1; y1 = y0;
						}
					}
					phi += (uint32_t)OS * dphi;
				}
				p.dec[(size_t)(m + g) * p.n_chp + ch] = make_float2(f2_lo(y0), f2_hi(y0));
				if(PH) {
					if(owed) {
						if(ph_slow) ph_prev = vdl2_phase_of(f2_lo(yprev), f2_hi(yprev));
						phase[(size_t)(m + g - 1u) * p.n_chp] = ph_prev;
					}
					yprev = y0;
					owed = true;
				}
			}
		}
		m += ng;
		pos += ng * OS;
		__syncthreads();                                           /* every warp is done with this buffer */
		if(tid == 0 && tile + 2 < n_tiles) request_tile(tile + 2, tile & 1u);
	}
	};
	if(mis) tile_loop(std::integral_constant<int, 1>{}); else tile_loop(std::integral_constant<int, 0>{});
	if(PH && active && owed) phase[(size_t)(m - 1u) * p.n_chp] = k1_phase_exact(f2_lo(yprev), f2_hi(yprev), s_atan);
	/* tail: fewer than OS samples left */
	if(active) {
		for(; pos < n_pairs; pos++) {
			u64 y0 = k1_packed_step(samples[pos], lut[((phi >> 16) & 0xFFu) * NLUT], phi, dphi, x1, x2, y1, y2, c);
			if(++cnt == OS) {
				cnt = 0;
				p.dec[(size_t)m * p.n_chp + ch] = make_float2(f2_lo(y0), f2_hi(y0));
				if(PH) phase[(size_t)m * p.n_chp] = k1_phase_exact(f2_lo(y0), f2_hi(y0), s_atan);
				m++;
			}
		}
		k1_store_state(p, ch, f2_lo(x1), f2_lo(x2), f2_hi(x1), f2_hi(x2), f2_lo(y1), f2_lo(y2), f2_hi(y1), f2_hi(y2), phi);
	}
	if(tid == 0) vdl2_trace_end(p.trace_blocks, trace_k);
}

/* ------------------------------------------------------------------------------------------------
 * K1, one stream per channel ("independent streams", every channel thread of the reference streams its own sample
 * buffer: src/demod.c:302-310).  samples = float2[n_pairs][stride] time-major across streams (k0_convert_lanes), so a
 * block of 128 channels reads 1 KB of contiguous bytes per sample: the algorithmic 8 B per channel-sample are real HBM
 * traffic here.  Rows are fetched by TMA bulk copies (one 1 KB cp.async.bulk per sample row) into a double-buffered
 * shared-memory tile of 80 rows per buffer; with one block per SM ~160 KB per SM (24 MB over the GPU) are in flight,
 * above the bandwidth-delay product of HBM.  Arithmetic and NCO table layout as in the packed kernel.
 * ---------------------------------------------------------------------------------------------- */
#define K1L_BLOCK 128
#define K1L_TILE_ROWS 80
#define K1L_SMEM_BYTES (257 * 8 * 16 + 2 * K1L_TILE_ROWS * K1L_BLOCK * 8 + 16)

template<int OS, bool SYM>
__global__ void __launch_bounds__(K1L_BLOCK) k1_mix_iir_decimate_lanes(vdl2_k1_params p) {
	constexpr int TG = K1L_TILE_ROWS / OS;                 /* groups per tile */
	constexpr int LA = 10, MA = 5;
	constexpr int NLUT = 8;
	extern __shared__ __align__(128) unsigned char k1l_smem[];
	float2 *s_tiles = reinterpret_cast<float2 *>(k1l_smem);                                            /* [2][TG*OS][128] */
	float4 *s_lut = reinterpret_cast<float4 *>(k1l_smem + 2 * K1L_TILE_ROWS * K1L_BLOCK * 8);           /* [257][8] */
	uint64_t *s_bar = reinterpret_cast<uint64_t *>(k1l_smem + 2 * K1L_TILE_ROWS * K1L_BLOCK * 8 + 257 * 8 * 16);
	const uint32_t tid = threadIdx.x;
	const uint32_t ch = blockIdx.x * K1L_BLOCK + tid;
	uint32_t chan;
	const bool active = vdl2_slot_channel(ch, p.lanes, p.full_warps, p.n_ch, chan);
	const uint32_t n_pairs = p.ca ? p.ca->n_pairs : p.n_pairs, cnt0 = p.ca ? p.ca->cnt0 : p.cnt0;
	const size_t stride = p.stream_stride;                 /* float2 elements between consecutive samples */
	const float2 *samples = p.samples + (size_t)blockIdx.x * K1L_BLOCK;      /* this block's 128 columns */
	for(uint32_t i = tid; i < 257 * NLUT; i += K1L_BLOCK) s_lut[i] = p.lut[i / NLUT];
	const float4 *lut = s_lut + (tid & (NLUT - 1));
	const uint32_t lane_bytes = (tid & (NLUT - 1)) * 16u;
	if(tid == 0) { mbar_init(&s_bar[0], 1); mbar_init(&s_bar[1], 1); mbar_fence_init(); }
	float xr1 = 0, xr2 = 0, xi1 = 0, xi2 = 0, yr1 = 0, yr2 = 0, yi1 = 0, yi2 = 0;
	uint32_t phi = 0, dphi = 0;
	if(active) k1_load_state(p, ch, xr1, xr2, xi1, xi2, yr1, yr2, yi1, yi2, phi, dphi);
	u64 x1 = f2_pack(xr1, xi1), x2 = f2_pack(xr2, xi2), y1 = f2_pack(yr1, yi1), y2 = f2_pack(yr2, yi2);
	k1_packed_consts c;
	c.ONE = f2_pack(p.one, p.one); c.SGN = f2_pack(p.neg_one, p.one);
	c.A0 = f2_pack(p.a0, p.a0); c.A1 = f2_pack(p.a1, p.a1); c.A2 = f2_pack(p.a2, p.a2);
	c.B1 = f2_pack(p.b1, p.b1); c.B2 = f2_pack(p.b2, p.b2); c.TWO = f2_pack(p.two, p.two);
	c.one = p.one; c.neg_one = p.neg_one;
	/* the last block may reach past the allocated columns when n_chp is not a multiple of 128: clamp the column */
	const uint32_t col = min(tid, (uint32_t)(p.stream_stride - 1 - (size_t)blockIdx.x * K1L_BLOCK));
	__syncthreads();

	uint32_t cnt = cnt0, m = 0, pos = 0;
	const uint32_t head = min(n_pairs, (OS - cnt0 % OS) % OS);
	if(active) {
		for(; pos < head; pos++) {
			u64 y0 = k1_packed_step(samples[(size_t)pos * stride + col], lut[((phi >> 16) & 0xFFu) * NLUT], phi, dphi, x1, x2, y1, y2, c);
			if(++cnt == OS) { cnt = 0; p.dec[(size_t)m * p.n_chp + ch] = make_float2(f2_lo(y0), f2_hi(y0)); m++; }
		}
	}
	pos = head;
	m = (cnt0 + head) / OS;
	cnt = (cnt0 + head) % OS;
	u64 P1 = f2_mul(c.A0, x1), P2 = f2_mul(c.A0, x2);
	const uint32_t n_groups = (n_pairs - pos) / OS;
	const uint32_t n_tiles = (n_groups + TG - 1) / TG;
	/* bytes of one row that exist in the sample plane for this block (a full 1 KB except in a ragged last block) */
	const uint32_t row_bytes = (uint32_t)min((size_t)K1L_BLOCK, stride - (size_t)blockIdx.x * K1L_BLOCK) * 8u;
	/* thread 0 arms the barrier with the tile's byte count (`arm`, before a block barrier), then threads 0..rows-1 request
	 * one row each (`request`, after it) */
	auto arm = [&](uint32_t t, uint32_t buf) {
		const uint32_t rows = min((uint32_t)TG, n_groups - t * TG) * OS;
		if(tid == 0)
			asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(&s_bar[buf])), "r"(rows * row_bytes) : "memory");
	};
	auto request = [&](uint32_t t, uint32_t buf) {
		const uint32_t rows = min((uint32_t)TG, n_groups - t * TG) * OS;
		const float2 *src = samples + (size_t)(head + (size_t)t * TG * OS) * stride;
		for(uint32_t r = tid; r < rows; r += K1L_BLOCK)
			asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
					:: "r"(smem_u32(&s_tiles[((size_t)buf * TG * OS + r) * K1L_BLOCK])), "l"(src + (size_t)r * stride), "r"(row_bytes), "r"(smem_u32(&s_bar[buf])) : "memory");
	};
	for(uint32_t t = 0; t < 2 && t < n_tiles; t++) arm(t, t);
	__syncthreads();
	for(uint32_t t = 0; t < 2 && t < n_tiles; t++) request(t, t);
	for(uint32_t g0 = 0, tile = 0; g0 < n_groups; g0 += TG, tile++) {
		const uint32_t ng = min((uint32_t)TG, n_groups - g0);
		const float2 *s_tile = s_tiles + (size_t)(tile & 1u) * TG * OS * K1L_BLOCK + tid;
		mbar_wait(&s_bar[tile & 1u], (tile >> 1) & 1u);
		if(active) {
			for(uint32_t g = 0; g < ng; g++) {
				const float2 *sp = &s_tile[g * OS * K1L_BLOCK];
				u64 y0 = 0;
				float2 S[OS];
				float4 E[OS];
				float FR[OS];
				u64 X0[OS];
#pragma unroll
				for(int k = -LA; k < OS; k++) {
					const int kl = k + LA, km = k + MA;
					if(kl < OS) {
						const uint32_t ph = phi + (uint32_t)kl * dphi;
						E[kl] = k1_lut_entry<NLUT>(s_lut, ph, lane_bytes);
						FR[kl] = (float)(ph & 0xFFFFu);
						S[kl] = sp[kl * K1L_BLOCK];
					}
					if(km >= 0 && km < OS) {
						const u64 CS = f2_fma(f2_mul(f2_pack(E[km].z, E[km].w), f2_pack(FR[km], FR[km])), c.ONE, f2_pack(E[km].x, E[km].y));
						X0[km] = k1_mix(S[km], CS, c);
					}
					if(k >= 0) {
						const u64 x0 = X0[k];
						u64 r;
						if(SYM) {
							const u64 P0 = f2_mul(c.A0, x0);
							r = f2_fma(P0, c.ONE, f2_fma(P1, c.TWO, P2));
							P2 = P1; P1 = P0;
						} else {
							const u64 t = f2_fma(f2_mul(c.A1, x1), c.ONE, f2_mul(c.A2, x2));
							r = f2_fma(f2_mul(c.A0, x0), c.ONE, t);
						}
						const u64 u = f2_fma(f2_mul(c.B1, y1), c.ONE, f2_mul(c.B2, y2));
						y0 = f2_fma(r, c.ONE, u);
						x2 = x1; x1 = x0; y2 = y1; y1 = y0;
					}
				}
				phi += (uint32_t)OS * dphi;
				p.dec[(size_t)(m + g) * p.n_chp + ch] = make_float2(f2_lo(y0), f2_hi(y0));
			}
		}
		m += ng;
		pos += ng * OS;
		if(tile + 2 < n_tiles) arm(tile + 2, tile & 1u);           /* arming does not touch the tile's data */
		__syncthreads();                                           /* every warp is done with this buffer, the barrier is armed */
		if(tile + 2 < n_tiles) request(tile + 2, tile & 1u);
	}
	if(active) {
		for(; pos < n_pairs; pos++) {
			u64 y0 = k1_packed_step(samples[(size_t)pos * stride + col], lut[((phi >> 16) & 0xFFu) * NLUT], phi, dphi, x1, x2, y1, y2, c);
			if(++cnt == OS) { cnt = 0; p.dec[(size_t)m * p.n_chp + ch] = make_float2(f2_lo(y0), f2_hi(y0)); m++; }
		}
		k1_store_state(p, ch, f2_lo(x1), f2_lo(x2), f2_hi(x1), f2_hi(x2), f2_lo(y1), f2_lo(y2), f2_hi(y1), f2_hi(y2), phi);
	}
}

/* ------------------------------------------------------------------------------------------------
 * K1, receiver farm (vdl2gpu_create_streams): many raw IQ streams, each with its own centre frequency and any number of
 * channels, the channels stream-major in the slots.  A 128-slot block reads only the streams its channels belong to (the
 * host lists them per block: vdl2_k1_farm.list, .col).  Per tile of R = groups x OS rows, thread j of the block fetches
 * listed stream j's raw bytes (cu8 or cs16, straight from the caller's buffer) with one cp.async.bulk into a double-
 * buffered raw tile, arriving on the tile's mbarrier with its own byte count.  The block then converts the tile once per
 * stream-sample (vdl2_iq_u8 / vdl2_iq_s16, the arithmetic of K0) into a float2 tile [R][row], and lane `slot` reads
 * column col[slot] of each row: the lanes of a warp hold channels of one or a few neighbouring streams, so a row read is
 * a broadcast or a single wavefront.  No K0 launch and no float sample plane.  The filter arithmetic and the eight-copy
 * NCO table are those of the lanes kernel; head and tail samples (outside whole tiles) are converted per lane from the
 * raw bytes.
 *
 * A stream's segment of tile t starts at s * n_pairs * bpp + (head + t R) * bpp, not 16-byte aligned in general (the
 * caller chooses len and the buffer): the copy fetches from the 16-byte boundary at or below it, rounds the size up to
 * 16 bytes and the conversion skips the `off` leading bytes.  The extra bytes lie in 16-byte granules that also hold
 * bytes of the segment, so they are always mapped.
 *
 * Shared memory (dynamic, k1f_layout): NCO table 257 x 8 x 16 B = 32,896 B; float tile R x row x 8 B with row = the
 * longest list of any block, made odd so that the conversion's column writes (32 rows of one stream) avoid bank
 * conflicts; raw tiles 2 x n x W with W = roundup16(15 + R x bpp); two mbarriers; the block's list (4 B) and window
 * offsets (2 x 1 B) per stream.  The host takes the longest tile (at most 640 samples, like the packed kernel) that
 * keeps the total within K1F_SMEM_MAX = 90 KB, so that one farm block fits beside one K2 block (120,848 B) in the
 * 228 KB of an SM, as the packed K1 does.  Worst case, 128 streams in a block, cs16: at OS 10 and 20 R = 20 ->
 * 32,896 + 20 x 129 x 8 + 2 x 128 x 96 + 16 + 768 = 78,896 B; at OS 13 R = 13 -> 32,896 + 13,424 (13 x 129 x 8 rounded to
 * 16) + 2 x 128 x 80 + 16 + 768 = 67,584 B (R = 26 would need 93,280 B).
 * ---------------------------------------------------------------------------------------------- */
#define K1F_SMEM_MAX (90 * 1024)
#define K1F_LUT_BYTES (257 * 8 * 16)
#define K1F_MAX_TILE 640

struct k1f_layout {
	uint32_t row, win, ft, raw, bar, list, off, total;       /* float2 per tile row, bytes per raw window, byte offsets */
	__host__ __device__ k1f_layout(uint32_t rows, uint32_t max_list, uint32_t bpp) {
		row = max_list | 1u;
		win = (15u + rows * bpp + 15u) & ~15u;
		ft = K1F_LUT_BYTES;
		raw = ft + ((rows * row * 8u + 15u) & ~15u);
		bar = raw + 2u * max_list * win;
		list = bar + 16u;
		off = list + 4u * max_list;
		total = off + 2u * max_list;
	}
};

template<int OS, bool SYM>
__global__ void __launch_bounds__(K1F_BLOCK) k1_mix_iir_decimate_farm(vdl2_k1_params p, vdl2_k1_farm f) {
	constexpr int LA = 10, MA = 5;
	constexpr int NLUT = 8;
	extern __shared__ __align__(128) unsigned char k1f_smem[];
	const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31u;
	const int trace_k = tid == 0 ? vdl2_trace_begin(p.trace_blocks, 1) : -1;
	const uint32_t ch = blockIdx.x * K1F_BLOCK + tid;
	uint32_t chan;
	const bool active = vdl2_slot_channel(ch, p.lanes, p.full_warps, p.n_ch, chan);
	const uint32_t n_pairs = p.ca ? p.ca->n_pairs : p.n_pairs, cnt0 = p.ca ? p.ca->cnt0 : p.cnt0;
	const uint8_t *raw = static_cast<const uint8_t *>(p.ca ? p.ca->raw : f.raw);
	const bool s16 = f.fmt == 1u;
	const uint32_t bpp = s16 ? 4u : 2u;
	const size_t stride = (size_t)n_pairs * bpp;                  /* bytes between consecutive streams */
	const uint32_t *blist = f.list + (size_t)blockIdx.x * (1u + K1F_BLOCK);
	const uint32_t n_list = blist[0], G = f.groups, R = G * OS;
	const k1f_layout lay(R, f.max_list, bpp);
	float4 *s_lut = reinterpret_cast<float4 *>(k1f_smem);
	float2 *s_ft = reinterpret_cast<float2 *>(k1f_smem + lay.ft);
	uint8_t *s_raw = k1f_smem + lay.raw;
	uint64_t *s_bar = reinterpret_cast<uint64_t *>(k1f_smem + lay.bar);
	uint32_t *s_list = reinterpret_cast<uint32_t *>(k1f_smem + lay.list);
	uint8_t *s_off = k1f_smem + lay.off;                          /* [2][max_list]: where the segment starts in its window */
	for(uint32_t i = tid; i < 257 * NLUT; i += K1F_BLOCK) s_lut[i] = p.lut[i / NLUT];
	const float4 *lut = s_lut + (tid & (NLUT - 1));
	const uint32_t lane_bytes = (tid & (NLUT - 1)) * 16u;
	if(tid < n_list) s_list[tid] = blist[1 + tid];
	if(tid == 0 && n_list) { mbar_init(&s_bar[0], n_list); mbar_init(&s_bar[1], n_list); mbar_fence_init(); }
	float xr1 = 0, xr2 = 0, xi1 = 0, xi2 = 0, yr1 = 0, yr2 = 0, yi1 = 0, yi2 = 0;
	uint32_t phi = 0, dphi = 0;
	if(active) k1_load_state(p, ch, xr1, xr2, xi1, xi2, yr1, yr2, yi1, yi2, phi, dphi);
	u64 x1 = f2_pack(xr1, xi1), x2 = f2_pack(xr2, xi2), y1 = f2_pack(yr1, yi1), y2 = f2_pack(yr2, yi2);
	k1_packed_consts c;
	c.ONE = f2_pack(p.one, p.one); c.SGN = f2_pack(p.neg_one, p.one);
	c.A0 = f2_pack(p.a0, p.a0); c.A1 = f2_pack(p.a1, p.a1); c.A2 = f2_pack(p.a2, p.a2);
	c.B1 = f2_pack(p.b1, p.b1); c.B2 = f2_pack(p.b2, p.b2); c.TWO = f2_pack(p.two, p.two);
	c.one = p.one; c.neg_one = p.neg_one;
	const uint32_t col = active ? f.col[ch] : 0u;
	__syncthreads();
	if(n_list == 0) { if(tid == 0) vdl2_trace_end(p.trace_blocks, trace_k); return; }      /* no channel in this block */
	const uint8_t *mine = raw + (size_t)s_list[col] * stride;     /* this lane's stream (head and tail samples) */
	auto sample_at = [&](uint32_t i) -> float2 {
		const uint8_t *b = mine + (size_t)i * bpp;
		return s16 ? vdl2_iq_s16(*reinterpret_cast<const short2 *>(b)) : vdl2_iq_u8(*reinterpret_cast<const uchar2 *>(b), f.levels);
	};

	uint32_t cnt = cnt0, m = 0, pos = 0;
	const uint32_t head = min(n_pairs, (OS - cnt0 % OS) % OS);
	if(active) {
		for(; pos < head; pos++) {
			u64 y0 = k1_packed_step(sample_at(pos), lut[((phi >> 16) & 0xFFu) * NLUT], phi, dphi, x1, x2, y1, y2, c);
			if(++cnt == OS) { cnt = 0; p.dec[(size_t)m * p.n_chp + ch] = make_float2(f2_lo(y0), f2_hi(y0)); m++; }
		}
	}
	pos = head;
	m = (cnt0 + head) / OS;
	cnt = (cnt0 + head) % OS;
	u64 P1 = f2_mul(c.A0, x1), P2 = f2_mul(c.A0, x2);
	const uint32_t n_groups = (n_pairs - pos) / OS;
	const uint32_t n_tiles = (n_groups + G - 1) / G;
	/* thread j < n_list: stream j's segment of tile t into raw buffer `buf`, one bulk copy, one arrival on the buffer's barrier */
	auto request = [&](uint32_t t, uint32_t buf) {
		const uint32_t rows = min(G, n_groups - t * G) * OS;
		const uint8_t *src = raw + (size_t)s_list[tid] * stride + (size_t)(head + t * R) * bpp;
		const uint32_t off = (uint32_t)(reinterpret_cast<uintptr_t>(src) & 15u);
		s_off[buf * f.max_list + tid] = (uint8_t)off;
		tma_load_tile(s_raw + (size_t)(buf * f.max_list + tid) * lay.win, src - off, (off + rows * bpp + 15u) & ~15u, &s_bar[buf]);
	};
	if(tid < n_list)
		for(uint32_t t = 0; t < 2 && t < n_tiles; t++) request(t, t);
	for(uint32_t g0 = 0, tile = 0; g0 < n_groups; g0 += G, tile++) {
		const uint32_t ng = min(G, n_groups - g0), rows = ng * OS, buf = tile & 1u;
		mbar_wait(&s_bar[buf], (tile >> 1) & 1u);
		/* conversion, once per stream-sample: warp w takes streams w, w + 4, ..., its lanes consecutive rows */
		for(uint32_t j = warp; j < n_list; j += K1F_BLOCK / 32) {
			const uint8_t *w = s_raw + (size_t)(buf * f.max_list + j) * lay.win + s_off[buf * f.max_list + j];
			for(uint32_t r = lane; r < rows; r += 32)
				s_ft[r * lay.row + j] = s16 ? vdl2_iq_s16(*reinterpret_cast<const short2 *>(w + r * 4u))
				                            : vdl2_iq_u8(*reinterpret_cast<const uchar2 *>(w + r * 2u), f.levels);
		}
		__syncthreads();                                           /* the float tile is complete, raw buffer `buf` is free */
		if(tid < n_list && tile + 2 < n_tiles) request(tile + 2, buf);
		if(active) {
			for(uint32_t g = 0; g < ng; g++) {
				const float2 *sp = s_ft + (size_t)g * OS * lay.row + col;
				u64 y0 = 0;
				float2 S[OS];
				float4 E[OS];
				float FR[OS];
				u64 X0[OS];
#pragma unroll
				for(int k = -LA; k < OS; k++) {
					const int kl = k + LA, km = k + MA;
					if(kl < OS) {
						const uint32_t ph = phi + (uint32_t)kl * dphi;
						E[kl] = k1_lut_entry<NLUT>(s_lut, ph, lane_bytes);
						FR[kl] = (float)(ph & 0xFFFFu);
						S[kl] = sp[kl * lay.row];
					}
					if(km >= 0 && km < OS) {
						const u64 CS = f2_fma(f2_mul(f2_pack(E[km].z, E[km].w), f2_pack(FR[km], FR[km])), c.ONE, f2_pack(E[km].x, E[km].y));
						X0[km] = k1_mix(S[km], CS, c);
					}
					if(k >= 0) {
						const u64 x0 = X0[k];
						u64 r;
						if(SYM) {
							const u64 P0 = f2_mul(c.A0, x0);
							r = f2_fma(P0, c.ONE, f2_fma(P1, c.TWO, P2));
							P2 = P1; P1 = P0;
						} else {
							const u64 t = f2_fma(f2_mul(c.A1, x1), c.ONE, f2_mul(c.A2, x2));
							r = f2_fma(f2_mul(c.A0, x0), c.ONE, t);
						}
						const u64 u = f2_fma(f2_mul(c.B1, y1), c.ONE, f2_mul(c.B2, y2));
						y0 = f2_fma(r, c.ONE, u);
						x2 = x1; x1 = x0; y2 = y1; y1 = y0;
					}
				}
				phi += (uint32_t)OS * dphi;
				p.dec[(size_t)(m + g) * p.n_chp + ch] = make_float2(f2_lo(y0), f2_hi(y0));
			}
		}
		m += ng;
		pos += rows;
		__syncthreads();                                           /* every warp is done with the float tile */
	}
	if(active) {
		for(; pos < n_pairs; pos++) {
			u64 y0 = k1_packed_step(sample_at(pos), lut[((phi >> 16) & 0xFFu) * NLUT], phi, dphi, x1, x2, y1, y2, c);
			if(++cnt == OS) { cnt = 0; p.dec[(size_t)m * p.n_chp + ch] = make_float2(f2_lo(y0), f2_hi(y0)); m++; }
		}
		k1_store_state(p, ch, f2_lo(x1), f2_lo(x2), f2_hi(x1), f2_hi(x2), f2_lo(y1), f2_lo(y2), f2_hi(y1), f2_hi(y2), phi);
	}
	if(tid == 0) vdl2_trace_end(p.trace_blocks, trace_k);
}

/* ------------------------------------------------------------------------------------------------
 * K2: one thread per channel walks the chunk's decimated samples through the demodulator state
 * machine (vdl2_demod_step).  The 160-deep phase ring lives in shared memory, one column per thread
 * (bank = lane, conflict-free whatever the per-channel ring position).
 * ---------------------------------------------------------------------------------------------- */
#define K2_PREFETCH 8

/* K2a: phase and magnitude of every decimated sample of the chunk (src/demod.c:232,238,256), one thread per
 * (time, channel) element: the double-precision atan2/sqrt run at full occupancy here instead of inside the
 * sequential per-channel walk of K2.
 * FAST: the phase comes from vdl2_phase_fast (vdl2_fastmath.cuh: 9 break points, one division, degree-5 polynomial,
 * ~22 FP64 operations) whose float result is the correctly rounded fl32(atan2), the magnitude from vdl2_mag_fast
 * (exact sum of squares, Newton square root); only when one of them reports that its double lies within 2^-44 of a
 * float rounding boundary, or for zero / non-finite / extreme inputs (about one sample in 3e5), the libdevice
 * routine / the IEEE square root decide, as they do for every sample when FAST is off. */

template<bool FAST>
__global__ void __launch_bounds__(256) k2a_phase_mag(const float2 *__restrict__ dec, float *__restrict__ phase,
		float *__restrict__ mag, uint32_t n_elems_p, uint32_t n_chp, uint32_t lanes, const vdl2_chunk_args *__restrict__ ca) {
	__shared__ double s_atan[VDL2_ATAN_TABLE_DOUBLES];
	if(FAST) {
		/* the break-point table is indexed per lane: shared memory (a __constant__ look-up with divergent indices serialises) */
		if(threadIdx.x < VDL2_ATAN_TABLE_DOUBLES) s_atan[threadIdx.x] = c_atan_tab[threadIdx.x];
		__syncthreads();
	}
	const uint32_t n_elems = ca ? ca->n_dec * n_chp : n_elems_p;
	uint32_t i = blockIdx.x * 256u + threadIdx.x;
	if(i >= n_elems || (i & 31u) >= lanes) return;            /* n_chp is a multiple of 32: i & 31 is the lane of the slot (a warp
	                                                            * with lanes - 1 channels computes one idle element: harmless) */
	const float2 d = dec[i];
	float ph, mg;
	if(FAST) {
		int slow_p, slow_m;
		ph = vdl2_phase_fast(d.x, d.y, s_atan, &slow_p);
		mg = vdl2_mag_fast(d.x, d.y, &slow_m);
		if(slow_p) ph = vdl2_phase_of(d.x, d.y);
		if(slow_m) mg = vdl2_mag_of(d.x, d.y);
	} else {
		ph = vdl2_phase_of(d.x, d.y);
		mg = vdl2_mag_of(d.x, d.y);
	}
	phase[i] = ph;
	mag[i] = mg;
}

/* K2a, resident form used by the streaming pipeline: one 128-thread block per SM-sized group of slots, laid out like K1's and
 * K2's blocks (warp w owns slots 32 w .. 32 w + 31), so that the three kernels of three consecutive chunks sit side by
 * side on every SM: K1 of chunk c+2, K2a of chunk c+1, K2 of chunk c.  Each thread walks its channel's decimated samples
 * four at a time (four independent evaluations in flight).  Before that it copies the previous plane's last 160 phase rows
 * into this plane's history rows (the planes alternate between chunks; with n_dec < 160 the source range still lies inside
 * the previous plane, history rows included, so short chunks need no special case). */
template<bool FAST>
__global__ void __launch_bounds__(128, 8) k2a_phase_mag_warps(vdl2_k2a_params p) {      /* <= 64 registers: 32 warps per SM */
	__shared__ double s_atan[VDL2_ATAN_TABLE_DOUBLES];
	if(FAST) {
		if(threadIdx.x < VDL2_ATAN_TABLE_DOUBLES) s_atan[threadIdx.x] = c_atan_tab[threadIdx.x];
		__syncthreads();
	}
	const uint32_t nblk = (p.n_chp + 127u) / 128u, slice = blockIdx.x / nblk;
	const uint32_t slot = (blockIdx.x % nblk) * 128u + threadIdx.x;
	uint32_t chan;
	if(!vdl2_slot_channel(slot, p.lanes, p.full_warps, p.n_ch, chan)) return;
	const uint32_t n_all = p.ca ? p.ca->n_dec : p.n_dec, prev_n_dec = p.ca ? p.ca->prev_n_dec : p.prev_n_dec;
	/* this block's time slice [t, n_dec) of the chunk, boundaries on multiples of 4 samples */
	const uint32_t per = ((n_all + p.split - 1u) / p.split + 3u) & ~3u;
	const uint32_t n_dec = min(n_all, (slice + 1u) * per);
	const size_t s = p.n_chp;
	if(slice == 0) {
		const float *src = p.phase_prev + (size_t)prev_n_dec * s + slot;
		float *dst = p.phase + slot;
#pragma unroll 8
		for(uint32_t i = 0; i < VDL2_SYNC_BUFLEN; i++) dst[(size_t)i * s] = src[(size_t)i * s];
	}
	const float2 *dec = p.dec + slot;
	float *ph = p.phase + (size_t)VDL2_SYNC_BUFLEN * s + slot, *mg = p.mag + slot;
	uint32_t t = min(n_all, slice * per);
	const bool want_mag = p.mag != nullptr;
	/* four samples per step; the next four are requested before the current four are evaluated, so that the loads'
	 * latency hides behind ~400 instructions of arithmetic (the kernel was long-scoreboard bound without it).  FAST: the
	 * straight-line form of the fast atan2 lets the four FP64 chains of a step interleave. */
	float2 nx[4];
	if(t + 4 <= n_dec) {
#pragma unroll
		for(int k = 0; k < 4; k++) nx[k] = dec[(size_t)(t + k) * s];
	}
	for(; t + 4 <= n_dec; t += 4) {
		float2 d[4];
		float a[4], m[4];
		int sp[4], sm[4];
#pragma unroll
		for(int k = 0; k < 4; k++) d[k] = nx[k];
		if(t + 8 <= n_dec) {
#pragma unroll
			for(int k = 0; k < 4; k++) nx[k] = dec[(size_t)(t + 4 + k) * s];
		}
#pragma unroll
		for(int k = 0; k < 4; k++) {
			sm[k] = 1; m[k] = 0.f;
			if(FAST) { a[k] = vdl2_phase_fast_nb(d[k].x, d[k].y, s_atan, &sp[k]); if(want_mag) m[k] = vdl2_mag_fast(d[k].x, d[k].y, &sm[k]); }
			else { sp[k] = 1; a[k] = 0.f; }
		}
#pragma unroll
		for(int k = 0; k < 4; k++) {
			if(VDL2_UNLIKELY(sp[k])) a[k] = vdl2_phase_of(d[k].x, d[k].y);
			ph[(size_t)(t + k) * s] = a[k];
			if(want_mag) {
				if(sm[k]) m[k] = vdl2_mag_of(d[k].x, d[k].y);
				mg[(size_t)(t + k) * s] = m[k];
			}
		}
	}
	for(; t < n_dec; t++) {
		const float2 d = dec[(size_t)t * s];
		ph[(size_t)t * s] = vdl2_phase_of(d.x, d.y);
		if(p.mag != nullptr) mg[(size_t)t * s] = vdl2_mag_of(d.x, d.y);
	}
}

/* carry the last 160 phase rows over to the front of the plane for the next chunk: rows [n_dec, n_dec+160) -> [0, 160) */
__global__ void __launch_bounds__(256) k_copy_rows(const float *__restrict__ src, float *__restrict__ dst, uint32_t n) {
	uint32_t i = blockIdx.x * 256u + threadIdx.x;
	if(i < n) dst[i] = src[i];
}
/* the same with the row offset taken from the chunk arguments (n_dec >= 160: source and destination do not overlap) */
__global__ void __launch_bounds__(256) k_copy_hist(float *__restrict__ phase, uint32_t n, uint32_t n_chp, uint32_t n_dec_p,
		const vdl2_chunk_args *__restrict__ ca) {
	const uint32_t n_dec = ca ? ca->n_dec : n_dec_p;
	uint32_t i = blockIdx.x * 256u + threadIdx.x;
	if(i < n) phase[i] = phase[(size_t)n_dec * n_chp + i];
}

/* 4-byte asynchronous global->shared copies (LDGSTS): completion is tracked per thread by commit/wait groups, not
 * by the register scoreboards, so a look-ahead built on them cannot alias with its own consumer. */
__device__ __forceinline__ void k2_cp_async4(float *smem_dst, const float *gsrc) {
	const unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
	asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" :: "r"(sa), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void k2_cp_async8(float2 *smem_dst, const float2 *gsrc) {
	const unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
	asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" :: "r"(sa), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void k2_cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void k2_cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

/* MODE: 0 sync attempts from the phase plane, TwoSum unwrap; 1 phase plane, table unwrap (default); 2 phase ring,
 * block inputs loaded one block ahead into registers; 3 phase ring, block inputs staged one block ahead in shared
 * memory by cp.async (VDL2GPU_K2_VARIANT=4); 4 phase ring, ALL block inputs (phase, magnitude, decimated samples)
 * staged one block ahead by cp.async (VDL2GPU_K2_VARIANT=5) */
/* staging floats per thread: mode 4 two buffers of (12 phase + 12 float2 samples), mode 3 two buffers of 16 */
#define K2_STAGE_FLOATS(MODE) ((MODE) == 4 ? 2 * (VDL2_WALK_BLOCK + 2 * VDL2_WALK_BLOCK) : (MODE) == 3 ? 2 * 16 : 0)
#define K2_SMEM_BYTES(BLOCK, MODE) ((VDL2_SYNC_BUFLEN + K2_STAGE_FLOATS(MODE)) * (BLOCK) * 4 + 36 * 4 + VDL2_UNWRAP_STATES * 6 * 4)

template<int BLOCK, bool BLOCKED, int MODE>
__global__ void __launch_bounds__(BLOCK) k2_sync_slice(vdl2_k2_params p) {
	/* dynamic shared memory (K2_SMEM_BYTES): phase ring [160][BLOCK], staging area (modes 3 and 4), constants, unwrap table.
	 * BLOCK = 128: the four warps of a block sit on the four sub-partitions of one SM, one each, exactly like K1's, so
	 * that a K1 block and a K2 block always fit side by side (a 250-register warp takes half a sub-partition's register
	 * file: with one-warp blocks two of them could land on the same sub-partition and lock the other kernel out). */
	extern __shared__ __align__(16) unsigned char k2_smem[];
	float *s_ring = reinterpret_cast<float *>(k2_smem);
	float *s_stage_area = s_ring + VDL2_SYNC_BUFLEN * BLOCK;                     /* K2_STAGE_FLOATS(MODE) * BLOCK floats */
	float *s_consts = s_stage_area + K2_STAGE_FLOATS(MODE) * BLOCK;
	uint32_t *s_unwrap = reinterpret_cast<uint32_t *>(s_consts + 36);
	static_assert(MODE >= 0 && MODE <= 4, "walk mode");
	const uint32_t tid = threadIdx.x;
	const int trace_k = tid == 0 ? vdl2_trace_begin(p.trace_blocks, 2) : -1;
	const uint32_t ch = blockIdx.x * BLOCK + tid;
	if(tid < 16) { s_consts[tid] = p.tables->pr_phase[tid]; s_consts[16 + tid] = p.tables->lr_X[tid]; }
	if(tid == 0) s_consts[32] = p.tables->lr_denom;
	if(MODE) for(uint32_t i = tid; i < VDL2_UNWRAP_STATES * 6; i += BLOCK) s_unwrap[i] = p.tables->unwrap_lut[i];
	__syncthreads();
	uint32_t chan;                                    /* public channel number (events, burst records); ch = slot */
	if(!vdl2_slot_channel(ch, p.lanes, p.full_warps, p.n_ch, chan)) return;
	const uint32_t s = p.n_chp;
	uint32_t *st = p.state;
	vdl2_chan v;
	v.prev_phi = __uint_as_float(st[K2_PREV_PHI * s + ch]); v.prev_dphi = __uint_as_float(st[K2_PREV_DPHI * s + ch]);
	v.dphi = __uint_as_float(st[K2_DPHI * s + ch]); v.pherr0 = __uint_as_float(st[K2_PHERR0 * s + ch]);
	v.pherr1 = __uint_as_float(st[K2_PHERR1 * s + ch]); v.pherr2 = __uint_as_float(st[K2_PHERR2 * s + ch]);
	v.ppm_error = __uint_as_float(st[K2_PPM * s + ch]); v.mag_lp = __uint_as_float(st[K2_MAG_LP * s + ch]);
	v.mag_nf = __uint_as_float(st[K2_MAG_NF * s + ch]); v.frame_pwr = __uint_as_float(st[K2_FRAME_PWR * s + ch]);
	v.ring_pos = (int32_t)st[K2_RING_POS * s + ch]; v.sclk = (int32_t)st[K2_SCLK * s + ch];
	v.nfcnt = (int32_t)st[K2_NFCNT * s + ch]; v.frame_pwr_cnt = (int32_t)st[K2_FRAME_PWR_CNT * s + ch];
	v.state = st[K2_STATE * s + ch];
	v.acc = (uint64_t)st[K2_ACC_LO * s + ch] | ((uint64_t)st[K2_ACC_HI * s + ch] << 32);
	v.nbits = st[K2_NBITS * s + ch]; v.need_bits = st[K2_NEED_BITS * s + ch];
	v.datalen = st[K2_DATALEN * s + ch]; v.syndrome = st[K2_SYNDROME * s + ch];
	v.slot = (int32_t)st[K2_SLOT * s + ch]; v.burst_seq = st[K2_BURST_SEQ * s + ch];
	v.sync_dec_index = (uint64_t)st[K2_SYNC_LO * s + ch] | ((uint64_t)st[K2_SYNC_HI * s + ch] << 32);
	v.freq = st[K2_FREQ * s + ch];
	v.cnt_sync = st[K2_CNT_SYNC * s + ch]; v.cnt_hdr_good = st[K2_CNT_HDR_GOOD * s + ch];
	v.pure_run = st[K2_PURE_RUN * s + ch];
	float *ring = &s_ring[tid];
#pragma unroll 4
	for(int i = 0; i < VDL2_SYNC_BUFLEN; i++) ring[i * BLOCK] = p.ring[(size_t)i * s + ch];

	vdl2_k2_env env;
	env.pr_phase = s_consts; env.lr_X = s_consts + 16; env.lr_denom = s_consts[32];
	env.max_ppm = p.max_ppm; env.s27 = p.s27; env.unwrap_lut = s_unwrap;
	env.pool = p.pool; env.free_list = p.free_list; env.ready = p.ready; env.ctl = p.ctl;
	env.events = reinterpret_cast<vdl2_event_rec *>(p.events); env.event_cap = p.event_cap; env.trace = p.trace;

	const float2 *dec = p.dec + ch;
	const float *phs = p.phase + (size_t)VDL2_SYNC_BUFLEN * s + ch;      /* row 0 of phs = first sample of this chunk */
	const float *mgs = p.mag + ch;
	const uint32_t n_dec = p.ca ? p.ca->n_dec : p.n_dec;
	const uint64_t dec_base = p.ca ? p.ca->dec_base : p.dec_base;
	uint32_t m = 0;
	if(BLOCKED) {
		if(MODE == 4) {
			/* Everything a block of 12 samples can need - its 12 phases and 12 decimated samples (the magnitudes are computed
			 * from those) - is staged one block ahead in shared memory by cp.async (24 LDGSTS per lane and block): neither the searching path nor the
			 * symbol slicing of a channel that is inside a burst ever waits for global memory, whatever mix of states the 32
			 * channels of the warp are in. */
			float (*s_st)[VDL2_WALK_BLOCK][BLOCK] = reinterpret_cast<float (*)[VDL2_WALK_BLOCK][BLOCK]>(s_stage_area);   /* [2][12]: phases */
			float2 (*s_sd)[VDL2_WALK_BLOCK][BLOCK] = reinterpret_cast<float2 (*)[VDL2_WALK_BLOCK][BLOCK]>(s_stage_area + 2 * VDL2_WALK_BLOCK * BLOCK);
			auto stage = [&](uint32_t buf, size_t o) {
#pragma unroll
				for(int t = 0; t < VDL2_WALK_BLOCK; t++) {
					k2_cp_async4(&s_st[buf][t][tid], phs + o + (size_t)t * s);
					k2_cp_async8(&s_sd[buf][t][tid], dec + o + (size_t)t * s);
				}
				k2_cp_async_commit();
			};
			uint32_t b = 0;
			if(m + VDL2_WALK_BLOCK <= n_dec) stage(0, 0);
#pragma unroll 1
			for(; m + VDL2_WALK_BLOCK <= n_dec; m += VDL2_WALK_BLOCK, b ^= 1u) {
				k2_cp_async_wait_all();
				if(m + 2 * VDL2_WALK_BLOCK <= n_dec) stage(b ^ 1u, (size_t)(m + VDL2_WALK_BLOCK) * s);
				vdl2_walk_pref pf;
				const int first = vdl2_walk_first(v);
#pragma unroll
				for(int t = 0; t < VDL2_WALK_BLOCK; t++) pf.pw[t] = s_st[b][t][tid];
				/* the four magnitudes the block's sync attempts use (src/demod.c:238) straight from the staged samples: the
				 * Ziv-guarded square root, IEEE square root when it asks for it; no magnitude plane is read in this mode */
				int mg_slow = 0;
#pragma unroll
				for(int j = 0; j < 4; j++) {                 /* four independent FP64 chains, no branch between them */
					const float2 dj = s_sd[b][first + VDL2_SYNC_SKIP * j][tid];
					int slow;
					pf.mg[j] = vdl2_mag_fast_nb(dj.x, dj.y, &slow);
					mg_slow |= slow << j;
				}
				if(VDL2_UNLIKELY(mg_slow)) {
#pragma unroll
					for(int j = 0; j < 4; j++) {
						if((mg_slow >> j) & 1) {
							const float2 dj = s_sd[b][first + VDL2_SYNC_SKIP * j][tid];
							pf.mg[j] = vdl2_mag_of(dj.x, dj.y);
						}
					}
				}
				pf.first = first; pf.valid = 1;
				vdl2_walk_block_ring<true>(v, ring, BLOCK, env, chan, dec_base + m, &s_sd[b][0][tid], &s_st[b][0][tid],
						nullptr, BLOCK, pf, false);
			}
			k2_cp_async_wait_all();
		} else if(MODE == 3) {
			/* stage[buf][k][lane]: k = 0..11 the block's phases, 12..15 the magnitudes at the predicted attempt offsets */
			float *stg = s_stage_area + tid;                         /* [2][16][BLOCK] */
			int first_cur = 0;                                   /* attempt offset the buffer about to be consumed was staged for */
			uint32_t b = 0;
			if(m + VDL2_WALK_BLOCK <= n_dec) {
				const int f0 = vdl2_walk_first(v);
#pragma unroll
				for(int t = 0; t < VDL2_WALK_BLOCK; t++) k2_cp_async4(stg + t * BLOCK, phs + (size_t)t * s);
#pragma unroll
				for(int j = 0; j < 4; j++) k2_cp_async4(stg + (12 + j) * BLOCK, mgs + (size_t)(f0 + VDL2_SYNC_SKIP * j) * s);
				k2_cp_async_commit();
				first_cur = f0;
			}
#pragma unroll 1
			for(; m + VDL2_WALK_BLOCK <= n_dec; m += VDL2_WALK_BLOCK, b ^= 1u) {
				const size_t o = (size_t)m * s;
				k2_cp_async_wait_all();
				vdl2_walk_pref pf;
				const float *cur = stg + b * 16 * BLOCK;
#pragma unroll
				for(int t = 0; t < VDL2_WALK_BLOCK; t++) pf.pw[t] = cur[t * BLOCK];
#pragma unroll
				for(int j = 0; j < 4; j++) pf.mg[j] = cur[(12 + j) * BLOCK];
				pf.first = first_cur; pf.valid = 1;
				if(m + 2 * VDL2_WALK_BLOCK <= n_dec) {             /* next block's inputs into the other buffer */
					const int fn = vdl2_walk_first(v);                /* prediction: the attempt offset repeats every block */
					float *nxt = stg + (b ^ 1u) * 16 * BLOCK;
					const float *ph_n = phs + o + (size_t)VDL2_WALK_BLOCK * s;
					const float *mg_n = mgs + o + (size_t)VDL2_WALK_BLOCK * s;
#pragma unroll
					for(int t = 0; t < VDL2_WALK_BLOCK; t++) k2_cp_async4(nxt + t * BLOCK, ph_n + (size_t)t * s);
#pragma unroll
					for(int j = 0; j < 4; j++) k2_cp_async4(nxt + (12 + j) * BLOCK, mg_n + (size_t)(fn + VDL2_SYNC_SKIP * j) * s);
					first_cur = fn;
				}
				k2_cp_async_commit();
				vdl2_walk_block_ring(v, ring, BLOCK, env, chan, dec_base + m, dec + o, phs + o, mgs + o, s, pf, false);
			}
			k2_cp_async_wait_all();
		} else if(MODE == 2) {
			vdl2_walk_pref pf;
			pf.valid = 0; pf.first = 0;
#pragma unroll
			for(int t = 0; t < VDL2_WALK_BLOCK; t++) pf.pw[t] = 0.f;
#pragma unroll
			for(int j = 0; j < 4; j++) pf.mg[j] = 0.f;
#pragma unroll 1
			for(; m + VDL2_WALK_BLOCK <= n_dec; m += VDL2_WALK_BLOCK) {
				const size_t o = (size_t)m * s;
				vdl2_walk_block_ring(v, ring, BLOCK, env, chan, dec_base + m, dec + o, phs + o, mgs + o, s, pf,
						m + 2 * VDL2_WALK_BLOCK <= n_dec);
			}
		} else {
#pragma unroll 1
			for(; m + VDL2_WALK_BLOCK <= n_dec; m += VDL2_WALK_BLOCK) {
				const size_t o = (size_t)m * s;
				vdl2_walk_block<MODE == 1>(v, ring, BLOCK, env, chan, dec_base + m, dec + o, phs + o, mgs + o, s);
			}
		}
	}
#pragma unroll 1
	for(; m < n_dec; m++) {
		const size_t o = (size_t)m * s;
		const float2 d = __ldg(&dec[o]);
		vdl2_demod_step_pm(v, ring, BLOCK, env, chan, dec_base + m, d.x, d.y, __ldg(&phs[o]), MODE == 4 ? vdl2_mag_of(d.x, d.y) : __ldg(&mgs[o]), false, 0.f, 0.f);
	}

#pragma unroll 4
	for(int i = 0; i < VDL2_SYNC_BUFLEN; i++) p.ring[(size_t)i * s + ch] = ring[i * BLOCK];
	st[K2_PREV_PHI * s + ch] = __float_as_uint(v.prev_phi); st[K2_PREV_DPHI * s + ch] = __float_as_uint(v.prev_dphi);
	st[K2_DPHI * s + ch] = __float_as_uint(v.dphi); st[K2_PHERR0 * s + ch] = __float_as_uint(v.pherr0);
	st[K2_PHERR1 * s + ch] = __float_as_uint(v.pherr1); st[K2_PHERR2 * s + ch] = __float_as_uint(v.pherr2);
	st[K2_PPM * s + ch] = __float_as_uint(v.ppm_error); st[K2_MAG_LP * s + ch] = __float_as_uint(v.mag_lp);
	st[K2_MAG_NF * s + ch] = __float_as_uint(v.mag_nf); st[K2_FRAME_PWR * s + ch] = __float_as_uint(v.frame_pwr);
	st[K2_RING_POS * s + ch] = (uint32_t)v.ring_pos; st[K2_SCLK * s + ch] = (uint32_t)v.sclk;
	st[K2_NFCNT * s + ch] = (uint32_t)v.nfcnt; st[K2_FRAME_PWR_CNT * s + ch] = (uint32_t)v.frame_pwr_cnt;
	st[K2_STATE * s + ch] = v.state;
	st[K2_ACC_LO * s + ch] = (uint32_t)v.acc; st[K2_ACC_HI * s + ch] = (uint32_t)(v.acc >> 32);
	st[K2_NBITS * s + ch] = v.nbits; st[K2_NEED_BITS * s + ch] = v.need_bits;
	st[K2_DATALEN * s + ch] = v.datalen; st[K2_SYNDROME * s + ch] = v.syndrome;
	st[K2_SLOT * s + ch] = (uint32_t)v.slot; st[K2_BURST_SEQ * s + ch] = v.burst_seq;
	st[K2_SYNC_LO * s + ch] = (uint32_t)v.sync_dec_index; st[K2_SYNC_HI * s + ch] = (uint32_t)(v.sync_dec_index >> 32);
	st[K2_CNT_SYNC * s + ch] = v.cnt_sync; st[K2_CNT_HDR_GOOD * s + ch] = v.cnt_hdr_good;
	st[K2_PURE_RUN * s + ch] = v.pure_run;
	if(tid == 0) vdl2_trace_end(p.trace_blocks, trace_k);       /* thread 0's own end: an approximation of the block's */
}

/* ------------------------------------------------------------------------------------------------
 * K3: one block per completed burst (grid-stride over the ready list).
 * ---------------------------------------------------------------------------------------------- */
#define K3_BLOCK 128

/* RS(255,249) errors-and-erasures decode of one block by one warp (src/rs.c:32-49 -> decode_rs.h:71-298): the lanes
 * share the two long loops - syndromes (each lane sums 8 of the 255 symbols, XOR butterfly over the warp) and the Chien
 * search (each lane tests 8 of the 255 positions, roots collected in position order with ballots) - and all evaluate
 * the short Berlekamp-Massey recursion redundantly; lane 0 applies the corrections.  Same return value and same
 * corrected block as the serial vdl2_rs_verify (stepped lane by lane against the oracle in tests/test_hostsim.py). */
__device__ __forceinline__ int k3_rs_block(uint8_t *data, int fec_octets, const uint8_t *gexp, const uint8_t *glog,
		const uint8_t *rootmul, uint32_t lane) {
	if(fec_octets == 0) return 0;
	uint64_t part = vdl2_rs_syndrome_partial(data, lane, gexp, glog, rootmul);
#pragma unroll
	for(int off = 16; off > 0; off >>= 1) part ^= __shfl_xor_sync(0xFFFFFFFFu, part, off);
	if(part == 0) return 0;
	uint8_t S[VDL2_RS_NR], lambda[VDL2_RS_NR + 1];
#pragma unroll
	for(int i = 0; i < VDL2_RS_NR; i++) S[i] = (uint8_t)(part >> (8 * i));
	const int deg = vdl2_rs_locator(S, fec_octets, gexp, glog, lambda);
	const uint32_t mask = vdl2_rs_chien_lane(lambda, deg, lane, gexp, glog);
	int root[VDL2_RS_NR + 1], count = 0;
	for(uint32_t k = 0; k < 8; k++) {
		uint32_t b = __ballot_sync(0xFFFFFFFFu, (mask >> k) & 1u);
		while(b) {
			const int l = __ffs((int)b) - 1;
			b &= b - 1u;
			if(count <= VDL2_RS_NR) root[count < VDL2_RS_NR ? count : VDL2_RS_NR] = l + 1 + 32 * (int)k;
			count++;
		}
	}
	if(deg != count) return -1;
	if(lane == 0) vdl2_rs_forney(data, S, lambda, deg, root, count, gexp, glog);
	__syncwarp();
	return count;
}

__global__ void __launch_bounds__(K3_BLOCK) k3_burst_fec(vdl2_k3_params p) {
	__shared__ vdl2_burst_work w;
	__shared__ uint8_t s_gexp[512];
	__shared__ uint8_t s_glog[256];
	__shared__ uint8_t s_rootmul[6 * 256];
	__shared__ uint16_t s_crctab[256];
	__shared__ uint8_t s_utab[VDL2_UNSTUFF_TABLE_BYTES];
	__shared__ uint16_t s_foff[VDL2_MAX_FRAMES];
	__shared__ uint32_t s_out_off;
	const uint32_t tid = threadIdx.x;
	for(uint32_t i = tid; i < 512; i += K3_BLOCK) s_gexp[i] = p.tables->gf_exp[i];
	for(uint32_t i = tid; i < 256; i += K3_BLOCK) s_glog[i] = p.tables->gf_log[i];
	const uint32_t n_ready = p.ctl->n_ready;
	if(blockIdx.x >= n_ready) return;                         /* nothing for this block: skip the table set-up */
	__syncthreads();
	vdl2_rs_build_rootmul(s_rootmul, s_gexp, s_glog, tid, K3_BLOCK);
	vdl2_crc16_build_table(s_crctab, tid, K3_BLOCK);
	vdl2_unstuff_build_table(s_utab, tid, K3_BLOCK);
	for(uint32_t b = blockIdx.x; b < n_ready; b += gridDim.x) {
		__syncthreads();
		const uint32_t slot_idx = p.ready[b];
		const vdl2_burst_slot *slot = &p.pool[slot_idx];
		if(tid == 0) vdl2_burst_geometry(w, slot->datalen_bits, slot->nbits);
		for(uint32_t i = tid; i < VDL2_MAX_BLOCKS * 256 / 4; i += K3_BLOCK) reinterpret_cast<uint32_t *>(w.tab)[i] = 0;
		__syncthreads();
		if(w.status == VDL2_BURST_OK) {
			vdl2_burst_unpack(w, slot->words, p.tables->lfsr_words, tid, K3_BLOCK);
			__syncthreads();
			for(uint32_t r = tid >> 5; r < w.num_blocks; r += K3_BLOCK / 32) {          /* one warp per RS block */
				const int nfec = (r == w.num_blocks - 1) ? (int)w.last_fec : (VDL2_RS_N - VDL2_RS_K);
				const int ret = k3_rs_block(w.tab[r], nfec, s_gexp, s_glog, s_rootmul, tid & 31u);
				if((tid & 31u) == 0) w.rs_ret[r] = ret;
			}
			__syncthreads();
			if(tid == 0) {
				/* blocks are judged in order; the first failure drops the burst (src/decode.c:305-334) */
				for(uint32_t r = 0; r < w.num_blocks; r++) {
					int nfec = (r == w.num_blocks - 1) ? (int)w.last_fec : (VDL2_RS_N - VDL2_RS_K);
					int ret = w.rs_ret[r];
					if(ret < 0) {
						w.status = VDL2_ERR_FEC_BAD;
						for(uint32_t q = r + 1; q < w.num_blocks; q++) w.rs_ret[q] = -128;
						break;
					}
					if(ret > 0) w.fec_corr += ret - (VDL2_RS_N - VDL2_RS_K - nfec);
				}
				if(w.status == VDL2_BURST_OK) vdl2_burst_unstuff(w, s_utab);
				uint32_t off = 0;
				for(uint32_t k = 0; k < w.n_frames; k++) { s_foff[k] = (uint16_t)off; off += w.flen[k]; }
			}
			__syncthreads();
			for(uint32_t k = tid; k < w.n_frames; k += K3_BLOCK)          /* K4 */
				w.fcrc[k] = vdl2_crc16_tab(&w.frames[s_foff[k]], w.flen[k], s_crctab);
		}
		__syncthreads();
		/* record -> host-mapped output region */
		const uint32_t rec_bytes = (uint32_t)((sizeof(vdl2_burst_record) + 4u * w.n_frames + w.frame_bytes + 15u) & ~15u);
		if(tid == 0) {
			uint32_t off = atomicAdd(&p.ctl->out_used, rec_bytes);
			if(off + rec_bytes > p.out_cap) { atomicAdd(&p.ctl->out_overflows, 1u); off = 0xFFFFFFFFu; }
			else atomicAdd(&p.ctl->out_records, 1u);
			s_out_off = off;
		}
		__syncthreads();
		if(s_out_off != 0xFFFFFFFFu) {
			uint8_t *dst = p.out + sizeof(vdl2_out_header) + s_out_off;
			if(tid == 0) {
				vdl2_burst_record r;
				r.rec_bytes = rec_bytes; r.channel = slot->channel; r.burst_seq = slot->burst_seq; r.status = w.status;
				r.n_frames = w.n_frames; r.datalen_bits = slot->datalen_bits; r.syndrome = slot->syndrome;
				r.num_fec_corrections = w.fec_corr; r.frame_pwr = slot->frame_pwr; r.mag_nf = slot->mag_nf;
				r.ppm_error = slot->ppm_error; r.num_blocks = w.num_blocks; r.sync_lo = slot->sync_lo; r.sync_hi = slot->sync_hi;
				r.freq = slot->freq; r.frame_bytes = w.frame_bytes;
				for(int q = 0; q < 12; q++) r.rs_ret[q] = (int8_t)w.rs_ret[q];
				r.pad = 0;
				const uint32_t *src = reinterpret_cast<const uint32_t *>(&r);
				uint32_t *d32 = reinterpret_cast<uint32_t *>(dst);
				for(uint32_t q = 0; q < sizeof(r) / 4; q++) d32[q] = src[q];
			}
			uint32_t *tab32 = reinterpret_cast<uint32_t *>(dst + sizeof(vdl2_burst_record));
			for(uint32_t k = tid; k < w.n_frames; k += K3_BLOCK) tab32[k] = (uint32_t)w.flen[k] | ((uint32_t)w.fcrc[k] << 16);
			uint32_t *fr32 = tab32 + w.n_frames;
			const uint32_t *fsrc = reinterpret_cast<const uint32_t *>(w.frames);
			for(uint32_t k = tid; k < (w.frame_bytes + 3u) / 4u; k += K3_BLOCK) fr32[k] = fsrc[k];
		}
		/* per-channel counters (names: src/decode.c statsd counters) */
		if(tid == 0) {
			const uint32_t c = slot->channel, s = p.n_chp;
			atomicAdd(&p.counters[VDL2_CNT_BURSTS * s + c], 1u);
			if(w.status != VDL2_BURST_OK) atomicAdd(&p.counters[VDL2_CNT_BURST_ERR * s + c], 1u);
			uint32_t run = 0, ok = 0;
			for(uint32_t r = 0; r < w.num_blocks && r < VDL2_MAX_BLOCKS; r++)
				if(w.rs_ret[r] != -128) { run++; if(w.rs_ret[r] >= 0) ok++; }
			atomicAdd(&p.counters[VDL2_CNT_BLOCKS_PROCESSED * s + c], run);
			atomicAdd(&p.counters[VDL2_CNT_BLOCKS_FEC_OK * s + c], ok);
			atomicAdd(&p.counters[VDL2_CNT_MSG_GOOD * s + c], w.n_frames);
			uint32_t good = 0, bad = 0;
			for(uint32_t k = 0; k < w.n_frames; k++)
				if(w.flen[k] >= 11) { if(w.fcrc[k] == 0xF0B8u) good++; else bad++; }
			atomicAdd(&p.counters[VDL2_CNT_FCS_GOOD * s + c], good);
			atomicAdd(&p.counters[VDL2_CNT_FCS_BAD * s + c], bad);
			/* give the slot back */
			int32_t top = atomicAdd(&p.ctl->free_top, 1);
			p.free_list[top] = (int32_t)slot_idx;
		}
	}
}

/* publish the chunk's totals into the mapped region and re-arm the queues for the next chunk */
__global__ void k_chunk_finish(vdl2_k3_params p) {
	vdl2_out_header *h = reinterpret_cast<vdl2_out_header *>(p.out);
	h->bytes_used = min(p.ctl->out_used, p.out_cap);
	h->n_records = p.ctl->out_records;
	h->pool_overflows = p.ctl->pool_overflows;
	h->out_overflows = p.ctl->out_overflows;
	h->n_events_total = p.ctl->n_events;
	p.ctl->n_ready = 0;
	p.ctl->out_used = 0;
	p.ctl->out_records = 0;
	__threadfence_system();
}

/* stand-alone K4 and RS kernels behind the raw launch stubs */
__global__ void k4_fcs_crc16(const uint8_t *frames, const uint32_t *offsets, const uint32_t *lens, uint32_t n, uint16_t *out) {
	uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if(i < n) out[i] = vdl2_crc16(frames + offsets[i], lens[i]);
}

__global__ void k_rs_verify(uint8_t *blocks, const int32_t *fec_octets, uint32_t n, int32_t *ret, const vdl2_tables *tables) {
	__shared__ uint8_t s_gexp[512];
	__shared__ uint8_t s_glog[256];
	for(uint32_t i = threadIdx.x; i < 512; i += blockDim.x) s_gexp[i] = tables->gf_exp[i];
	for(uint32_t i = threadIdx.x; i < 256; i += blockDim.x) s_glog[i] = tables->gf_log[i];
	__shared__ uint8_t s_rootmul[6 * 256];
	__syncthreads();
	vdl2_rs_build_rootmul(s_rootmul, s_gexp, s_glog, threadIdx.x, blockDim.x);
	__syncthreads();
	uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if(i < n) ret[i] = vdl2_rs_verify(blocks + (size_t)i * VDL2_RS_N, fec_octets[i], s_gexp, s_glog, s_rootmul);
}

/* ------------------------------------------------------------------------------------------------
 * launch stubs
 * ---------------------------------------------------------------------------------------------- */
#define K1_BLOCK 128     /* four warps = the four sub-partitions of an SM share the sample tiles and the 8-copy NCO table */
#define K1_BLOCK1 32     /* one warp per block: independent streams with fewer than 128 channels per stream */
#define K2_BLOCK 128     /* four warps per block, one per sub-partition: see k2_sync_slice */

/* One shared-memory carve-out for every kernel of the chain, so that an SM never has to drain to re-partition
 * its L1/shared memory when kernels of two chunks are resident together (the default two-stream pipeline, see
 * vdl2_host.cu).  Function attributes are per device: vdl2gpu_create calls this after cudaSetDevice, once per device. */
template<typename K> static void vdl2_set_carveout(K kernel, int pct) {
	if(pct >= 0) cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
}

static std::once_flag g_dev_once[64];

extern "C" int vdl2_kernels_init_device(int device) {
	if(device < 0 || device >= 64) return 0;
	std::call_once(g_dev_once[device], [] {
		const char *ev = getenv("VDL2GPU_CARVEOUT");
		const int pct = ev ? atoi(ev) : 100;      /* default: maximum shared memory, the same for every kernel */
		vdl2_set_carveout(k1_mix_iir_decimate_packed<20, K1_BLOCK, 10, true>, pct);
		vdl2_set_carveout(k1_mix_iir_decimate_packed<20, K1_BLOCK, 10, false>, pct);
		vdl2_set_carveout(k1_mix_iir_decimate_packed<20, K1_BLOCK, 0, false>, pct);
		vdl2_set_carveout(k1_mix_iir_decimate_packed<10, K1_BLOCK, 10, true>, pct);
		vdl2_set_carveout(k1_mix_iir_decimate_packed<10, K1_BLOCK, 10, false>, pct);
		vdl2_set_carveout(k1_mix_iir_decimate_packed<10, K1_BLOCK, 0, false>, pct);
		vdl2_set_carveout(k1_mix_iir_decimate_packed<13, K1_BLOCK, 10, true>, pct);
		vdl2_set_carveout(k1_mix_iir_decimate_packed<13, K1_BLOCK, 10, false>, pct);
		vdl2_set_carveout(k1_mix_iir_decimate_packed<20, K1_BLOCK1, 10, true>, pct);
		vdl2_set_carveout(k1_mix_iir_decimate_packed<20, K1_BLOCK1, 10, false>, pct);
		vdl2_set_carveout(k1_mix_iir_decimate_packed<10, K1_BLOCK1, 10, true>, pct);
		vdl2_set_carveout(k1_mix_iir_decimate_packed<10, K1_BLOCK1, 10, false>, pct);
		vdl2_set_carveout(k1_mix_iir_decimate_packed<20, K1_BLOCK, 10, true, true>, pct);
		vdl2_set_carveout(k1_mix_iir_decimate_packed<20, K1_BLOCK, 10, false, true>, pct);
		vdl2_set_carveout(k1_mix_iir_decimate_packed<10, K1_BLOCK, 10, true, true>, pct);
		vdl2_set_carveout(k1_mix_iir_decimate_packed<10, K1_BLOCK, 10, false, true>, pct);
		vdl2_set_carveout(k1_mix_iir_decimate_packed<13, K1_BLOCK, 10, true, true>, pct);
		vdl2_set_carveout(k1_mix_iir_decimate_packed<13, K1_BLOCK, 10, false, true>, pct);
		vdl2_set_carveout(k1_mix_iir_decimate_scalar<K1_BLOCK1>, pct);
		vdl2_set_carveout(k0_convert, pct);
		vdl2_set_carveout(k0_convert_lanes, pct);
		vdl2_set_carveout(k1_mix_iir_decimate_lanes<20, true>, pct);
		vdl2_set_carveout(k1_mix_iir_decimate_lanes<20, false>, pct);
		vdl2_set_carveout(k1_mix_iir_decimate_lanes<10, true>, pct);
		vdl2_set_carveout(k1_mix_iir_decimate_lanes<10, false>, pct);
		cudaFuncSetAttribute(k1_mix_iir_decimate_lanes<20, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, K1L_SMEM_BYTES);
		cudaFuncSetAttribute(k1_mix_iir_decimate_lanes<20, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, K1L_SMEM_BYTES);
		cudaFuncSetAttribute(k1_mix_iir_decimate_lanes<10, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, K1L_SMEM_BYTES);
		cudaFuncSetAttribute(k1_mix_iir_decimate_lanes<10, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, K1L_SMEM_BYTES);
#define K1F_SETUP(OS, SYM) do { vdl2_set_carveout(k1_mix_iir_decimate_farm<OS, SYM>, pct); \
		cudaFuncSetAttribute(k1_mix_iir_decimate_farm<OS, SYM>, cudaFuncAttributeMaxDynamicSharedMemorySize, K1F_SMEM_MAX); } while(0)
		K1F_SETUP(20, true); K1F_SETUP(20, false); K1F_SETUP(10, true); K1F_SETUP(10, false); K1F_SETUP(13, true); K1F_SETUP(13, false);
#undef K1F_SETUP
		vdl2_set_carveout(k2a_phase_mag<true>, pct);
		vdl2_set_carveout(k2a_phase_mag_warps<true>, pct);
		vdl2_set_carveout(k2a_phase_mag_warps<false>, pct);
		vdl2_set_carveout(k2a_phase_mag<false>, pct);
#define K2_SETUP(BLK, BLOCKED, MODE) do { vdl2_set_carveout(k2_sync_slice<BLK, BLOCKED, MODE>, pct); \
		cudaFuncSetAttribute(k2_sync_slice<BLK, BLOCKED, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, K2_SMEM_BYTES(BLK, MODE)); } while(0)
		K2_SETUP(K2_BLOCK, true, 4); K2_SETUP(K2_BLOCK, true, 3); K2_SETUP(K2_BLOCK, true, 2); K2_SETUP(K2_BLOCK, true, 1);
		K2_SETUP(K2_BLOCK, true, 0); K2_SETUP(K2_BLOCK, false, 0);
		K2_SETUP(32, true, 4); K2_SETUP(32, true, 1);
#undef K2_SETUP
		vdl2_set_carveout(k_copy_rows, pct);
		vdl2_set_carveout(k_copy_hist, pct);
		vdl2_set_carveout(k3_burst_fec, pct);
		vdl2_set_carveout(k_chunk_finish, pct);
	});
	return (int)cudaGetLastError();
}

extern "C" int vdl2_launch_k0(const void *raw, uint32_t n_pairs, uint32_t fmt, const float *levels, float *out2, uint32_t n_streams,
		uint32_t raw_stride, uint32_t out_stride, const vdl2_chunk_args *ca, cudaStream_t st) {
	if(n_pairs == 0 || n_streams == 0) return 0;
	k0_convert<<<dim3((n_pairs + 255) / 256, n_streams), 256, 0, st>>>(static_cast<const uint8_t *>(raw), n_pairs, fmt, levels,
			reinterpret_cast<float2 *>(out2), raw_stride, out_stride, ca);
	return (int)cudaGetLastError();
}

extern "C" int vdl2_launch_k0_lanes(const void *raw, uint32_t n_pairs, uint32_t fmt, const float *levels, float *out2, uint32_t n_streams,
		uint32_t raw_stride, uint32_t out_stride, uint32_t lanes, uint32_t full_warps, const vdl2_chunk_args *ca, cudaStream_t st) {
	if(n_pairs == 0 || n_streams == 0) return 0;
	k0_convert_lanes<<<dim3((n_pairs + 31) / 32, (out_stride + 31) / 32), dim3(32, 32), 0, st>>>(static_cast<const uint8_t *>(raw), n_pairs, fmt,
			levels, reinterpret_cast<float2 *>(out2), n_streams, raw_stride, out_stride, lanes, full_warps, ca);
	return (int)cudaGetLastError();
}

template<int OS, int BLOCK>
static void k1_launch_packed(const vdl2_k1_params *p, int variant, bool sym, cudaStream_t st) {
	const uint32_t blocks = (p->n_chp + BLOCK - 1) / BLOCK;
	if(BLOCK == K1_BLOCK && variant != 0 && p->phase != nullptr) {            /* fused phase pass */
		if(sym) k1_mix_iir_decimate_packed<OS, K1_BLOCK, 10, true, true><<<blocks, K1_BLOCK, 0, st>>>(*p);
		else k1_mix_iir_decimate_packed<OS, K1_BLOCK, 10, false, true><<<blocks, K1_BLOCK, 0, st>>>(*p);
		return;
	}
	if(variant == 0 && BLOCK == K1_BLOCK) k1_mix_iir_decimate_packed<OS, K1_BLOCK, 0, false><<<blocks, BLOCK, 0, st>>>(*p);
	else if(sym) k1_mix_iir_decimate_packed<OS, BLOCK, 10, true><<<blocks, BLOCK, 0, st>>>(*p);
	else k1_mix_iir_decimate_packed<OS, BLOCK, 10, false><<<blocks, BLOCK, 0, st>>>(*p);
}

extern "C" int vdl2_k1_fuses_phase(uint32_t oversample, uint32_t ch_per_stream, int force_scalar, int variant) {
	if(force_scalar || variant == 0 || variant == 8 || ch_per_stream == 1) return 0;
	if(ch_per_stream != 0 && ch_per_stream % K1_BLOCK != 0) return 0;
	return oversample == 20 || oversample == 10 || oversample == 13;
}

/* variant: 0 un-pipelined packed kernel, 4 no symmetric-tap specialisation, 8 one warp per block (single NCO table copy),
 * anything else the default (four warps per block, eight table copies) */
extern "C" int vdl2_launch_k1(const vdl2_k1_params *p, int force_scalar, int variant, cudaStream_t st) {
	if(p->n_pairs == 0 || p->n_ch == 0) return 0;
	const bool sym = (p->a1 == 2.0f * p->a0) && (p->a2 == p->a0) && variant != 4;
	if(p->ch_per_stream == 1) {                       /* one stream per channel: samples are float2[n_pairs][stream_stride] */
		const uint32_t blocks = (p->n_chp + K1L_BLOCK - 1) / K1L_BLOCK;
		if(p->oversample == 20) {
			if(sym) k1_mix_iir_decimate_lanes<20, true><<<blocks, K1L_BLOCK, K1L_SMEM_BYTES, st>>>(*p);
			else k1_mix_iir_decimate_lanes<20, false><<<blocks, K1L_BLOCK, K1L_SMEM_BYTES, st>>>(*p);
		} else if(p->oversample == 10) {
			if(sym) k1_mix_iir_decimate_lanes<10, true><<<blocks, K1L_BLOCK, K1L_SMEM_BYTES, st>>>(*p);
			else k1_mix_iir_decimate_lanes<10, false><<<blocks, K1L_BLOCK, K1L_SMEM_BYTES, st>>>(*p);
		} else return (int)cudaErrorInvalidValue;
		return (int)cudaGetLastError();
	}
	/* a 128-channel block must not straddle two streams */
	const bool wide = variant != 8 && (p->ch_per_stream == 0 || p->ch_per_stream % K1_BLOCK == 0);
	if(!force_scalar && p->oversample == 20) {
		if(wide) k1_launch_packed<20, K1_BLOCK>(p, variant, sym, st); else k1_launch_packed<20, K1_BLOCK1>(p, variant, sym, st);
	} else if(!force_scalar && p->oversample == 10) {
		if(wide) k1_launch_packed<10, K1_BLOCK>(p, variant, sym, st); else k1_launch_packed<10, K1_BLOCK1>(p, variant, sym, st);
	} else if(!force_scalar && p->oversample == 13 && variant != 0 && wide) {      /* 1.365 Msps (Mirics, src/mirics.h:23) */
		k1_launch_packed<13, K1_BLOCK>(p, variant, sym, st);
	} else {
		const uint32_t blocks = (p->n_chp + K1_BLOCK1 - 1) / K1_BLOCK1;
		k1_mix_iir_decimate_scalar<K1_BLOCK1><<<blocks, K1_BLOCK1, 0, st>>>(*p);
	}
	return (int)cudaGetLastError();
}

extern "C" int vdl2_k1_farm_layout(uint32_t oversample, uint32_t fmt, uint32_t max_list, vdl2_k1_farm *f) {
	if((oversample != 10 && oversample != 13 && oversample != 20) || fmt > 1u || max_list == 0 || max_list > K1F_BLOCK) return (int)cudaErrorInvalidValue;
	const uint32_t bpp = fmt == 1u ? 4u : 2u;
	for(uint32_t g = K1F_MAX_TILE / oversample; g >= 1; g--) {
		const k1f_layout lay(g * oversample, max_list, bpp);
		if(lay.total <= K1F_SMEM_MAX) { f->groups = g; f->max_list = max_list; f->fmt = fmt; f->smem_bytes = lay.total; return 0; }
	}
	return (int)cudaErrorInvalidValue;
}

extern "C" int vdl2_launch_k1_farm(const vdl2_k1_params *p, const vdl2_k1_farm *f, cudaStream_t st) {
	if(p->n_pairs == 0 || p->n_ch == 0) return 0;
	const bool sym = (p->a1 == 2.0f * p->a0) && (p->a2 == p->a0);
	const uint32_t blocks = (p->n_chp + K1F_BLOCK - 1) / K1F_BLOCK;
#define K1F_GO(OS) do { if(sym) k1_mix_iir_decimate_farm<OS, true><<<blocks, K1F_BLOCK, f->smem_bytes, st>>>(*p, *f); \
		else k1_mix_iir_decimate_farm<OS, false><<<blocks, K1F_BLOCK, f->smem_bytes, st>>>(*p, *f); } while(0)
	if(p->oversample == 20) K1F_GO(20);
	else if(p->oversample == 10) K1F_GO(10);
	else if(p->oversample == 13) K1F_GO(13);
	else return (int)cudaErrorInvalidValue;
#undef K1F_GO
	return (int)cudaGetLastError();
}

extern "C" int vdl2_launch_k2a(const vdl2_k2_params *p, cudaStream_t st) {
	if(p->n_dec == 0 || p->n_ch == 0) return 0;
	const uint32_t n_elems = p->n_dec * p->n_chp;
	const uint32_t hist = VDL2_SYNC_BUFLEN * p->n_chp;
	if(p->k2a_mode) k2a_phase_mag<true><<<(n_elems + 255u) / 256u, 256, 0, st>>>(p->dec, p->phase + hist, p->mag, n_elems, p->n_chp, p->lanes ? p->lanes : 32u, p->ca);
	else k2a_phase_mag<false><<<(n_elems + 255u) / 256u, 256, 0, st>>>(p->dec, p->phase + hist, p->mag, n_elems, p->n_chp, p->lanes ? p->lanes : 32u, p->ca);
	return (int)cudaGetLastError();
}

extern "C" int vdl2_launch_k2a_warps(const vdl2_k2a_params *p, cudaStream_t st) {
	if(p->n_ch == 0) return 0;
	const uint32_t blocks = ((p->n_chp + 127u) / 128u) * (p->split ? p->split : 1u);
	if(p->mode) k2a_phase_mag_warps<true><<<blocks, 128, 0, st>>>(*p);
	else k2a_phase_mag_warps<false><<<blocks, 128, 0, st>>>(*p);
	return (int)cudaGetLastError();
}

/* variant: 0 per-sample walk; 1 blocked, phase plane, TwoSum unwrap; 2 blocked, phase plane, table unwrap; 3 blocked,
 * phase ring, block inputs one block ahead in registers; 4 the same with cp.async staging; anything else (5, the
 * default): phase ring with every block input (phase, magnitude, samples) staged one block ahead by cp.async */
extern "C" int vdl2_launch_k2(const vdl2_k2_params *p, cudaStream_t st) {
	if(p->n_dec == 0 || p->n_ch == 0) return 0;
	uint32_t blocks = (p->n_chp + K2_BLOCK - 1) / K2_BLOCK;
	const uint32_t variant = p->variant & 0xFFu;
	if(p->variant & 0x100u) {                     /* A/B: one warp per block (VDL2GPU_K2_VARIANT = 256 + variant) */
		blocks = (p->n_chp + 31u) / 32u;
		if(variant == 2) k2_sync_slice<32, true, 1><<<blocks, 32, K2_SMEM_BYTES(32, 1), st>>>(*p);
		else k2_sync_slice<32, true, 4><<<blocks, 32, K2_SMEM_BYTES(32, 4), st>>>(*p);
		return (int)cudaGetLastError();
	}
#define K2_GO(BLOCKED, MODE) k2_sync_slice<K2_BLOCK, BLOCKED, MODE><<<blocks, K2_BLOCK, K2_SMEM_BYTES(K2_BLOCK, MODE), st>>>(*p)
	if(variant == 0) K2_GO(false, 0);
	else if(variant == 1) K2_GO(true, 0);
	else if(variant == 2) K2_GO(true, 1);
	else if(variant == 3) K2_GO(true, 2);
	else if(variant == 4) K2_GO(true, 3);
	else K2_GO(true, 4);                       /* default (5, or any unknown value) */
#undef K2_GO
	return (int)cudaGetLastError();
}

/* history for the next chunk: phase rows [n_dec, n_dec+160) -> [0, 160) */
extern "C" int vdl2_launch_copy_hist(const vdl2_k2_params *p, cudaStream_t st) {
	if(p->n_dec == 0 || p->n_ch == 0) return 0;
	const uint32_t hist = VDL2_SYNC_BUFLEN * p->n_chp;
	if(p->n_dec >= VDL2_SYNC_BUFLEN) {
		k_copy_hist<<<(hist + 255u) / 256u, 256, 0, st>>>(p->phase, hist, p->n_chp, p->n_dec, p->ca);
	} else {
		k_copy_rows<<<(hist + 255u) / 256u, 256, 0, st>>>(p->phase + (size_t)p->n_dec * p->n_chp, p->hist_tmp, hist);
		k_copy_rows<<<(hist + 255u) / 256u, 256, 0, st>>>(p->hist_tmp, p->phase, hist);
	}
	return (int)cudaGetLastError();
}

extern "C" int vdl2_launch_k3(const vdl2_k3_params *p, uint32_t grid, cudaStream_t st) {
	k3_burst_fec<<<grid, K3_BLOCK, 0, st>>>(*p);
	int e = (int)cudaGetLastError();
	if(e) return e;
	k_chunk_finish<<<1, 1, 0, st>>>(*p);
	return (int)cudaGetLastError();
}

extern "C" int vdl2_launch_k4(const uint8_t *frames, const uint32_t *offsets, const uint32_t *lens, uint32_t n, uint16_t *out, cudaStream_t st) {
	if(n == 0) return 0;
	k4_fcs_crc16<<<(n + 127) / 128, 128, 0, st>>>(frames, offsets, lens, n, out);
	return (int)cudaGetLastError();
}

extern "C" int vdl2_launch_rs(uint8_t *blocks, const int32_t *fec_octets, uint32_t n, int32_t *ret, const vdl2_tables *tables, cudaStream_t st) {
	if(n == 0) return 0;
	k_rs_verify<<<(n + 63) / 64, 64, 0, st>>>(blocks, fec_octets, n, ret, tables);
	return (int)cudaGetLastError();
}
