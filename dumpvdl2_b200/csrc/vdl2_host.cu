/*
 * vdl2_host.cu — host runtime of libvdl2gpu.so: start-up tables, device-resident channel state, the
 * pinned staging ring, stream-ordered kernel chain per IQ chunk, and harvesting of burst records into
 * avlc_decoder_queue_push-shaped frames.  C-ABI in include/vdl2gpu.h.
 *
 * Host arithmetic for the start-up tables restates the reference's init code read strictly
 * (compiled with -ffp-contract=off, no fast-math); citations are file:line under /root/reference.
 * There is no CPU implementation of the sample path in this library: every data-path entry point
 * needs a CUDA device and fails with VDL2GPU_ENODEV / VDL2GPU_ECUDA otherwise.
 */
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/time.h>
#include <algorithm>
#include <deque>
#include <mutex>
#include <string>
#include <vector>
#include "../../include/vdl2gpu.h"
#include "vdl2_kernels.h"
#include "vdl2_types.h"
#include "vdl2_tables_host.h"

static thread_local char g_last_error[512] = "";

extern "C" void vdl2gpu_set_last_error(const char *msg) {          /* for the other translation units of the library */
	snprintf(g_last_error, sizeof(g_last_error), "%s", msg ? msg : "");
}

static int fail_cuda(cudaError_t e, const char *what, int line) {
	snprintf(g_last_error, sizeof(g_last_error), "%s failed at vdl2_host.cu:%d: %s", what, line, cudaGetErrorString(e));
	return (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) ? VDL2GPU_ENODEV : VDL2GPU_ECUDA;
}
#define CU(call) do { cudaError_t e_ = (call); if(e_ != cudaSuccess) return fail_cuda(e_, #call, __LINE__); } while(0)
#define KL(call) do { int e_ = (call); if(e_ != 0) return fail_cuda((cudaError_t)e_, #call, __LINE__); } while(0)

/* ------------------------------------------------------------------------------------------------
 * context
 * ---------------------------------------------------------------------------------------------- */
/* frames harvested but not yet delivered; their octets live in per-chunk blobs (one copy per chunk) */
struct pending_frame {
	vdl2gpu_frame f;
	uint32_t blob, offset;
};

struct chunk_slot {
	uint8_t *h_raw = nullptr, *d_raw = nullptr;
	uint8_t *h_out = nullptr, *d_out = nullptr;
	cudaEvent_t done = nullptr;
	cudaEvent_t tk[8] = { nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr };   /* front: 0,1,2  mid: 3,6  back: 7,4,5 */
	bool busy = false, timed = false;
	uint64_t seq = 0;
	/* per-chunk arguments (pinned host copy, device copy made by the first node of the front graph) and the three
	 * CUDA graphs of this slot per decimated-sample buffer: front {args copy, K0, K1}, K2a, back {K2, history, K3, finish} */
	vdl2_chunk_args *h_args = nullptr, *d_args = nullptr;
	cudaGraphExec_t g_front[6] = { nullptr }, g_k2a[6] = { nullptr }, g_back[6] = { nullptr };    /* index = chunk number mod 6 (dec buffer, plane) */
	uint32_t graph_pairs[6] = { 0 };
	uint64_t first_pair = 0, dec_base = 0;
	uint32_t n_pairs = 0, n_dec = 0;
	struct timeval arrival = { 0, 0 };
};

struct vdl2gpu_ctx {
	vdl2gpu_config cfg;
	std::vector<uint32_t> freqs;
	int device = 0;
	/* `stream` (front) carries H2D + K0 + K1 of chunk c+1 while `s_back` carries K2a/K2/K3 of chunk c.  Both stages
	 * are latency-bound with one warp per SM sub-partition at 16 k channels, so co-residency raises issue-slot use:
	 * 12.1 -> 8.7 ms per chunk on B200.  This only works because every kernel of the chain requests the SAME
	 * shared-memory carve-out (vdl2_kernels.cu): with per-kernel defaults the SMs drain to re-partition L1/shared
	 * memory and the overlap is a 1.7x slow-down.  VDL2GPU_FLAG_NO_OVERLAP puts everything on one stream. */
	cudaStream_t stream = nullptr, s_mid = nullptr, s_back = nullptr;
	/* three stages, three chunks in flight: K0+K1 of chunk c+2 (front), K2a of chunk c+1 (mid), K2+K3 of chunk c (back).
	 * dec is triple-buffered (written by K1, read by K2a and K2), the phase / magnitude planes alternate (written by K2a,
	 * read by K2; K2a of chunk c takes its 160 history rows from the other plane, i.e. from chunk c-1). */
	cudaEvent_t ev_k1_done[3] = { nullptr, nullptr, nullptr }, ev_back_done[3] = { nullptr, nullptr, nullptr }, ev_k2a_done[2] = { nullptr, nullptr };
	uint64_t chunk_seq = 0;
	cudaEvent_t ev_input_ready = nullptr, ev_input_consumed = nullptr;
	uint32_t n_ch = 0, n_chp = 0, max_pairs = 0, max_dec = 0, n_slots = 0, out_cap = 0, event_cap = 0;
	uint64_t events_dropped = 0;                        /* trace events lost to a full buffer, not yet reported by vdl2gpu_read_events */
	uint32_t lanes = 32, full_warps = 0xFFFFFFFFu;      /* channel slot mapping (see create_impl) */
	int n_sms = 148;
	uint32_t n_streams = 1, ch_per_stream = 0;          /* independent-streams mode: n_streams > 1, channels [s*C, (s+1)*C) on stream s */
	bool lane_streams = false;                          /* C == 1: samples kept time-major across streams, one lane per stream in K1 */
	bool farm = false;                                  /* receiver farm (vdl2gpu_create_streams): any channel count per stream, K1 reads the raw bytes */
	vdl2_k1_farm k1f;                                   /* farm: per-block stream lists (d_farm) and the farm K1's tile shape */
	uint32_t *d_farm = nullptr;
	uint32_t raw_bytes = 0;                             /* size of each slot's raw staging buffers (allocated on the first host submit) */
	int k1_variant = 2, k2_variant = 5, k2a_mode = 1;   /* A/B knobs (VDL2GPU_K1_VARIANT, VDL2GPU_K2_VARIANT, VDL2GPU_K2A), read at create */
	bool use_graphs = true;
	uint32_t k2a_split = 64;                            /* time slices of the K2a grid (VDL2GPU_K2A_SPLIT) */
	int stages = 2;                                     /* 2: K2a runs alone between K1 of chunk c and K1 of chunk c+1 (default, see run_chain);
	                                                     * 3: K2a of chunk c+1 beside K1 of chunk c+2 and K2 of chunk c (VDL2GPU_STAGES=3) */
	bool fuse_phase = false;                            /* VDL2GPU_FUSE_PHASE=1: K1 writes the phase plane itself, no K2a launch (measured slower than the separate pass: DESIGN.md) */
	bool k2a_exclusive = true;                          /* K1 of chunk c+1 waits for K2a of chunk c (VDL2GPU_K2A_EXCLUSIVE=0: let them overlap) */
	uint64_t overflows_reported = 0;
	host_tables tab;
	vdl2_tables *d_tab = nullptr;
	float2 *d_samples = nullptr;
	float2 *d_dec3[3] = { nullptr, nullptr, nullptr };
	float *d_phase2[2] = { nullptr, nullptr }, *d_mag2[2] = { nullptr, nullptr };
	uint32_t *d_k1 = nullptr, *d_k2 = nullptr, *d_counters = nullptr, *d_ready = nullptr;
	float *d_ring = nullptr;
	vdl2_burst_slot *d_pool = nullptr;
	int32_t *d_free = nullptr;
	vdl2_queue_ctl *d_ctl = nullptr;
	void *d_events = nullptr;
	std::vector<chunk_slot> chunks;
	std::deque<uint32_t> inflight;
	uint32_t next_slot = 0;
	uint32_t decim_cnt = 0, last_n_dec = 0;
	uint64_t total_pairs = 0, total_dec = 0;
	uint32_t events_read = 0;
	bool timing = false;
	double k_ms[5] = { 0, 0, 0, 0, 0 };                 /* K0, K1, K2a, K2 (+history copy), K3 (+finish) */
	uint64_t k_launches[5] = { 0, 0, 0, 0, 0 };
	vdl2_block_trace *d_block_trace = nullptr;          /* VDL2GPU_BLOCK_TRACE=1: per-block scheduling records of K1 / K2 */
	uint32_t block_trace_cap = 0;
	uint32_t graph_nominal = 0;                         /* chunk shape (n_pairs) the graphs are kept for */
	cudaEvent_t ev_t0 = nullptr;                        /* origin of the timeline (recorded by vdl2gpu_enable_timing) */
	std::vector<float> timeline;                        /* 8 floats per timed chunk: chunk number, then the 7 stage boundaries in ms since ev_t0 */
	vdl2gpu_stats stats;
	std::vector<pending_frame> pending;
	std::vector<std::vector<uint8_t>> blobs;
	cudaEvent_t ev_drain = nullptr;
};

static uint32_t dphi_for(uint32_t centerfreq, uint32_t freq, uint32_t rate) {      /* src/demod.c:385 */
	return (uint32_t)(int)(((float)centerfreq - (float)freq) / (float)rate * 256.0f * 65536.0f);
}

static void initial_state(const vdl2gpu_config &cfg, const uint32_t *freqs, const uint32_t *centers, uint32_t n_ch, uint32_t n_chp, uint32_t lanes,
		uint32_t full_warps, std::vector<uint32_t> &k1, std::vector<uint32_t> &k2);
/* channel -> slot: the first full_warps warps hold `lanes` channels each, the others lanes - 1 */
static inline uint32_t slot_of(uint32_t ch, uint32_t lanes, uint32_t full_warps) {
	const uint32_t head = full_warps * lanes;
	if(ch < head) return (ch / lanes) * 32u + ch % lanes;
	const uint32_t c = ch - head;
	return (full_warps + c / (lanes - 1u)) * 32u + c % (lanes - 1u);
}

extern "C" int vdl2gpu_abi_version(void) { return VDL2GPU_ABI_VERSION; }

extern "C" int vdl2gpu_device_count(void) {
	int n = 0;
	if(cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
	return n;
}

extern "C" const char *vdl2gpu_last_error(void) { return g_last_error; }

extern "C" const char *vdl2gpu_strerror(int code) {
	switch(code) {
		case VDL2GPU_OK: return "ok";
		case VDL2GPU_EINVAL: return "invalid argument";
		case VDL2GPU_ENODEV: return "no usable CUDA device";
		case VDL2GPU_ECUDA: return "CUDA runtime error";
		case VDL2GPU_ENOMEM: return "out of memory";
		case VDL2GPU_ETOOBIG: return "chunk larger than max_chunk_bytes";
		case VDL2GPU_EOVERFLOW: return "device queue overflow, bursts dropped";
		default: return "unknown error";
	}
}

static int free_ctx(vdl2gpu_ctx *c) {
	if(!c) return VDL2GPU_OK;
	cudaSetDevice(c->device);
	if(c->stream) cudaStreamSynchronize(c->stream);
	if(c->s_mid) cudaStreamSynchronize(c->s_mid);
	if(c->s_back) cudaStreamSynchronize(c->s_back);
	for(auto &s : c->chunks) {
		if(s.h_raw) cudaFreeHost(s.h_raw);
		if(s.d_raw) cudaFree(s.d_raw);
		if(s.h_out) cudaFreeHost(s.h_out);
		if(s.done) cudaEventDestroy(s.done);
		for(auto &e : s.tk) if(e) cudaEventDestroy(e);
		for(int i = 0; i < 6; i++) {
			if(s.g_front[i]) cudaGraphExecDestroy(s.g_front[i]);
			if(s.g_k2a[i]) cudaGraphExecDestroy(s.g_k2a[i]);
			if(s.g_back[i]) cudaGraphExecDestroy(s.g_back[i]);
		}
		if(s.h_args) cudaFreeHost(s.h_args);
		if(s.d_args) cudaFree(s.d_args);
	}
	cudaFree(c->d_tab); cudaFree(c->d_samples);
	for(int i = 0; i < 3; i++) cudaFree(c->d_dec3[i]);
	for(int i = 0; i < 2; i++) { cudaFree(c->d_phase2[i]); cudaFree(c->d_mag2[i]); }
	cudaFree(c->d_k1); cudaFree(c->d_k2);
	cudaFree(c->d_counters); cudaFree(c->d_ready); cudaFree(c->d_ring); cudaFree(c->d_pool); cudaFree(c->d_free);
	cudaFree(c->d_ctl); cudaFree(c->d_events); cudaFree(c->d_block_trace); cudaFree(c->d_farm);
	if(c->ev_input_ready) cudaEventDestroy(c->ev_input_ready);
	if(c->ev_input_consumed) cudaEventDestroy(c->ev_input_consumed);
	if(c->ev_drain) cudaEventDestroy(c->ev_drain);
	if(c->ev_t0) cudaEventDestroy(c->ev_t0);
	for(int i = 0; i < 2; i++) if(c->ev_k2a_done[i]) cudaEventDestroy(c->ev_k2a_done[i]);
	for(int i = 0; i < 3; i++) { if(c->ev_k1_done[i]) cudaEventDestroy(c->ev_k1_done[i]); if(c->ev_back_done[i]) cudaEventDestroy(c->ev_back_done[i]); }
	if(c->s_mid && c->s_mid != c->stream && c->s_mid != c->s_back) cudaStreamDestroy(c->s_mid);
	if(c->s_back && c->s_back != c->stream) cudaStreamDestroy(c->s_back);
	if(c->stream) cudaStreamDestroy(c->stream);
	delete c;
	return VDL2GPU_OK;
}

/* layout: NULL for vdl2gpu_create, the (validated) receiver-farm layout for vdl2gpu_create_streams */
static int create_impl(const vdl2gpu_config *cfg, const vdl2gpu_stream_layout *layout, vdl2gpu_ctx *c) {
	int ndev = 0;
	cudaError_t e = cudaGetDeviceCount(&ndev);
	if(e != cudaSuccess || ndev == 0) {
		cudaGetLastError();
		snprintf(g_last_error, sizeof(g_last_error), "no CUDA device (%s); libvdl2gpu has no CPU fallback",
				e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
		return VDL2GPU_ENODEV;
	}
	if(cfg->device >= 0) { c->device = cfg->device; CU(cudaSetDevice(c->device)); }
	else CU(cudaGetDevice(&c->device));
	cudaDeviceProp prop;
	CU(cudaGetDeviceProperties(&prop, c->device));
	if(prop.major < 10) {
		snprintf(g_last_error, sizeof(g_last_error), "device %d is sm_%d%d; this library carries sm_100a code only", c->device, prop.major, prop.minor);
		return VDL2GPU_ENODEV;
	}
	KL(vdl2_kernels_init_device(c->device));             /* per device: function attributes do not carry over */
	c->cfg = *cfg;
	c->farm = layout != nullptr;
	c->n_streams = c->farm ? layout->n_streams : cfg->n_streams ? cfg->n_streams : 1u;
	c->cfg.n_streams = c->n_streams;
	c->lane_streams = !c->farm && c->n_streams > 1 && c->n_streams == cfg->n_channels;     /* one stream per channel */
	if(c->lane_streams) {
		c->ch_per_stream = 1;
	} else if(!c->farm && c->n_streams > 1) {
		if(cfg->n_channels % c->n_streams != 0 || (cfg->n_channels / c->n_streams) % 32u != 0) {
			snprintf(g_last_error, sizeof(g_last_error), "independent-streams mode needs n_channels = n_streams x C with C = 1 or a multiple of 32 (got %u channels, %u streams)",
					cfg->n_channels, c->n_streams);
			return VDL2GPU_EINVAL;
		}
		c->ch_per_stream = cfg->n_channels / c->n_streams;
	}
	{
		const char *e;
		if((e = getenv("VDL2GPU_K1_VARIANT"))) c->k1_variant = atoi(e);
		if((e = getenv("VDL2GPU_K2_VARIANT"))) c->k2_variant = atoi(e);
		if((e = getenv("VDL2GPU_K2A"))) c->k2a_mode = atoi(e);
		if((e = getenv("VDL2GPU_NO_GRAPH")) && atoi(e)) c->use_graphs = false;
		if((e = getenv("VDL2GPU_BLOCK_TRACE")) && atoi(e)) c->block_trace_cap = 1u << 16;
		if((e = getenv("VDL2GPU_K2A_EXCLUSIVE"))) c->k2a_exclusive = atoi(e) != 0;
		if((e = getenv("VDL2GPU_STAGES")) && atoi(e) == 3) { c->stages = 3; c->k2a_split = 3; }
		if((e = getenv("VDL2GPU_K2A_SPLIT")) && atoi(e) >= 1 && atoi(e) <= 256) c->k2a_split = (uint32_t)atoi(e);
	}
	{
		/* fused phase pass (opt-in): needs the K1 kernel that implements it, the fast (Ziv-guarded) atan2 and a walk that takes its
		 * magnitudes from the samples (no magnitude plane, hence nothing left for K2a to do) */
		const char *e = getenv("VDL2GPU_FUSE_PHASE");
		const int k2v = c->k2_variant & 0xFF;
		c->fuse_phase = (e && atoi(e) != 0) && !c->farm && c->k2a_mode == 1 && !(k2v >= 0 && k2v <= 4) && c->stages == 2
			&& vdl2_k1_fuses_phase(cfg->oversample, c->ch_per_stream, (cfg->flags & VDL2GPU_FLAG_K1_SCALAR) ? 1 : 0, c->k1_variant);
	}
	if(cfg->flags & (VDL2GPU_FLAG_NO_GRAPH | VDL2GPU_FLAG_TRACE)) c->use_graphs = false;
	c->freqs.assign(cfg->freqs, cfg->freqs + cfg->n_channels);
	c->cfg.freqs = c->freqs.data();
	c->n_ch = cfg->n_channels;
	c->n_chp = (c->n_ch + 31u) & ~31u;
	c->n_sms = prop.multiProcessorCount;
	c->lanes = 32; c->full_warps = 0xFFFFFFFFu;
	/* Slot mapping.  K1 and K2 run four-warp blocks, one warp per SM sub-partition, and a chunk's K2 overlaps the next
	 * chunk's K1.  The block scheduler places a new block on the SM with the most free resources: when a grid leaves SMs
	 * empty (128 blocks on 148 SMs at 16384 channels), the OTHER kernel's blocks pile up on those SMs two and three deep
	 * instead of sitting beside the first kernel's blocks, one per SM, and run two to three times slower (measured with
	 * the per-block trace, tools/block_trace.py).  So when the channels fill more than half of the machine's
	 * sub-partitions, they are dealt out evenly over ALL of them: every warp holds floor or ceil of n_ch / (4 x SMs)
	 * channels instead of 32 (27 or 28 at 16384 channels on 148 SMs), each of the two kernels launches exactly one block
	 * per SM, every block lives for the whole kernel, and every SM looks the same to the scheduler. */
	if(c->farm || cfg->n_streams <= 1 || cfg->n_streams == cfg->n_channels) {
		const uint32_t warps_all = 4u * (uint32_t)c->n_sms;
		if(c->n_ch > 16u * warps_all && c->n_ch <= 32u * warps_all) {
			const char *e = getenv("VDL2GPU_BALANCE");
			if(!e || atoi(e)) {
				c->lanes = (c->n_ch + warps_all - 1u) / warps_all;
				c->full_warps = c->n_ch - (c->lanes - 1u) * warps_all;       /* warps with `lanes` channels; the rest have lanes - 1 */
				c->n_chp = warps_all * 32u;
			}
		}
	}
	const uint32_t max_bytes = cfg->max_chunk_bytes ? cfg->max_chunk_bytes : (1u << 20);
	c->cfg.max_chunk_bytes = max_bytes;
	c->max_pairs = max_bytes / (cfg->sample_fmt == VDL2GPU_FMT_S16_LE ? 4u : 2u);
	c->max_dec = c->max_pairs / cfg->oversample + 2;
	if((uint64_t)(c->max_dec + VDL2_SYNC_BUFLEN) * c->n_chp >= (1ull << 32)) {
		snprintf(g_last_error, sizeof(g_last_error), "%u channels x %u decimated samples per chunk exceed the 32-bit element index of the kernels; "
				"use a smaller max_chunk_bytes or shard the channels", c->n_ch, c->max_dec);
		return VDL2GPU_ETOOBIG;
	}
	c->n_slots = std::max(256u, 3u * c->n_ch);
	c->out_cap = std::max(4u << 20, c->n_ch * 512u);
	const uint32_t n_inflight = cfg->n_inflight ? cfg->n_inflight : 4u;
	c->cfg.n_inflight = n_inflight;
	c->event_cap = (cfg->flags & VDL2GPU_FLAG_TRACE) ? (1u << 20) : 1u;
	make_tables(c->tab, cfg->sample_rate);
	memset(&c->stats, 0, sizeof(c->stats));

	/* equal (default) priorities: raising either stage's priority slowed the pair down (tools/probe_overlap.py) */
	CU(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
	if(cfg->flags & VDL2GPU_FLAG_NO_OVERLAP) { c->s_back = c->stream; c->s_mid = c->stream; }
	else {
		CU(cudaStreamCreateWithFlags(&c->s_back, cudaStreamNonBlocking));
		if(c->stages == 3) CU(cudaStreamCreateWithFlags(&c->s_mid, cudaStreamNonBlocking));
		else c->s_mid = c->s_back;
	}
	for(int i = 0; i < 2; i++) CU(cudaEventCreateWithFlags(&c->ev_k2a_done[i], cudaEventDisableTiming));
	for(int i = 0; i < 3; i++) {
		CU(cudaEventCreateWithFlags(&c->ev_k1_done[i], cudaEventDisableTiming));
		CU(cudaEventCreateWithFlags(&c->ev_back_done[i], cudaEventDisableTiming));
	}
	CU(cudaEventCreateWithFlags(&c->ev_input_ready, cudaEventDisableTiming));
	CU(cudaEventCreateWithFlags(&c->ev_input_consumed, cudaEventDisableTiming));
	CU(cudaEventCreateWithFlags(&c->ev_drain, cudaEventDisableTiming));
	if(c->block_trace_cap) {
		const size_t bytes = sizeof(vdl2_block_trace) + (size_t)c->block_trace_cap * sizeof(vdl2_block_rec);
		CU(cudaMalloc(&c->d_block_trace, bytes));
		CU(cudaMemset(c->d_block_trace, 0, bytes));
		CU(cudaMemcpy(&c->d_block_trace->cap, &c->block_trace_cap, 4, cudaMemcpyHostToDevice));
	}
	CU(cudaMalloc(&c->d_tab, sizeof(vdl2_tables)));
	CU(cudaMemcpy(c->d_tab, &c->tab.t, sizeof(vdl2_tables), cudaMemcpyHostToDevice));
	if(c->lane_streams) CU(cudaMalloc(&c->d_samples, (size_t)c->max_pairs * c->n_chp * sizeof(float2)));
	else if(!c->farm) CU(cudaMalloc(&c->d_samples, (size_t)c->n_streams * c->max_pairs * sizeof(float2)));     /* the farm K1 reads raw bytes */
	for(int i = 0; i < 3; i++) {
		CU(cudaMalloc(&c->d_dec3[i], (size_t)c->max_dec * c->n_chp * sizeof(float2)));
		CU(cudaMemset(c->d_dec3[i], 0, (size_t)c->max_dec * c->n_chp * sizeof(float2)));
	}
	for(int i = 0; i < 2; i++) {
		CU(cudaMalloc(&c->d_phase2[i], (size_t)(c->max_dec + VDL2_SYNC_BUFLEN) * c->n_chp * sizeof(float)));
		CU(cudaMemset(c->d_phase2[i], 0, (size_t)(c->max_dec + VDL2_SYNC_BUFLEN) * c->n_chp * sizeof(float)));
		CU(cudaMalloc(&c->d_mag2[i], (size_t)c->max_dec * c->n_chp * sizeof(float)));
	}
	CU(cudaMalloc(&c->d_k1, (size_t)K1_NFIELDS * c->n_chp * 4));
	CU(cudaMalloc(&c->d_k2, (size_t)K2_NFIELDS * c->n_chp * 4));
	CU(cudaMalloc(&c->d_counters, (size_t)VDL2_NUM_COUNTERS * c->n_chp * 4));
	CU(cudaMalloc(&c->d_ring, (size_t)VDL2_SYNC_BUFLEN * c->n_chp * 4));
	CU(cudaMalloc(&c->d_pool, (size_t)c->n_slots * sizeof(vdl2_burst_slot)));
	CU(cudaMalloc(&c->d_free, (size_t)c->n_slots * 4));
	CU(cudaMalloc(&c->d_ready, (size_t)c->n_slots * 4));
	CU(cudaMalloc(&c->d_ctl, sizeof(vdl2_queue_ctl)));
	CU(cudaMalloc(&c->d_events, (size_t)c->event_cap * sizeof(vdl2gpu_event)));
	CU(cudaMemset(c->d_counters, 0, (size_t)VDL2_NUM_COUNTERS * c->n_chp * 4));
	CU(cudaMemset(c->d_ring, 0, (size_t)VDL2_SYNC_BUFLEN * c->n_chp * 4));
	CU(cudaMemset(c->d_pool, 0, (size_t)c->n_slots * sizeof(vdl2_burst_slot)));

	std::vector<uint32_t> centers;                      /* farm: the centre frequency of every channel's stream */
	if(c->farm) {
		/* per 128-slot K1 block: the streams its channels read (compacted: a stream without a channel in the block is not
		 * listed) and every slot's column in that list.  Channels are stream-major and the slot mapping is monotone, so a
		 * block's list comes out in ascending order and a warp holds channels of one or a few neighbouring streams. */
		std::vector<uint32_t> stream_of(c->n_ch);
		centers.resize(c->n_ch);
		for(uint32_t s = 0, k = 0; s < layout->n_streams; s++)
			for(uint32_t i = 0; i < layout->channels_per_stream[s]; i++, k++) {
				stream_of[k] = s;
				centers[k] = layout->centerfreqs ? layout->centerfreqs[s] : cfg->centerfreq;
			}
		const uint32_t blocks = (c->n_chp + K1F_BLOCK - 1) / K1F_BLOCK;
		std::vector<uint32_t> tab((size_t)blocks * (1 + K1F_BLOCK) + c->n_chp, 0u);
		uint32_t *col = tab.data() + (size_t)blocks * (1 + K1F_BLOCK);
		uint32_t max_list = 1;
		for(uint32_t ch = 0; ch < c->n_ch; ch++) {
			const uint32_t slot = slot_of(ch, c->lanes, c->full_warps);
			uint32_t *l = tab.data() + (size_t)(slot / K1F_BLOCK) * (1 + K1F_BLOCK);
			if(l[0] == 0 || l[l[0]] != stream_of[ch]) { l[1 + l[0]] = stream_of[ch]; l[0]++; }
			col[slot] = l[0] - 1;
			max_list = std::max(max_list, l[0]);
		}
		if(vdl2_k1_farm_layout(cfg->oversample, cfg->sample_fmt, max_list, &c->k1f) != 0) {
			snprintf(g_last_error, sizeof(g_last_error), "no receiver-farm K1 tile fits for oversample %u, format %u, %u streams per block",
					cfg->oversample, cfg->sample_fmt, max_list);
			return VDL2GPU_EINVAL;
		}
		CU(cudaMalloc(&c->d_farm, tab.size() * 4));
		CU(cudaMemcpy(c->d_farm, tab.data(), tab.size() * 4, cudaMemcpyHostToDevice));
		c->k1f.raw = nullptr;
		c->k1f.list = c->d_farm;
		c->k1f.col = c->d_farm + (size_t)blocks * (1 + K1F_BLOCK);
		c->k1f.levels = c->d_tab->levels;
	}
	std::vector<uint32_t> k1, k2;
	initial_state(c->cfg, c->freqs.data(), c->farm ? centers.data() : nullptr, c->n_ch, c->n_chp, c->lanes, c->full_warps, k1, k2);
	CU(cudaMemcpy(c->d_k1, k1.data(), k1.size() * 4, cudaMemcpyHostToDevice));
	CU(cudaMemcpy(c->d_k2, k2.data(), k2.size() * 4, cudaMemcpyHostToDevice));
	std::vector<int32_t> fl(c->n_slots);
	for(uint32_t i = 0; i < c->n_slots; i++) fl[i] = (int32_t)i;
	CU(cudaMemcpy(c->d_free, fl.data(), fl.size() * 4, cudaMemcpyHostToDevice));
	vdl2_queue_ctl ctl;
	memset(&ctl, 0, sizeof(ctl));
	ctl.free_top = (int32_t)c->n_slots;
	CU(cudaMemcpy(c->d_ctl, &ctl, sizeof(ctl), cudaMemcpyHostToDevice));

	c->chunks.resize(n_inflight);
	for(auto &s : c->chunks) {
		/* h_raw / d_raw (max_chunk_bytes x n_streams each) are allocated by the first vdl2gpu_submit: hosts that only
		 * use vdl2gpu_submit_device never need them */
		CU(cudaHostAlloc((void **)&s.h_args, sizeof(vdl2_chunk_args), cudaHostAllocDefault));
		CU(cudaMalloc(&s.d_args, sizeof(vdl2_chunk_args)));
		CU(cudaHostAlloc((void **)&s.h_out, sizeof(vdl2_out_header) + c->out_cap, cudaHostAllocMapped));
		CU(cudaHostGetDevicePointer((void **)&s.d_out, s.h_out, 0));
		memset(s.h_out, 0, sizeof(vdl2_out_header));
		CU(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
		for(auto &ev : s.tk) CU(cudaEventCreate(&ev));
	}
	return VDL2GPU_OK;
}

static int check_config(const vdl2gpu_config *cfg, vdl2gpu_ctx **out) {
	if(!cfg || !out || !cfg->freqs || cfg->n_channels == 0 || cfg->oversample == 0 || cfg->sample_fmt > 1
			|| cfg->sample_rate != (uint32_t)VDL2_SYMBOL_RATE * VDL2_SPS * cfg->oversample) {
		snprintf(g_last_error, sizeof(g_last_error), "bad vdl2gpu_config (sample_rate must be 105000*oversample)");
		return VDL2GPU_EINVAL;
	}
	return VDL2GPU_OK;
}

static int create_checked(const vdl2gpu_config *cfg, const vdl2gpu_stream_layout *layout, vdl2gpu_ctx **out) {
	vdl2gpu_ctx *c = new vdl2gpu_ctx();
	int rc = create_impl(cfg, layout, c);
	if(rc != VDL2GPU_OK) { free_ctx(c); *out = nullptr; return rc; }
	*out = c;
	return VDL2GPU_OK;
}

extern "C" int vdl2gpu_create(const vdl2gpu_config *cfg, vdl2gpu_ctx **out) {
	int rc = check_config(cfg, out);
	return rc ? rc : create_checked(cfg, nullptr, out);
}

/* receiver farm: the whole layout is checked here, before any device call */
extern "C" int vdl2gpu_create_streams(const vdl2gpu_config *cfg, const vdl2gpu_stream_layout *layout, vdl2gpu_ctx **out) {
	int rc = check_config(cfg, out);
	if(rc) return rc;
#define FARM_BAD(...) do { snprintf(g_last_error, sizeof(g_last_error), "vdl2gpu_create_streams: " __VA_ARGS__); return VDL2GPU_EINVAL; } while(0)
	if(!layout || !layout->channels_per_stream || layout->n_streams == 0) FARM_BAD("a layout with n_streams >= 1 and channels_per_stream is required");
	if(cfg->n_streams != 0 && cfg->n_streams != layout->n_streams) FARM_BAD("cfg->n_streams (%u) must be 0 or layout->n_streams (%u)", cfg->n_streams, layout->n_streams);
	uint64_t sum = 0;
	for(uint32_t s = 0; s < layout->n_streams; s++) sum += layout->channels_per_stream[s];
	if(sum != cfg->n_channels) FARM_BAD("channels_per_stream sums to %llu, n_channels is %u", (unsigned long long)sum, cfg->n_channels);
	if(cfg->oversample != 10 && cfg->oversample != 13 && cfg->oversample != 20) FARM_BAD("oversample must be 10, 13 or 20 (got %u)", cfg->oversample);
	if(cfg->flags & VDL2GPU_FLAG_K1_SCALAR) FARM_BAD("VDL2GPU_FLAG_K1_SCALAR is not available for receiver farms");
	for(uint32_t s = 0, k = 0; s < layout->n_streams; s++) {
		const int64_t centre = layout->centerfreqs ? layout->centerfreqs[s] : cfg->centerfreq;
		for(uint32_t i = 0; i < layout->channels_per_stream[s]; i++, k++) {
			const int64_t d = (int64_t)cfg->freqs[k] - centre;
			if(2 * (d < 0 ? -d : d) >= (int64_t)cfg->sample_rate)
				FARM_BAD("channel %u (%u Hz) is not within sample_rate/2 of its stream %u's centre %lld Hz", k, cfg->freqs[k], s, (long long)centre);
		}
	}
#undef FARM_BAD
	return create_checked(cfg, layout, out);
}

extern "C" int vdl2gpu_destroy(vdl2gpu_ctx *ctx) { return free_ctx(ctx); }

/* ------------------------------------------------------------------------------------------------
 * harvesting: burst records (mapped pinned memory) -> frames
 * ---------------------------------------------------------------------------------------------- */
static uint32_t synd_weight_of(uint32_t syn) {       /* src/decode.c:98-100 */
	static const uint8_t w[32] = { 0, 1, 1, 2, 1, 2, 1, 1, 1, 1, 1, 1, 1, 2, 1, 1, 1, 1, 2, 1, 2, 1, 1, 2, 1, 1, 1, 1, 1, 1, 1, 1 };
	return w[syn & 31u];
}

/* burst records (region = vdl2_out_header + records) -> frames.  Offsets in the pending frames are relative to the
 * first record.  `dec_end` / `arrival` place the burst in time (see burst_timestamp below). */
static void parse_region(const uint8_t *region, uint32_t out_cap, double rate, struct timeval arrival, uint64_t dec_end,
		uint32_t blob_id, std::vector<pending_frame> &pending, vdl2gpu_stats &stats) {
	vdl2_out_header h;
	memcpy(&h, region, sizeof(h));
	const uint8_t *base = region + sizeof(vdl2_out_header);
	const uint32_t used = std::min(h.bytes_used, out_cap);
	stats.out_bytes += h.bytes_used;            /* out_bytes: record bytes written by K3 (D2H traffic) */
	std::vector<const vdl2_burst_record *> recs;
	recs.reserve(h.n_records);
	uint32_t off = 0;
	for(uint32_t k = 0; k < h.n_records && off + sizeof(vdl2_burst_record) <= used; k++) {
		const vdl2_burst_record *r = reinterpret_cast<const vdl2_burst_record *>(base + off);
		if(r->rec_bytes < sizeof(vdl2_burst_record) || off + r->rec_bytes > used) break;
		recs.push_back(r);
		off += r->rec_bytes;
	}
	std::sort(recs.begin(), recs.end(), [](const vdl2_burst_record *a, const vdl2_burst_record *b) {
		return a->channel != b->channel ? a->channel < b->channel : a->burst_seq < b->burst_seq;
	});
	stats.pool_overflows = h.pool_overflows;
	stats.out_overflows = h.out_overflows;
	for(const vdl2_burst_record *r : recs) {
		stats.bursts++;
		if(r->status != VDL2_BURST_OK) stats.burst_errors++;
		for(uint32_t q = 0; q < r->num_blocks && q < VDL2_MAX_BLOCKS; q++)
			if(r->rs_ret[q] != -128) { stats.blocks_processed++; if(r->rs_ret[q] >= 0) stats.blocks_fec_ok++; }
		const uint32_t *tab = reinterpret_cast<const uint32_t *>(reinterpret_cast<const uint8_t *>(r) + sizeof(vdl2_burst_record));
		const uint8_t *bytes = reinterpret_cast<const uint8_t *>(tab + r->n_frames);
		uint32_t foff = 0;
		const uint64_t sync_idx = (uint64_t)r->sync_lo | ((uint64_t)r->sync_hi << 32);
		for(uint32_t k = 0; k < r->n_frames; k++) {
			const uint32_t len = tab[k] & 0xFFFFu, crc = tab[k] >> 16;
			pending_frame pf;
			memset(&pf.f, 0, sizeof(pf.f));
			pf.blob = blob_id;
			pf.offset = (uint32_t)((bytes + foff) - base);
			foff += len;
			pf.f.channel = r->channel; pf.f.freq = r->freq; pf.f.burst_seq = r->burst_seq; pf.f.idx = (int32_t)k;
			pf.f.len = len;
			pf.f.synd_weight = synd_weight_of(r->syndrome);
			pf.f.datalen_octets = r->datalen_bits / 8 + ((r->datalen_bits % 8) != 0);
			pf.f.num_fec_corrections = r->num_fec_corrections;
			pf.f.frame_pwr = r->frame_pwr; pf.f.mag_nf = r->mag_nf;
			pf.f.frame_pwr_dbfs = 10.0f * log10f(r->frame_pwr);                  /* src/decode.c:180 */
			pf.f.nf_pwr_dbfs = 20.0f * log10f(r->mag_nf + 0.001f);               /* src/decode.c:181 */
			pf.f.ppm_error = r->ppm_error;
			pf.f.sync_dec_index = sync_idx;
			/* the reference stamps gettimeofday() at sync (src/demod.c:246); here: arrival time of the chunk
			 * being processed when the burst completed, moved back by the distance to the sync sample */
			double back = dec_end > sync_idx ? ((double)dec_end - (double)sync_idx) / rate : 0.0;
			double ts = (double)arrival.tv_sec + 1e-6 * (double)arrival.tv_usec - back;
			pf.f.burst_timestamp.tv_sec = (time_t)floor(ts);
			pf.f.burst_timestamp.tv_usec = (suseconds_t)((ts - floor(ts)) * 1e6);
			pf.f.fcs_residue = (uint16_t)crc;
			pf.f.fcs_ok = (len >= 11 && crc == 0xF0B8u) ? 1 : 0;
			stats.msg_good++;
			if(len >= 11) { if(crc == 0xF0B8u) stats.fcs_good++; else stats.fcs_bad++; }
			pending.push_back(pf);
		}
	}
}

static void harvest(vdl2gpu_ctx *c, chunk_slot &s) {
	if(s.timed) {
		static const int from[5] = { 0, 1, 3, 7, 4 }, to[5] = { 1, 2, 6, 4, 5 };   /* K0, K1 front stream; K2a middle stream; K2, K3 back stream */
		for(int k = c->farm ? 1 : 0; k < 5; k++) {              /* a farm has no K0 */
			float ms = 0.f;
			if(cudaEventElapsedTime(&ms, s.tk[from[k]], s.tk[to[k]]) == cudaSuccess) { c->k_ms[k] += ms; c->k_launches[k]++; }
		}
		if(c->ev_t0 && c->timeline.size() < 8u * 4096u) {
			static const int order[7] = { 0, 2, 3, 6, 7, 4, 5 };   /* front start, K1 end, K2a start, K2a end, K2 start, K2|K3, K3 end */
			c->timeline.push_back((float)s.seq);
			for(int k = 0; k < 7; k++) {
				float ms = -1.f;
				if(cudaEventElapsedTime(&ms, c->ev_t0, s.tk[order[k]]) != cudaSuccess) { cudaGetLastError(); ms = -1.f; }
				c->timeline.push_back(ms);
			}
		}
		s.timed = false;
	}
	/* one copy out of the mapped region (header + the bytes K3 used), so the region can be handed back to the device at once */
	const vdl2_out_header *h = reinterpret_cast<const vdl2_out_header *>(s.h_out);
	const uint32_t used = std::min(h->bytes_used, c->out_cap);
	c->blobs.emplace_back(s.h_out, s.h_out + sizeof(vdl2_out_header) + used);
	const uint32_t blob_id = (uint32_t)c->blobs.size() - 1;
	const double rate = (double)c->cfg.sample_rate / (double)c->cfg.oversample;     /* decimated samples per second */
	parse_region(c->blobs.back().data(), c->out_cap, rate, s.arrival, s.dec_base + s.n_dec, blob_id, c->pending, c->stats);
	c->stats.chunks_completed++;
	s.busy = false;
}

static int deliver(vdl2gpu_ctx *c, vdl2gpu_frame_cb cb, void *user) {
	int n = (int)c->pending.size();
	/* bursts dropped on the device (burst pool or output region exhausted) are an error the caller must see, once per
	 * increase; the frames that did arrive are still delivered first */
	const uint64_t ov = c->stats.pool_overflows + c->stats.out_overflows;
	if(ov > c->overflows_reported) {
		snprintf(g_last_error, sizeof(g_last_error), "%llu burst(s) dropped on the device: burst pool overflows %llu, output region overflows %llu",
				(unsigned long long)(ov - c->overflows_reported), (unsigned long long)c->stats.pool_overflows, (unsigned long long)c->stats.out_overflows);
		c->overflows_reported = ov;
		n = VDL2GPU_EOVERFLOW;
	}
	if(cb) {
		for(auto &pf : c->pending) {
			pf.f.data = c->blobs[pf.blob].data() + sizeof(vdl2_out_header) + pf.offset;
			cb(&pf.f, user);
		}
	}
	c->pending.clear();
	c->blobs.clear();
	return n;
}

/* ------------------------------------------------------------------------------------------------
 * data path
 * ---------------------------------------------------------------------------------------------- */
static int ensure_raw(vdl2gpu_ctx *c, chunk_slot &s) {
	if(s.h_raw) return VDL2GPU_OK;
	const size_t bytes = (size_t)c->cfg.max_chunk_bytes * c->n_streams;
	if(bytes >= ((size_t)1 << 32)) {          /* the host path stages all streams of a chunk in one pinned buffer */
		snprintf(g_last_error, sizeof(g_last_error), "vdl2gpu_submit: n_streams x max_chunk_bytes must stay below 4 GiB (use vdl2gpu_submit_device)");
		return VDL2GPU_ETOOBIG;
	}
	CU(cudaHostAlloc((void **)&s.h_raw, bytes, cudaHostAllocDefault));
	CU(cudaMalloc(&s.d_raw, bytes));
	return VDL2GPU_OK;
}

static int acquire_slot(vdl2gpu_ctx *c, chunk_slot **out) {
	chunk_slot &s = c->chunks[c->next_slot];
	if(s.busy) {
		/* back-pressure: the producer blocks until the oldest chunk has drained (cf. the demods_ready
		 * barrier in src/demod.c:342) */
		CU(cudaEventSynchronize(s.done));
		harvest(c, s);
		if(!c->inflight.empty() && c->inflight.front() == c->next_slot) c->inflight.pop_front();
	}
	*out = &s;
	return VDL2GPU_OK;
}

/* parameter blocks of one chunk (number `seq`).  With `ca` the per-chunk values come from the device copy of the chunk
 * arguments (graph replay); the sizes given here then only size the grids. */
static void fill_params(vdl2gpu_ctx *c, chunk_slot &s, uint64_t seq, uint32_t n_pairs, uint32_t cnt0, uint32_t n_dec, uint32_t prev_n_dec,
		uint64_t dec_base, const vdl2_chunk_args *ca, vdl2_k1_params &p1, vdl2_k2a_params &pa, vdl2_k2_params &p2, vdl2_k3_params &p3) {
	float2 *d_dec = c->d_dec3[seq % 3u];
	const int pb = (int)(seq & 1u);
	p1.samples = c->d_samples; p1.n_pairs = n_pairs; p1.oversample = c->cfg.oversample; p1.cnt0 = cnt0;
	p1.n_ch = c->n_ch; p1.n_chp = c->n_chp; p1.lanes = c->lanes; p1.full_warps = c->full_warps; p1.dec = d_dec; p1.state = c->d_k1;
	p1.lut = reinterpret_cast<const float4 *>(c->d_tab->lut);
	p1.a0 = c->tab.t.A[0]; p1.a1 = c->tab.t.A[1]; p1.a2 = c->tab.t.A[2]; p1.b1 = c->tab.t.B[1]; p1.b2 = c->tab.t.B[2];
	p1.one = 1.0f; p1.neg_one = -1.0f; p1.two = 2.0f;
	p1.trace_blocks = c->d_block_trace; p2.trace_blocks = c->d_block_trace;
	p1.ch_per_stream = c->ch_per_stream; p1.stream_stride = c->lane_streams ? c->n_chp : c->max_pairs; p1.ca = ca;
	p1.phase = c->fuse_phase ? c->d_phase2[pb] : nullptr; p1.phase_prev = c->d_phase2[pb ^ 1]; p1.prev_n_dec = prev_n_dec;
	/* the default walk (variant 5) computes the four magnitudes a block needs from the staged samples: no magnitude plane */
	const bool need_mag = (c->k2_variant & 0xFF) >= 0 && (c->k2_variant & 0xFF) <= 4;
	pa.dec = d_dec; pa.phase = c->d_phase2[pb]; pa.mag = need_mag ? c->d_mag2[pb] : nullptr; pa.phase_prev = c->d_phase2[pb ^ 1];
	pa.n_dec = n_dec; pa.prev_n_dec = prev_n_dec; pa.n_ch = c->n_ch; pa.n_chp = c->n_chp; pa.lanes = c->lanes; pa.full_warps = c->full_warps;
	pa.mode = (uint32_t)c->k2a_mode; pa.split = c->k2a_split; pa.ca = ca;
	p2.dec = d_dec; p2.phase = c->d_phase2[pb]; p2.mag = c->d_mag2[pb]; p2.hist_tmp = nullptr; p2.n_dec = n_dec; p2.n_ch = c->n_ch; p2.n_chp = c->n_chp;
	p2.lanes = c->lanes; p2.full_warps = c->full_warps; p2.dec_base = dec_base;
	p2.state = c->d_k2; p2.ring = c->d_ring; p2.tables = c->d_tab; p2.max_ppm = c->cfg.max_ppm; p2.s27 = c->tab.s27;
	p2.pool = c->d_pool; p2.free_list = c->d_free; p2.ready = c->d_ready; p2.ctl = c->d_ctl;
	p2.events = c->d_events; p2.event_cap = c->event_cap; p2.trace = (c->cfg.flags & VDL2GPU_FLAG_TRACE) ? 1u : 0u;
	p2.variant = (uint32_t)c->k2_variant; p2.k2a_mode = (uint32_t)c->k2a_mode; p2.ca = ca;
	p3.pool = c->d_pool; p3.free_list = c->d_free; p3.ready = c->d_ready; p3.ctl = c->d_ctl; p3.tables = c->d_tab;
	p3.out = s.d_out; p3.out_cap = c->out_cap; p3.n_chp = c->n_chp; p3.counters = c->d_counters;
}

#define K3_GRID (148u * 16u)      /* 16 resident blocks per SM: ~1.5 bursts per block per chunk at the bench traffic */

/* One CUDA graph per stage, captured once per (slot, chunk number mod 6 = dec buffer and plane) for the chunk shape
 * (n_pairs) and replayed: a chunk then costs three graph launches and a handful of event calls instead of seven kernel
 * launches.  Everything that differs between two chunks of the same shape (input pointer, decimation phase, sample
 * counts, absolute sample index) travels in the chunk-argument block the front graph copies to the device first. */
static int capture_one(cudaStream_t st, cudaGraphExec_t *out, int (*body)(void *), void *arg) {
	cudaGraph_t g = nullptr;
	CU(cudaStreamBeginCapture(st, cudaStreamCaptureModeRelaxed));
	int rc = body(arg);
	cudaError_t e = cudaStreamEndCapture(st, &g);
	if(rc != 0 || e != cudaSuccess) { if(g) cudaGraphDestroy(g); cudaGetLastError(); return rc ? rc : fail_cuda(e, "cudaStreamEndCapture", __LINE__); }
	e = cudaGraphInstantiate(out, g, 0);
	cudaGraphDestroy(g);
	if(e != cudaSuccess) return fail_cuda(e, "cudaGraphInstantiate", __LINE__);
	return VDL2GPU_OK;
}

struct capture_env { vdl2gpu_ctx *c; chunk_slot *s; uint64_t seq; uint32_t n_pairs; uint32_t k0_fmt; };
#define CAPTURE_PARAMS \
	capture_env *e = static_cast<capture_env *>(a); \
	vdl2gpu_ctx *c = e->c; \
	vdl2_k1_params p1; vdl2_k2a_params pa; vdl2_k2_params p2; vdl2_k3_params p3; \
	const uint32_t os = c->cfg.oversample; \
	fill_params(c, *e->s, e->seq, e->n_pairs, 0, (os - 1 + e->n_pairs) / os, 0, 0, e->s->d_args, p1, pa, p2, p3)

static int body_front(void *a) {
	CAPTURE_PARAMS;
	(void)pa; (void)p2; (void)p3;
	CU(cudaMemcpyAsync(e->s->d_args, e->s->h_args, sizeof(vdl2_chunk_args), cudaMemcpyHostToDevice, c->stream));
	const uint32_t bpp = c->cfg.sample_fmt == VDL2GPU_FMT_S16_LE ? 4u : 2u;
	if(c->farm) { KL(vdl2_launch_k1_farm(&p1, &c->k1f, c->stream)); return 0; }      /* no K0: the farm K1 reads ca->raw */
	if(c->lane_streams) KL(vdl2_launch_k0_lanes(nullptr, e->n_pairs, e->k0_fmt, c->d_tab->levels, reinterpret_cast<float *>(c->d_samples), c->n_streams,
			e->n_pairs * bpp, c->n_chp, c->lanes, c->full_warps, e->s->d_args, c->stream));
	else KL(vdl2_launch_k0(nullptr, e->n_pairs, e->k0_fmt, c->d_tab->levels, reinterpret_cast<float *>(c->d_samples), c->n_streams,
			e->n_pairs * bpp, c->max_pairs, e->s->d_args, c->stream));
	KL(vdl2_launch_k1(&p1, (c->cfg.flags & VDL2GPU_FLAG_K1_SCALAR) ? 1 : 0, c->k1_variant, c->stream));
	return 0;
}
static int body_k2a(void *a) {
	CAPTURE_PARAMS;
	(void)p1; (void)p2; (void)p3;
	KL(vdl2_launch_k2a_warps(&pa, c->s_mid));
	return 0;
}
static int body_back(void *a) {
	CAPTURE_PARAMS;
	(void)p1; (void)pa;
	KL(vdl2_launch_k2(&p2, c->s_back));
	KL(vdl2_launch_k3(&p3, K3_GRID, c->s_back));
	return 0;
}

static int ensure_graphs(vdl2gpu_ctx *c, chunk_slot &s, uint64_t seq, uint32_t n_pairs, uint32_t k0_fmt) {
	const int k = (int)(seq % 6u);
	if(s.g_front[k] && s.graph_pairs[k] == n_pairs) return VDL2GPU_OK;
	if(s.g_front[k]) { cudaGraphExecDestroy(s.g_front[k]); s.g_front[k] = nullptr; }
	if(s.g_k2a[k]) { cudaGraphExecDestroy(s.g_k2a[k]); s.g_k2a[k] = nullptr; }
	if(s.g_back[k]) { cudaGraphExecDestroy(s.g_back[k]); s.g_back[k] = nullptr; }
	capture_env e = { c, &s, seq, n_pairs, k0_fmt };
	int rc = capture_one(c->stream, &s.g_front[k], body_front, &e);
	if(rc == 0 && !c->fuse_phase) rc = capture_one(c->s_mid, &s.g_k2a[k], body_k2a, &e);
	if(rc == 0) rc = capture_one(c->s_back, &s.g_back[k], body_back, &e);
	if(rc == 0) s.graph_pairs[k] = n_pairs;
	return rc;
}

static int run_chain(vdl2gpu_ctx *c, chunk_slot &s, const void *d_raw, uint32_t n_pairs, uint32_t k0_fmt = 0xFFFFFFFFu) {
	const uint32_t os = c->cfg.oversample;
	const bool planar = k0_fmt != 0xFFFFFFFFu;
	if(!planar) k0_fmt = c->cfg.sample_fmt;
	s.first_pair = c->total_pairs;
	s.n_pairs = n_pairs;
	s.dec_base = c->total_dec;
	s.n_dec = (c->decim_cnt + n_pairs) / os;
	gettimeofday(&s.arrival, NULL);
	s.timed = c->timing;
	const uint64_t seq = c->chunk_seq;
	const int db = (int)(seq % 3u), pb = (int)(seq & 1u), gk = (int)(seq % 6u);
	const uint32_t bpp = c->cfg.sample_fmt == VDL2GPU_FMT_S16_LE ? 4u : 2u;
	const bool overlap = c->s_back != c->stream;
	s.seq = seq;
	bool graph = c->use_graphs && !planar && overlap;
	if(graph && c->graph_nominal == 0) c->graph_nominal = n_pairs;
	graph = graph && n_pairs == c->graph_nominal;            /* odd-sized chunks (the tail of a file) take the direct path */
	if(graph && ensure_graphs(c, s, seq, n_pairs, k0_fmt) != VDL2GPU_OK) { c->use_graphs = false; graph = false; }
	vdl2_k1_params p1; vdl2_k2a_params pa; vdl2_k2_params p2; vdl2_k3_params p3;
	fill_params(c, s, seq, n_pairs, c->decim_cnt, s.n_dec, c->last_n_dec, s.dec_base, nullptr, p1, pa, p2, p3);
	if(graph) {
		s.h_args->raw = d_raw; s.h_args->dec_base = s.dec_base; s.h_args->n_pairs = n_pairs; s.h_args->cnt0 = c->decim_cnt;
		s.h_args->n_dec = s.n_dec; s.h_args->prev_n_dec = c->last_n_dec;
	}
	/* ---- front stage: K0, K1 -> dec[db] (free once K2 of chunk c-3 is done) ---- */
	/* Fused phase pass: K1 also writes phase plane pb, which the walk of chunk c-2 read; the front stage then runs in lock
	 * step with the back stage of chunk c-1 - K1(c) and K2(c-1) start together once K3(c-2) has finished, again one block per
	 * SM each into an empty machine - and there is no middle stage. */
	if(c->fuse_phase) { if(seq >= 2 && overlap) CU(cudaStreamWaitEvent(c->stream, c->ev_back_done[(seq - 2) % 3u], 0)); }
	else if(seq >= 3) CU(cudaStreamWaitEvent(c->stream, c->ev_back_done[db], 0));
	/* Two-stage schedule (default): K1 of this chunk starts when K2a of the previous chunk has finished.  K2a is a short
	 * full-occupancy pass; when it ends the GPU is empty, and K2 of chunk c-1 and K1 of chunk c are then launched into that
	 * empty machine together, one block per SM each - the only arrangement in which the block scheduler was found to keep
	 * the two long kernels side by side on every SM, launch after launch (see the slot mapping in create_impl). */
	if(!c->fuse_phase && c->stages == 2 && seq >= 1 && overlap) CU(cudaStreamWaitEvent(c->stream, c->ev_k2a_done[pb ^ 1], 0));
	if(s.timed) { CU(cudaEventRecord(s.tk[0], c->stream)); if(graph) CU(cudaEventRecord(s.tk[1], c->stream)); }
	if(graph) {
		CU(cudaGraphLaunch(s.g_front[gk], c->stream));
	} else if(c->farm) {
		vdl2_k1_farm f = c->k1f;
		f.raw = d_raw;
		if(s.timed) CU(cudaEventRecord(s.tk[1], c->stream));
		KL(vdl2_launch_k1_farm(&p1, &f, c->stream));
	} else {
		if(c->lane_streams) KL(vdl2_launch_k0_lanes(d_raw, n_pairs, k0_fmt, c->d_tab->levels, reinterpret_cast<float *>(c->d_samples), c->n_streams,
				n_pairs * bpp, c->n_chp, c->lanes, c->full_warps, nullptr, c->stream));
		else KL(vdl2_launch_k0(d_raw, n_pairs, k0_fmt, c->d_tab->levels, reinterpret_cast<float *>(c->d_samples), c->n_streams,
				n_pairs * bpp, c->max_pairs, nullptr, c->stream));
		if(s.timed) CU(cudaEventRecord(s.tk[1], c->stream));
		KL(vdl2_launch_k1(&p1, (c->cfg.flags & VDL2GPU_FLAG_K1_SCALAR) ? 1 : 0, c->k1_variant, c->stream));
	}
	if(s.timed) CU(cudaEventRecord(s.tk[2], c->stream));
	CU(cudaEventRecord(c->ev_input_consumed, c->stream));
	CU(cudaEventRecord(c->ev_k1_done[db], c->stream));
	/* ---- middle stage: K2a -> plane[pb] (free once K2 of chunk c-2 is done), history from plane[pb ^ 1] (chunk c-1, same stream) ---- */
	if(c->fuse_phase) {
		if(s.timed) { CU(cudaEventRecord(s.tk[3], c->stream)); CU(cudaEventRecord(s.tk[6], c->stream)); }
		CU(cudaEventRecord(c->ev_k2a_done[pb], c->stream));
	} else {
		CU(cudaStreamWaitEvent(c->s_mid, c->ev_k1_done[db], 0));
		if(seq >= 2 && overlap) CU(cudaStreamWaitEvent(c->s_mid, c->ev_back_done[(seq - 2) % 3u], 0));
		if(s.timed) CU(cudaEventRecord(s.tk[3], c->s_mid));
		if(graph) CU(cudaGraphLaunch(s.g_k2a[gk], c->s_mid));
		else KL(vdl2_launch_k2a_warps(&pa, c->s_mid));
		if(s.timed) CU(cudaEventRecord(s.tk[6], c->s_mid));
		CU(cudaEventRecord(c->ev_k2a_done[pb], c->s_mid));
	}
	/* ---- back stage: K2, K3 ---- */
	CU(cudaStreamWaitEvent(c->s_back, c->ev_k2a_done[pb], 0));
	if(s.timed) CU(cudaEventRecord(s.tk[7], c->s_back));
	if(graph) {
		CU(cudaGraphLaunch(s.g_back[gk], c->s_back));
		if(s.timed) CU(cudaEventRecord(s.tk[4], c->s_back));
		c->stats.graph_launches += c->fuse_phase ? 2 : 3;
	} else {
		KL(vdl2_launch_k2(&p2, c->s_back));
		if(s.timed) CU(cudaEventRecord(s.tk[4], c->s_back));
		KL(vdl2_launch_k3(&p3, K3_GRID, c->s_back));
	}
	if(s.timed) CU(cudaEventRecord(s.tk[5], c->s_back));
	CU(cudaEventRecord(c->ev_back_done[db], c->s_back));
	CU(cudaEventRecord(s.done, c->s_back));
	c->chunk_seq++;
	s.busy = true;
	c->inflight.push_back(c->next_slot);
	c->next_slot = (c->next_slot + 1) % (uint32_t)c->chunks.size();
	c->decim_cnt = (c->decim_cnt + n_pairs) % os;
	c->total_pairs += n_pairs;
	c->total_dec += s.n_dec;
	c->last_n_dec = s.n_dec;
	c->stats.chunks_submitted++;
	c->stats.iq_samples += n_pairs;
	c->stats.dec_samples += s.n_dec;
	c->stats.kernel_launches += (n_pairs ? (c->farm ? 1 : 2) : 0) + (c->fuse_phase ? 0 : 1) + (s.n_dec ? 1 : 0) + 2;
	return VDL2GPU_OK;
}

extern "C" int vdl2gpu_submit(vdl2gpu_ctx *c, const void *iq, uint32_t len) {
	if(!c || (!iq && len)) return VDL2GPU_EINVAL;
	if(len == 0) return VDL2GPU_OK;                                   /* src/demod.c:341,358 */
	if(len > c->cfg.max_chunk_bytes) return VDL2GPU_ETOOBIG;
	const uint32_t bpp = c->cfg.sample_fmt == VDL2GPU_FMT_S16_LE ? 4u : 2u;
	const uint32_t n_pairs = len / bpp;
	if(n_pairs == 0) return VDL2GPU_OK;
	CU(cudaSetDevice(c->device));
	chunk_slot *s;
	int rc = acquire_slot(c, &s);
	if(rc) return rc;
	rc = ensure_raw(c, *s);
	if(rc) return rc;
	/* n_streams buffers of `len` bytes back to back; a ragged tail (len not a multiple of the sample size) is dropped
	 * per stream, so the streams are repacked at n_pairs * bpp */
	const size_t used = (size_t)n_pairs * bpp;
	for(uint32_t st = 0; st < c->n_streams; st++)
		memcpy(s->h_raw + st * used, static_cast<const uint8_t *>(iq) + (size_t)st * len, used);
	CU(cudaMemcpyAsync(s->d_raw, s->h_raw, used * c->n_streams, cudaMemcpyHostToDevice, c->stream));
	return run_chain(c, *s, s->d_raw, n_pairs);
}

extern "C" int vdl2gpu_submit_planar_s16(vdl2gpu_ctx *c, const int16_t *xi, const int16_t *xq, uint32_t n_pairs) {
	if(!c || ((!xi || !xq) && n_pairs)) return VDL2GPU_EINVAL;
	if(c->cfg.sample_fmt != VDL2GPU_FMT_S16_LE || c->n_streams != 1 || c->farm) return VDL2GPU_EINVAL;
	if(n_pairs == 0) return VDL2GPU_OK;
	if((uint64_t)n_pairs * 4u > c->cfg.max_chunk_bytes) return VDL2GPU_ETOOBIG;
	CU(cudaSetDevice(c->device));
	chunk_slot *s;
	int rc = acquire_slot(c, &s);
	if(rc) return rc;
	rc = ensure_raw(c, *s);
	if(rc) return rc;
	memcpy(s->h_raw, xi, (size_t)n_pairs * 2);
	memcpy(s->h_raw + (size_t)n_pairs * 2, xq, (size_t)n_pairs * 2);
	CU(cudaMemcpyAsync(s->d_raw, s->h_raw, (size_t)n_pairs * 4, cudaMemcpyHostToDevice, c->stream));
	return run_chain(c, *s, s->d_raw, n_pairs, 2u);
}

/* src/fmtr-binary.c + src/output-file.c:181-189: one raw frame in the reference's archive format, i.e. a 2-octet
 * big-endian length (its own two octets included) followed by the proto3 message dumpvdl2.raw_avlc_frame
 * (proto/dumpvdl2.proto:25-48).  Files made of these records replay through an unmodified
 * `dumpvdl2 --raw-frames-file` (src/input-raw_frames_file.c:33-75).  Returns the record size or a negative error. */
static size_t pb_varint(uint8_t *o, uint64_t v) { size_t n = 0; do { uint8_t b = v & 0x7Fu; v >>= 7; o[n++] = (uint8_t)(b | (v ? 0x80u : 0u)); } while(v); return n; }
static size_t pb_u32_field(uint8_t *o, int field, uint32_t v) { if(!v) return 0; size_t n = pb_varint(o, (uint64_t)field << 3); return n + pb_varint(o + n, v); }
static size_t pb_i64_field(uint8_t *o, int field, int64_t v) { if(!v) return 0; size_t n = pb_varint(o, (uint64_t)field << 3); return n + pb_varint(o + n, (uint64_t)v); }
static size_t pb_f32_field(uint8_t *o, int field, float v) { uint32_t u; memcpy(&u, &v, 4); if(!u) return 0; size_t n = pb_varint(o, ((uint64_t)field << 3) | 5u); memcpy(o + n, &u, 4); return n + 4; }

extern "C" int vdl2gpu_serialize_raw_frame(const vdl2gpu_frame *f, const char *station_id, uint8_t *out, size_t cap) {
	if(!f || !out || (f->len && !f->data)) return VDL2GPU_EINVAL;
	uint8_t ts[24], md[96 + 256];
	size_t nts = 0, nmd = 0;
	nts += pb_i64_field(ts + nts, 1, (int64_t)f->burst_timestamp.tv_sec);
	nts += pb_i64_field(ts + nts, 2, (int64_t)f->burst_timestamp.tv_usec);
	size_t sl = station_id ? strlen(station_id) : 0;
	if(sl > 255) sl = 255;                                          /* STATION_ID_LEN_MAX, src/dumpvdl2.h:193 */
	if(sl) { nmd += pb_varint(md + nmd, (1u << 3) | 2u); nmd += pb_varint(md + nmd, sl); memcpy(md + nmd, station_id, sl); nmd += sl; }
	nmd += pb_u32_field(md + nmd, 2, f->freq);
	nmd += pb_u32_field(md + nmd, 3, f->synd_weight);
	nmd += pb_u32_field(md + nmd, 4, f->datalen_octets);
	nmd += pb_f32_field(md + nmd, 5, f->frame_pwr_dbfs);
	nmd += pb_f32_field(md + nmd, 6, f->nf_pwr_dbfs);
	nmd += pb_f32_field(md + nmd, 7, f->ppm_error);
	nmd += pb_i64_field(md + nmd, 8, 1);                            /* metadata version, src/decode.c:177 */
	nmd += pb_i64_field(md + nmd, 9, (int64_t)f->num_fec_corrections);
	nmd += pb_i64_field(md + nmd, 10, (int64_t)f->idx);
	nmd += pb_varint(md + nmd, (11u << 3) | 2u); nmd += pb_varint(md + nmd, nts); memcpy(md + nmd, ts, nts); nmd += nts;
	uint8_t hdr[16];
	size_t nh = pb_varint(hdr, (1u << 3) | 2u); nh += pb_varint(hdr + nh, nmd);
	uint8_t dh[16];
	size_t nd = f->len ? pb_varint(dh, (2u << 3) | 2u) : 0;
	if(f->len) nd += pb_varint(dh + nd, f->len);
	const size_t total = 2 + nh + nmd + nd + f->len;
	if(total > 65535 || total > cap) return VDL2GPU_ETOOBIG;         /* OUT_BINARY_FRAME_LEN_MAX, src/output-file.h:26 */
	uint8_t *o = out;
	*o++ = (uint8_t)(total >> 8); *o++ = (uint8_t)total;
	memcpy(o, hdr, nh); o += nh; memcpy(o, md, nmd); o += nmd;
	memcpy(o, dh, nd); o += nd; if(f->len) memcpy(o, f->data, f->len);
	return (int)total;
}

extern "C" int vdl2gpu_submit_device(vdl2gpu_ctx *c, const void *dev_iq, uint32_t len, void *producer_stream) {
	if(!c || (!dev_iq && len)) return VDL2GPU_EINVAL;
	if(len == 0) return VDL2GPU_OK;
	if(len > c->cfg.max_chunk_bytes) return VDL2GPU_ETOOBIG;
	const uint32_t bpp = c->cfg.sample_fmt == VDL2GPU_FMT_S16_LE ? 4u : 2u;
	const uint32_t n_pairs = len / bpp;
	if(n_pairs == 0) return VDL2GPU_OK;
	if(c->n_streams > 1 && len % bpp != 0) return VDL2GPU_EINVAL;     /* streams are `len` bytes apart in dev_iq */
	CU(cudaSetDevice(c->device));
	chunk_slot *s;
	int rc = acquire_slot(c, &s);
	if(rc) return rc;
	CU(cudaEventRecord(c->ev_input_ready, (cudaStream_t)producer_stream));
	CU(cudaStreamWaitEvent(c->stream, c->ev_input_ready, 0));
	return run_chain(c, *s, dev_iq, n_pairs);
}

extern "C" int vdl2gpu_wait_input_consumed(vdl2gpu_ctx *c, void *stream) {
	if(!c) return VDL2GPU_EINVAL;
	CU(cudaStreamWaitEvent((cudaStream_t)stream, c->ev_input_consumed, 0));
	return VDL2GPU_OK;
}

extern "C" int vdl2gpu_stream_wait(vdl2gpu_ctx *c, void *stream) {
	if(!c) return VDL2GPU_EINVAL;
	CU(cudaSetDevice(c->device));
	CU(cudaEventRecord(c->ev_drain, c->s_back));        /* every chunk's chain ends on the back stream */
	CU(cudaStreamWaitEvent((cudaStream_t)stream, c->ev_drain, 0));
	return VDL2GPU_OK;
}

extern "C" int vdl2gpu_poll(vdl2gpu_ctx *c, vdl2gpu_frame_cb cb, void *user) {
	if(!c) return VDL2GPU_EINVAL;
	CU(cudaSetDevice(c->device));
	while(!c->inflight.empty()) {
		chunk_slot &s = c->chunks[c->inflight.front()];
		if(!s.busy) { c->inflight.pop_front(); continue; }
		cudaError_t q = cudaEventQuery(s.done);
		if(q == cudaErrorNotReady) break;
		if(q != cudaSuccess) return fail_cuda(q, "cudaEventQuery", __LINE__);
		harvest(c, s);
		c->inflight.pop_front();
	}
	return deliver(c, cb, user);
}

extern "C" int vdl2gpu_chunks_in_flight(vdl2gpu_ctx *c) {
	if(!c) return VDL2GPU_EINVAL;
	int n = 0;
	for(auto &s : c->chunks) n += s.busy ? 1 : 0;
	return n;
}

extern "C" int vdl2gpu_flush(vdl2gpu_ctx *c, vdl2gpu_frame_cb cb, void *user) {
	if(!c) return VDL2GPU_EINVAL;
	CU(cudaSetDevice(c->device));
	CU(cudaStreamSynchronize(c->stream));
	CU(cudaStreamSynchronize(c->s_back));
	while(!c->inflight.empty()) {
		chunk_slot &s = c->chunks[c->inflight.front()];
		if(s.busy) harvest(c, s);
		c->inflight.pop_front();
	}
	return deliver(c, cb, user);
}

static int read_counters(vdl2gpu_ctx *c, std::vector<uint32_t> &k3, std::vector<uint32_t> &sync, std::vector<uint32_t> &hdr) {
	CU(cudaSetDevice(c->device));
	CU(cudaStreamSynchronize(c->stream));
	CU(cudaStreamSynchronize(c->s_back));
	k3.resize((size_t)VDL2_NUM_COUNTERS * c->n_chp);
	sync.resize(c->n_chp); hdr.resize(c->n_chp);
	CU(cudaMemcpy(k3.data(), c->d_counters, k3.size() * 4, cudaMemcpyDeviceToHost));
	CU(cudaMemcpy(sync.data(), c->d_k2 + (size_t)K2_CNT_SYNC * c->n_chp, c->n_chp * 4, cudaMemcpyDeviceToHost));
	CU(cudaMemcpy(hdr.data(), c->d_k2 + (size_t)K2_CNT_HDR_GOOD * c->n_chp, c->n_chp * 4, cudaMemcpyDeviceToHost));
	return VDL2GPU_OK;
}

extern "C" int vdl2gpu_get_stats(vdl2gpu_ctx *c, vdl2gpu_stats *out) {
	if(!c || !out) return VDL2GPU_EINVAL;
	std::vector<uint32_t> k3, sync, hdr;
	int rc = read_counters(c, k3, sync, hdr);
	if(rc) return rc;
	uint64_t a = 0, b = 0;
	for(uint32_t ch = 0; ch < c->n_ch; ch++) { a += sync[slot_of(ch, c->lanes, c->full_warps)]; b += hdr[slot_of(ch, c->lanes, c->full_warps)]; }
	c->stats.demod_sync_good = a;
	c->stats.decoder_crc_good = b;
	*out = c->stats;
	return VDL2GPU_OK;
}

extern "C" int vdl2gpu_get_channel_counters(vdl2gpu_ctx *c, uint64_t *out, uint32_t n_channels) {
	if(!c || !out || n_channels > c->n_ch) return VDL2GPU_EINVAL;
	std::vector<uint32_t> k3, sync, hdr;
	int rc = read_counters(c, k3, sync, hdr);
	if(rc) return rc;
	for(uint32_t ch = 0; ch < n_channels; ch++) {
		uint64_t *o = out + (size_t)ch * VDL2_NUM_COUNTERS;
		for(int k = 0; k < VDL2_NUM_COUNTERS; k++) o[k] = k3[(size_t)k * c->n_chp + ch];
		o[VDL2_CNT_SYNC_GOOD] = sync[slot_of(ch, c->lanes, c->full_warps)];          /* K2's own counters live in its state planes, by slot */
		o[VDL2_CNT_HDR_CRC_GOOD] = hdr[slot_of(ch, c->lanes, c->full_warps)];
	}
	return VDL2GPU_OK;
}

extern "C" int vdl2gpu_get_tables(vdl2gpu_ctx *c, float levels[256], float sin_lut[257], float cos_lut[257],
		float A[3], float B[3], float lr_X[16], float *lr_denom, float pr_phase[16]) {
	if(!c) return VDL2GPU_EINVAL;
	if(levels) memcpy(levels, c->tab.t.levels, sizeof(c->tab.t.levels));
	if(sin_lut) memcpy(sin_lut, c->tab.sin_lut, sizeof(c->tab.sin_lut));
	if(cos_lut) memcpy(cos_lut, c->tab.cos_lut, sizeof(c->tab.cos_lut));
	if(A) memcpy(A, c->tab.t.A, 12);
	if(B) memcpy(B, c->tab.t.B, 12);
	if(lr_X) memcpy(lr_X, c->tab.t.lr_X, 64);
	if(lr_denom) *lr_denom = c->tab.t.lr_denom;
	if(pr_phase) memcpy(pr_phase, c->tab.t.pr_phase, 64);
	return VDL2GPU_OK;
}

extern "C" int vdl2gpu_read_dec(vdl2gpu_ctx *c, float *out, size_t cap_floats, uint32_t *n_dec) {
	if(!c || !out || !n_dec) return VDL2GPU_EINVAL;
	CU(cudaSetDevice(c->device));
	CU(cudaStreamSynchronize(c->stream));
	CU(cudaStreamSynchronize(c->s_back));
	*n_dec = c->last_n_dec;
	if((size_t)c->last_n_dec * c->n_ch * 2 > cap_floats) return VDL2GPU_ETOOBIG;
	if(c->last_n_dec == 0) return VDL2GPU_OK;
	if(c->lanes == 32) {
		CU(cudaMemcpy2D(out, (size_t)c->n_ch * sizeof(float2), c->d_dec3[(c->chunk_seq + 2) % 3u], (size_t)c->n_chp * sizeof(float2),
				(size_t)c->n_ch * sizeof(float2), c->last_n_dec, cudaMemcpyDeviceToHost));
	} else {
		std::vector<float2> tmp((size_t)c->last_n_dec * c->n_chp);
		CU(cudaMemcpy(tmp.data(), c->d_dec3[(c->chunk_seq + 2) % 3u], tmp.size() * sizeof(float2), cudaMemcpyDeviceToHost));
		for(uint32_t m = 0; m < c->last_n_dec; m++)
			for(uint32_t ch = 0; ch < c->n_ch; ch++) {
				const float2 v = tmp[(size_t)m * c->n_chp + slot_of(ch, c->lanes, c->full_warps)];
				out[((size_t)m * c->n_ch + ch) * 2] = v.x; out[((size_t)m * c->n_ch + ch) * 2 + 1] = v.y;
			}
	}
	return VDL2GPU_OK;
}

extern "C" int vdl2gpu_read_events(vdl2gpu_ctx *c, vdl2gpu_event *out, uint32_t cap) {
	if(!c || !out) return VDL2GPU_EINVAL;
	if(!(c->cfg.flags & VDL2GPU_FLAG_TRACE)) return 0;
	CU(cudaSetDevice(c->device));
	CU(cudaStreamSynchronize(c->stream));
	CU(cudaStreamSynchronize(c->s_back));
	vdl2_queue_ctl ctl;
	CU(cudaMemcpy(&ctl, c->d_ctl, sizeof(ctl), cudaMemcpyDeviceToHost));
	uint32_t total = std::min(ctl.n_events, c->event_cap);
	uint32_t n = total > c->events_read ? total - c->events_read : 0;
	if(n > cap) n = cap;
	if(n) CU(cudaMemcpy(out, (const vdl2gpu_event *)c->d_events + c->events_read, (size_t)n * sizeof(vdl2gpu_event), cudaMemcpyDeviceToHost));
	c->events_read += n;
	if(c->events_read == total) {
		/* drained: the buffer is not a ring, so start it over (nothing is running: both streams were synchronised above).
		 * Events the kernels could not store because it was full are counted and reported once the stored ones are out. */
		if(ctl.n_events > c->event_cap) c->events_dropped += ctl.n_events - c->event_cap;
		if(ctl.n_events) {
			const uint32_t zero = 0;
			CU(cudaMemcpy(reinterpret_cast<uint8_t *>(c->d_ctl) + offsetof(vdl2_queue_ctl, n_events), &zero, sizeof(zero), cudaMemcpyHostToDevice));
			c->events_read = 0;
		}
	}
	if(n == 0 && c->events_dropped) {
		snprintf(g_last_error, sizeof(g_last_error), "trace buffer overflow: %llu events were not recorded (drain more often)", (unsigned long long)c->events_dropped);
		c->events_dropped = 0;
		return VDL2GPU_EOVERFLOW;
	}
	return (int)n;
}

extern "C" int vdl2gpu_enable_timing(vdl2gpu_ctx *c, int on) {
	if(!c) return VDL2GPU_EINVAL;
	c->timing = on != 0;
	if(on && !c->ev_t0) {
		CU(cudaSetDevice(c->device));
		CU(cudaEventCreate(&c->ev_t0));
		CU(cudaEventRecord(c->ev_t0, c->stream));
	}
	return VDL2GPU_OK;
}

/* diagnostic: the per-block scheduling records (VDL2GPU_BLOCK_TRACE=1 at create): 6 x uint64 per record
 * {kernel (1 K1, 2 K2), block, SM id, 0, start ns, end ns}; synchronises; returns the number of records copied */
extern "C" int vdl2gpu_debug_block_trace(vdl2gpu_ctx *c, uint64_t *out, uint32_t cap_records) {
	if(!c || !out) return VDL2GPU_EINVAL;
	if(!c->d_block_trace) return 0;
	CU(cudaSetDevice(c->device));
	CU(cudaDeviceSynchronize());
	uint32_t n = 0;
	CU(cudaMemcpy(&n, &c->d_block_trace->n, 4, cudaMemcpyDeviceToHost));
	n = std::min(std::min(n, c->block_trace_cap), cap_records);
	std::vector<vdl2_block_rec> r(n);
	if(n) CU(cudaMemcpy(r.data(), c->d_block_trace->rec, (size_t)n * sizeof(vdl2_block_rec), cudaMemcpyDeviceToHost));
	for(uint32_t k = 0; k < n; k++) {
		out[6 * k] = r[k].kernel; out[6 * k + 1] = r[k].block; out[6 * k + 2] = r[k].smid; out[6 * k + 3] = 0;
		out[6 * k + 4] = r[k].t_start; out[6 * k + 5] = r[k].t_end;
	}
	return (int)n;
}

extern "C" int vdl2gpu_get_timeline(vdl2gpu_ctx *c, float *out, uint32_t cap_rows) {
	if(!c || !out) return VDL2GPU_EINVAL;
	const uint32_t n = std::min<uint32_t>(cap_rows, (uint32_t)(c->timeline.size() / 8));
	memcpy(out, c->timeline.data(), (size_t)n * 8 * sizeof(float));
	return (int)n;
}

extern "C" int vdl2gpu_get_kernel_ms(vdl2gpu_ctx *c, double ms[5], uint64_t launches[5]) {
	if(!c || !ms) return VDL2GPU_EINVAL;
	for(int k = 0; k < 5; k++) { ms[k] = c->k_ms[k]; if(launches) launches[k] = c->k_launches[k]; }
	return VDL2GPU_OK;
}

/* ------------------------------------------------------------------------------------------------
 * raw launch stubs (device pointers in, device pointers out; no allocation, no synchronisation)
 * ---------------------------------------------------------------------------------------------- */
/* GF tables for the stand-alone RS stub, one copy per device, made on first use on that device */
static vdl2_tables *g_stub_tables[64] = { nullptr };
static std::mutex g_stub_lock;

static int stub_tables(vdl2_tables **out) {
	int dev = 0;
	CU(cudaGetDevice(&dev));
	if(dev < 0 || dev >= 64) return VDL2GPU_EINVAL;
	std::lock_guard<std::mutex> lk(g_stub_lock);
	if(!g_stub_tables[dev]) {
		host_tables *h = new host_tables();
		memset(h, 0, sizeof(*h));
		make_gf(h->t);
		vdl2_tables *d = nullptr;
		cudaError_t e = cudaMalloc(&d, sizeof(vdl2_tables));
		if(e == cudaSuccess) e = cudaMemcpy(d, &h->t, sizeof(vdl2_tables), cudaMemcpyHostToDevice);
		delete h;
		if(e != cudaSuccess) { cudaFree(d); return fail_cuda(e, "RS stub tables", __LINE__); }
		g_stub_tables[dev] = d;
	}
	*out = g_stub_tables[dev];
	return VDL2GPU_OK;
}

extern "C" int vdl2gpu_launch_convert(const void *raw, uint32_t n_pairs, uint32_t sample_fmt, const float *levels256,
		float *samples_out, void *stream) {
	if(!raw || !samples_out || sample_fmt > 1 || (sample_fmt == 0 && !levels256)) return VDL2GPU_EINVAL;
	KL(vdl2_launch_k0(raw, n_pairs, sample_fmt, levels256, samples_out, 1, 0, 0, nullptr, (cudaStream_t)stream));
	return VDL2GPU_OK;
}

extern "C" int vdl2gpu_launch_fcs_crc16(const uint8_t *frames, const uint32_t *offsets, const uint32_t *lens,
		uint32_t n_frames, uint16_t *residues_out, void *stream) {
	if(n_frames && (!frames || !offsets || !lens || !residues_out)) return VDL2GPU_EINVAL;
	KL(vdl2_launch_k4(frames, offsets, lens, n_frames, residues_out, (cudaStream_t)stream));
	return VDL2GPU_OK;
}

extern "C" int vdl2gpu_launch_rs_verify(uint8_t *blocks, const int32_t *fec_octets, uint32_t n_blocks, int32_t *ret_out, void *stream) {
	if(n_blocks && (!blocks || !fec_octets || !ret_out)) return VDL2GPU_EINVAL;
	vdl2_tables *t = nullptr;
	int rc = stub_tables(&t);            /* first call on a device allocates; later calls only launch */
	if(rc) return rc;
	KL(vdl2_launch_rs(blocks, fec_octets, n_blocks, ret_out, t, (cudaStream_t)stream));
	return VDL2GPU_OK;
}

/* K2a on its own: phase_out[i] = (float)atan2((double)im, (double)re), mag_out[i] = hypotf(re, im) of n_elems
 * decimated samples (src/demod.c:232,238,256).  exact_libm = 0: the Ziv-guarded short evaluation the pipeline
 * uses (vdl2_fastmath.cuh); 1: the libdevice routine for every element.  Both give the same floats. */
extern "C" int vdl2gpu_launch_phase_mag(const float *dec, uint32_t n_elems, float *phase_out, float *mag_out, int exact_libm, void *stream) {
	if(n_elems && (!dec || !phase_out || !mag_out)) return VDL2GPU_EINVAL;
	if(n_elems == 0) return VDL2GPU_OK;
	int dev = 0;
	CU(cudaGetDevice(&dev));
	KL(vdl2_kernels_init_device(dev));
	vdl2_k2_params p2;
	memset(&p2, 0, sizeof(p2));
	/* one row of n_elems "channels": K2a is element-wise, the row structure does not matter */
	p2.dec = reinterpret_cast<const float2 *>(dec); p2.n_dec = 1; p2.n_ch = n_elems; p2.n_chp = n_elems; p2.lanes = 32; p2.full_warps = 0xFFFFFFFFu;
	p2.phase = phase_out - (size_t)VDL2_SYNC_BUFLEN * n_elems;       /* the launcher skips the 160 history rows */
	p2.mag = mag_out; p2.k2a_mode = exact_libm ? 0u : 1u;
	KL(vdl2_launch_k2a(&p2, (cudaStream_t)stream));
	return VDL2GPU_OK;
}

/* ---- stage stubs: K1, K2 (+K2a), K3 one at a time, on device memory the caller owns ---- */
struct vdl2gpu_stage {
	vdl2gpu_config cfg;
	std::vector<uint32_t> freqs;
	host_tables tab;
	uint32_t n_ch = 0, n_chp = 0, max_dec = 0, n_slots = 0, event_cap = 0;
	uint32_t decim_cnt = 0;
	uint64_t total_dec = 0;
	uint32_t events_read = 0;
	int k1_variant = 2, k2_variant = 5, k2a_mode = 1;
	vdl2_tables *d_tab = nullptr;
	uint32_t *d_k1 = nullptr, *d_k2 = nullptr, *d_counters = nullptr, *d_ready = nullptr;
	float *d_ring = nullptr, *d_phase = nullptr, *d_mag = nullptr, *d_hist_tmp = nullptr;
	vdl2_burst_slot *d_pool = nullptr;
	int32_t *d_free = nullptr;
	vdl2_queue_ctl *d_ctl = nullptr;
	void *d_events = nullptr;
};

static size_t al256(size_t x) { return (x + 255u) & ~(size_t)255u; }

struct stage_layout {
	size_t tab, k1, k2, counters, ring, phase, mag, hist, pool, free_list, ready, ctl, events, total;
};

static stage_layout stage_layout_of(uint32_t n_ch, uint32_t max_dec, uint32_t event_cap) {
	const size_t n_chp = (n_ch + 31u) & ~31u, n_slots = std::max(256u, 3u * n_ch);
	stage_layout L;
	size_t o = 0;
	L.tab = o; o += al256(sizeof(vdl2_tables));
	L.k1 = o; o += al256((size_t)K1_NFIELDS * n_chp * 4);
	L.k2 = o; o += al256((size_t)K2_NFIELDS * n_chp * 4);
	L.counters = o; o += al256((size_t)VDL2_NUM_COUNTERS * n_chp * 4);
	L.ring = o; o += al256((size_t)VDL2_SYNC_BUFLEN * n_chp * 4);
	L.phase = o; o += al256((size_t)(max_dec + VDL2_SYNC_BUFLEN) * n_chp * 4);
	L.mag = o; o += al256((size_t)max_dec * n_chp * 4);
	L.hist = o; o += al256((size_t)VDL2_SYNC_BUFLEN * n_chp * 4);
	L.pool = o; o += al256(n_slots * sizeof(vdl2_burst_slot));
	L.free_list = o; o += al256(n_slots * 4);
	L.ready = o; o += al256(n_slots * 4);
	L.ctl = o; o += al256(sizeof(vdl2_queue_ctl));
	L.events = o; o += al256((size_t)event_cap * sizeof(vdl2gpu_event));
	L.total = o;
	return L;
}

static uint32_t stage_event_cap(uint32_t flags) { return (flags & VDL2GPU_FLAG_TRACE) ? (1u << 18) : 1u; }

extern "C" size_t vdl2gpu_stage_device_bytes(uint32_t n_channels, uint32_t max_dec, uint32_t flags) {
	return stage_layout_of(n_channels, max_dec, stage_event_cap(flags)).total;
}

extern "C" uint32_t vdl2gpu_stage_row_stride(uint32_t n_channels) { return (n_channels + 31u) & ~31u; }

/* initial per-channel state: vdl2_channel_init + demod_reset (src/demod.c:205-220,379-392), process_samples locals
 * (src/demod.c:289-298); shared by the batch context and the stage stubs.  centers: the centre frequency of every
 * channel's stream (receiver farm), NULL = cfg.centerfreq for all */
static void initial_state(const vdl2gpu_config &cfg, const uint32_t *freqs, const uint32_t *centers, uint32_t n_ch, uint32_t n_chp, uint32_t lanes,
		uint32_t full_warps, std::vector<uint32_t> &k1, std::vector<uint32_t> &k2) {
	k1.assign((size_t)K1_NFIELDS * n_chp, 0u); k2.assign((size_t)K2_NFIELDS * n_chp, 0u);
	auto fbits = [](float f) { uint32_t u; memcpy(&u, &f, 4); return u; };
	for(uint32_t chan = 0; chan < n_ch; chan++) {
		const uint32_t ch = slot_of(chan, lanes, full_warps);          /* index into the per-channel planes */
		/* a channel on the centre frequency skips the mixer in the reference (src/demod.c:312); with a zero
		 * phase step the table gives cos = 1, sin = 0 and the products are exact, so no branch is needed */
		const uint32_t centre = centers ? centers[chan] : cfg.centerfreq;
		k1[(size_t)K1_DPHI * n_chp + ch] = (centre != freqs[chan]) ? dphi_for(centre, freqs[chan], cfg.sample_rate) : 0u;
		k2[(size_t)K2_MAG_NF * n_chp + ch] = fbits(2.0f);
		k2[(size_t)K2_PHERR1 * n_chp + ch] = fbits(1000.f);
		k2[(size_t)K2_PHERR2 * n_chp + ch] = fbits(1000.f);
		k2[(size_t)K2_STATE * n_chp + ch] = VDL2_DEC_HEADER << VDL2_DEC_SHIFT;
		k2[(size_t)K2_NEED_BITS * n_chp + ch] = VDL2_HEADER_LEN;
		k2[(size_t)K2_SLOT * n_chp + ch] = (uint32_t)-1;
		k2[(size_t)K2_FREQ * n_chp + ch] = freqs[chan];
		k2[(size_t)K2_PURE_RUN * n_chp + ch] = 0x40000000u;      /* VDL2_PURE_SATURATED: ring of zeros == history of zeros */
	}
}

extern "C" int vdl2gpu_stage_create(const vdl2gpu_config *cfg, uint32_t max_dec, void *device_mem, size_t device_bytes, vdl2gpu_stage **out) {
	if(!cfg || !out || !device_mem || !cfg->freqs || cfg->n_channels == 0 || cfg->oversample == 0 || max_dec == 0
			|| cfg->sample_rate != (uint32_t)VDL2_SYMBOL_RATE * VDL2_SPS * cfg->oversample) return VDL2GPU_EINVAL;
	const uint32_t ecap = stage_event_cap(cfg->flags);
	const stage_layout L = stage_layout_of(cfg->n_channels, max_dec, ecap);
	if(device_bytes < L.total || ((uintptr_t)device_mem & 255u)) return VDL2GPU_EINVAL;
	int dev = 0;
	CU(cudaGetDevice(&dev));
	KL(vdl2_kernels_init_device(dev));
	vdl2gpu_stage *st = new vdl2gpu_stage();
	st->cfg = *cfg;
	st->freqs.assign(cfg->freqs, cfg->freqs + cfg->n_channels);
	st->cfg.freqs = st->freqs.data();
	st->n_ch = cfg->n_channels; st->n_chp = (st->n_ch + 31u) & ~31u; st->max_dec = max_dec;
	st->n_slots = std::max(256u, 3u * st->n_ch); st->event_cap = ecap;
	const char *e;
	if((e = getenv("VDL2GPU_K1_VARIANT"))) st->k1_variant = atoi(e);
	if((e = getenv("VDL2GPU_K2_VARIANT"))) st->k2_variant = atoi(e);
	if((e = getenv("VDL2GPU_K2A"))) st->k2a_mode = atoi(e);
	make_tables(st->tab, cfg->sample_rate);
	uint8_t *b = static_cast<uint8_t *>(device_mem);
	st->d_tab = reinterpret_cast<vdl2_tables *>(b + L.tab); st->d_k1 = reinterpret_cast<uint32_t *>(b + L.k1);
	st->d_k2 = reinterpret_cast<uint32_t *>(b + L.k2); st->d_counters = reinterpret_cast<uint32_t *>(b + L.counters);
	st->d_ring = reinterpret_cast<float *>(b + L.ring); st->d_phase = reinterpret_cast<float *>(b + L.phase);
	st->d_mag = reinterpret_cast<float *>(b + L.mag); st->d_hist_tmp = reinterpret_cast<float *>(b + L.hist);
	st->d_pool = reinterpret_cast<vdl2_burst_slot *>(b + L.pool); st->d_free = reinterpret_cast<int32_t *>(b + L.free_list);
	st->d_ready = reinterpret_cast<uint32_t *>(b + L.ready); st->d_ctl = reinterpret_cast<vdl2_queue_ctl *>(b + L.ctl);
	st->d_events = b + L.events;
	std::vector<uint32_t> k1, k2;
	initial_state(st->cfg, st->freqs.data(), nullptr, st->n_ch, st->n_chp, 32u, 0xFFFFFFFFu, k1, k2);
	std::vector<int32_t> fl(st->n_slots);
	for(uint32_t i = 0; i < st->n_slots; i++) fl[i] = (int32_t)i;
	vdl2_queue_ctl ctl;
	memset(&ctl, 0, sizeof(ctl));
	ctl.free_top = (int32_t)st->n_slots;
	cudaError_t ce = cudaMemset(device_mem, 0, L.total);
	if(ce == cudaSuccess) ce = cudaMemcpy(st->d_tab, &st->tab.t, sizeof(vdl2_tables), cudaMemcpyHostToDevice);
	if(ce == cudaSuccess) ce = cudaMemcpy(st->d_k1, k1.data(), k1.size() * 4, cudaMemcpyHostToDevice);
	if(ce == cudaSuccess) ce = cudaMemcpy(st->d_k2, k2.data(), k2.size() * 4, cudaMemcpyHostToDevice);
	if(ce == cudaSuccess) ce = cudaMemcpy(st->d_free, fl.data(), fl.size() * 4, cudaMemcpyHostToDevice);
	if(ce == cudaSuccess) ce = cudaMemcpy(st->d_ctl, &ctl, sizeof(ctl), cudaMemcpyHostToDevice);
	if(ce != cudaSuccess) { delete st; return fail_cuda(ce, "vdl2gpu_stage_create", __LINE__); }
	*out = st;
	return VDL2GPU_OK;
}

extern "C" int vdl2gpu_stage_destroy(vdl2gpu_stage *st) { delete st; return VDL2GPU_OK; }

extern "C" int vdl2gpu_stage_levels(vdl2gpu_stage *st, const float **levels256_dev) {
	if(!st || !levels256_dev) return VDL2GPU_EINVAL;
	*levels256_dev = st->d_tab->levels;
	return VDL2GPU_OK;
}

/* K1 == the per-sample loop of process_samples (src/demod.c:288-337) for every channel of the stage */
extern "C" int vdl2gpu_launch_mix_iir_decimate(vdl2gpu_stage *st, const float *samples, uint32_t n_pairs, float *dec_out,
		uint32_t *n_dec_out, void *stream) {
	if(!st || (n_pairs && (!samples || !dec_out))) return VDL2GPU_EINVAL;
	const uint32_t os = st->cfg.oversample;
	const uint32_t n_dec = (st->decim_cnt + n_pairs) / os;
	if(n_dec > st->max_dec) return VDL2GPU_ETOOBIG;
	vdl2_k1_params p1;
	memset(&p1, 0, sizeof(p1));
	p1.samples = reinterpret_cast<const float2 *>(samples); p1.n_pairs = n_pairs; p1.oversample = os; p1.cnt0 = st->decim_cnt;
	p1.n_ch = st->n_ch; p1.n_chp = st->n_chp; p1.lanes = 32; p1.full_warps = 0xFFFFFFFFu; p1.dec = reinterpret_cast<float2 *>(dec_out); p1.state = st->d_k1;
	p1.lut = reinterpret_cast<const float4 *>(st->d_tab->lut);
	p1.a0 = st->tab.t.A[0]; p1.a1 = st->tab.t.A[1]; p1.a2 = st->tab.t.A[2]; p1.b1 = st->tab.t.B[1]; p1.b2 = st->tab.t.B[2];
	p1.one = 1.0f; p1.neg_one = -1.0f; p1.two = 2.0f;
	KL(vdl2_launch_k1(&p1, (st->cfg.flags & VDL2GPU_FLAG_K1_SCALAR) ? 1 : 0, st->k1_variant, (cudaStream_t)stream));
	st->decim_cnt = (st->decim_cnt + n_pairs) % os;
	if(n_dec_out) *n_dec_out = n_dec;
	return VDL2GPU_OK;
}

/* K2a + K2 == demod() (src/demod.c:222-286) + the header part of decode_vdl2_burst (src/decode.c:198-258) over n_dec
 * decimated samples of every channel; completed bursts queue up for vdl2gpu_launch_burst_fec */
extern "C" int vdl2gpu_launch_sync_slice(vdl2gpu_stage *st, const float *dec, uint32_t n_dec, void *stream) {
	if(!st || (n_dec && !dec)) return VDL2GPU_EINVAL;
	if(n_dec > st->max_dec) return VDL2GPU_ETOOBIG;
	if(n_dec == 0) return VDL2GPU_OK;
	vdl2_k2_params p2;
	memset(&p2, 0, sizeof(p2));
	p2.dec = reinterpret_cast<const float2 *>(dec); p2.phase = st->d_phase; p2.mag = st->d_mag; p2.hist_tmp = st->d_hist_tmp;
	p2.n_dec = n_dec; p2.n_ch = st->n_ch; p2.n_chp = st->n_chp; p2.lanes = 32; p2.full_warps = 0xFFFFFFFFu; p2.dec_base = st->total_dec;
	p2.state = st->d_k2; p2.ring = st->d_ring; p2.tables = st->d_tab; p2.max_ppm = st->cfg.max_ppm; p2.s27 = st->tab.s27;
	p2.pool = st->d_pool; p2.free_list = st->d_free; p2.ready = st->d_ready; p2.ctl = st->d_ctl;
	p2.events = st->d_events; p2.event_cap = st->event_cap; p2.trace = (st->cfg.flags & VDL2GPU_FLAG_TRACE) ? 1u : 0u;
	p2.variant = (uint32_t)st->k2_variant; p2.k2a_mode = (uint32_t)st->k2a_mode;
	KL(vdl2_launch_k2a(&p2, (cudaStream_t)stream));
	KL(vdl2_launch_k2(&p2, (cudaStream_t)stream));
	KL(vdl2_launch_copy_hist(&p2, (cudaStream_t)stream));
	st->total_dec += n_dec;
	return VDL2GPU_OK;
}

/* K3 (+K4) == the data part of decode_vdl2_burst (src/decode.c:259-380) for every queued burst.  `region` receives a
 * vdl2_out_header followed by the burst records (device memory or mapped pinned host memory, 16-byte aligned);
 * vdl2gpu_parse_records turns a host copy of it into frames. */
extern "C" int vdl2gpu_launch_burst_fec(vdl2gpu_stage *st, uint8_t *region, uint32_t region_bytes, void *stream) {
	if(!st || !region || region_bytes < sizeof(vdl2_out_header) + 256u || ((uintptr_t)region & 15u)) return VDL2GPU_EINVAL;
	vdl2_k3_params p3;
	memset(&p3, 0, sizeof(p3));
	p3.pool = st->d_pool; p3.free_list = st->d_free; p3.ready = st->d_ready; p3.ctl = st->d_ctl; p3.tables = st->d_tab;
	p3.out = region; p3.out_cap = region_bytes - (uint32_t)sizeof(vdl2_out_header); p3.n_chp = st->n_chp; p3.counters = st->d_counters;
	KL(vdl2_launch_k3(&p3, K3_GRID, (cudaStream_t)stream));
	return VDL2GPU_OK;
}

extern "C" int vdl2gpu_stage_read_events(vdl2gpu_stage *st, vdl2gpu_event *out, uint32_t cap) {
	if(!st || !out) return VDL2GPU_EINVAL;
	if(!(st->cfg.flags & VDL2GPU_FLAG_TRACE)) return 0;
	CU(cudaDeviceSynchronize());
	vdl2_queue_ctl ctl;
	CU(cudaMemcpy(&ctl, st->d_ctl, sizeof(ctl), cudaMemcpyDeviceToHost));
	uint32_t total = std::min(ctl.n_events, st->event_cap);
	uint32_t n = total > st->events_read ? total - st->events_read : 0;
	if(n > cap) n = cap;
	if(n) CU(cudaMemcpy(out, (const vdl2gpu_event *)st->d_events + st->events_read, (size_t)n * sizeof(vdl2gpu_event), cudaMemcpyDeviceToHost));
	st->events_read += n;
	return (int)n;
}

extern "C" int vdl2gpu_parse_records(const uint8_t *region_host, uint32_t region_bytes, uint32_t decimated_rate,
		vdl2gpu_frame_cb cb, void *user) {
	if(!region_host || region_bytes < sizeof(vdl2_out_header)) return VDL2GPU_EINVAL;
	std::vector<pending_frame> pending;
	vdl2gpu_stats stats;
	memset(&stats, 0, sizeof(stats));
	struct timeval now;
	gettimeofday(&now, NULL);
	parse_region(region_host, region_bytes - (uint32_t)sizeof(vdl2_out_header), (double)decimated_rate, now, 0, 0, pending, stats);
	const uint8_t *base = region_host + sizeof(vdl2_out_header);
	for(auto &pf : pending) {
		pf.f.data = base + pf.offset;
		if(cb) cb(&pf.f, user);
	}
	if(stats.pool_overflows || stats.out_overflows) return VDL2GPU_EOVERFLOW;
	return (int)pending.size();
}
