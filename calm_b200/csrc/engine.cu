// engine.cu -- host side of libcalm_b200.so: the reference's CUDA backend boundary
// (upload_cuda / prepare_cuda / forward_cuda / perf_cuda, reference src/run.c:22-25 and
// src/infer.cu:69-131, 651-801) implemented over the sm_100a kernels in stages.cuh.
//
// The per-token kernel sequence is captured once into CUDA graphs and replayed; per-token scalars
// live in a device-resident TokenParams record that the host (forward_cuda) or the device
// (greedy decode) rewrites between replays.

#include "../../include/calm_b200.h"

#include <dlfcn.h>
#include <math.h>
#include <string.h>

#include <vector>

#include "stages.cuh"
#include "attn.cuh"
#include "ring.cuh"
#include "prefill.cuh"

namespace {

#define MAX_STAMPS (2 + 5 * MAX_LAYERS)
#define TP_MAX_CAND 2048 // greedy candidates (classifier CTAs) per rank in the tensor-parallel gather area
enum Stage { ST_EMBED, ST_QKV, ST_ATTN, ST_WO, ST_FFN_UP, ST_FFN_DOWN, ST_OUTPUT, ST_COUNT };
const char* const kStageNames[ST_COUNT] = {"embed", "matmul_qkv", "attention", "matmul_attn", "matmul_ffn_up", "matmul_ffn_down", "output"};

struct Engine {
	bool ready = false;
	int device = -1;
	int sms = 0;
	cudaStream_t stream = nullptr;
	struct Config cfg;
	struct Weights w;
	int kvbits = 16;
	int nact = 1;
	int q_dim = 0, kv_dim = 0, kv_mul = 1;

	// device buffers
	float *x = nullptr, *xb = nullptr, *q = nullptr, *att = nullptr, *hb = nullptr, *logits_dev = nullptr;
	float* logits_host = nullptr; // pinned + mapped
	void *kc = nullptr, *vc = nullptr;
	float* rope_freq = nullptr;
	float2* rope_cs = nullptr; // (cos, sin) of the current token's RoPE angles, written by k_embed
	unsigned long long* attn_cells = nullptr; // k_attn2's slice fold: {value, epoch} cells
	int* dev_err = nullptr;                   // mapped host word: watchdog code of an in-kernel wait that gave up
	float* attn_partial = nullptr;
	unsigned* attn_counter = nullptr;
	MoeSel* moe_sel = nullptr;
	TokenParams* tp = nullptr;
	float* cand_val = nullptr;
	int* cand_idx = nullptr;
	int* out_tokens = nullptr;
	int out_tokens_cap = 0;
	int* last_token = nullptr; // pinned + mapped
	int ncand = 0;

	// attention launch shape
	int attn_hg = 1, attn_qgroups = 1, attn_nsplit = 1, attn_lpp = 1;
	// TMA-ring matvec kernels (ring.cuh): slots per warp / CTAs per SM for FFN-up and for wo / w2; u = 512-byte units per row and chunk (0: not used)
	int ring_up_ns = 2, ring_up_cps = 2, ring_res_ns = 2, ring_res_warps = 16; // measured: 16 consuming warps per SM are needed (profiles/r02_sweep_ring_*.jsonl)
	int ring_up_u = 0, ring_wo_u = 0, ring_down_u = 0, ring_wo_s = 1, ring_down_s = 1;
	int grid_up_ring = 0, grid_wo_ring = 0, grid_down_ring = 0;
	size_t smem_up_ring = 0, smem_wo_ring = 0, smem_down_ring = 0;
	bool attn2_cluster = false; // ... with the CTAs of a unit as one thread-block cluster (slices folded through distributed shared memory)
	bool attn2 = false; // k_attn2 (attn.cuh): KV slice requested into shared memory ahead of the dependency wait
	bool attn_mma = false; // k_attn_mma (attn.cuh): the same, scores and values on mma.sync (head_dim 128, 4 query heads per kv head)
	int attn_nbmax = 0;
	size_t attn2_smem = 0, attn_mma_smem = 0;

	// launch plan (grid sizes / dynamic shared memory), fixed at prepare time
	int grid_qkv = 0, grid_wo = 0, grid_up = 0, grid_down = 0, grid_out = 0;
	size_t smem_dim = 0, smem_qdim = 0, smem_hidden = 0;
	int cur_kv_len = 0; // host copy, for the perf table only
	int cur_pos = 0;
	int attn_nsplit_cap = 1 << 30;

	// L2 prefetch schedule (common.cuh Prefetch): what each stage requests for the stages after it.  Bytes, or flags.
	// Measured (profiles/r02_sweep_l2_prefetch_schedule.jsonl): no setting beats "off" -- the stage kernels are not waiting for
	// DRAM behind their boundaries, and requests for later stages only compete with the running one -- so the default is off;
	// CALM_B200_PF keeps the experiment reproducible.
	bool pf_kv = false;           // k_qkv / w2 request the KV prefix the next attention kernel reads
	bool pf_attn_wo = false;      // k_attn requests wo
	size_t pf_attn_up = 0;        // ... and this much of w1 + w3
	size_t pf_wo_up = 0;          // wo requests this much more of w1 + w3
	size_t pf_up_down = 0;        // k_ffn_up requests this much of w2
	bool pf_down_qkv = false;     // w2 requests the next layer's wq / wk / wv


	// tensor parallelism (staged engine): this process owns 1/tp_world of the heads and of the FFN rows
	int tp_rank = 0, tp_world = 1;
	void* tp_comm = nullptr;         // ncclComm_t
	float* xpart = nullptr;          // partial of wo / w2 before the all-reduce (NCCL path)
	bool tp_fused = false;           // wo / w2 sum their partials inside k_matres over peer memory (stages.cuh TpExchange)
	size_t up_expert_stride = 0;     // 16-byte vectors between experts of w1 / w3 once the rows are sharded
	int out_row0 = 0, out_row1 = 0;  // classifier rows of this rank (vocabulary split; the whole vocabulary without tensor parallelism)
	size_t tp_off_logits = 0, tp_off_cval = 0, tp_off_cidx = 0, tp_off_flags = 0; // byte offsets of the gather area inside every rank's exchange area
	void* tp_area = nullptr;         // this rank's exchange area: {partial, epoch} cells, then the logits gather area
	void* tp_peer[TP_MAX_WORLD] = {}; // every rank's area as mapped here (own entry == tp_area)
	int* tp_err = nullptr;           // mapped host word for the exchange watchdog
	std::vector<void*> tp_owned;     // shard copies made by prepare_cuda (wo / w2 column slices, packed biases)


	// one graph per call mode: 0 KV only, 1 logits to host, 2 greedy loop, 3 logits + argmax, 4 min-p sampling loop;
	// [1][mode] = the same token with stage stamps (perf_cuda)
	cudaGraphExec_t graph[2][5] = {};
	int graph_launches[2][5] = {};
	// device-side min-p sampler (stages.cuh k_sample_*)
	SampleState* sample_state = nullptr;
	int sample_chunks = 0;
	int* sample_count = nullptr;
	float* sample_csum = nullptr;
	int* sample_idx = nullptr;
	float* sample_prob = nullptr;
	bool use_graph = true;
	bool use_pdl = true;
	int carveout = -1;   // cudaFuncAttributePreferredSharedMemoryCarveout applied to every kernel of the token, or -1

	// profiling (perf_cuda): in-kernel %globaltimer stamps per launch of the production graph (stages.cuh stamp_begin/end)
	bool perf = false;
	bool debug = false;
	unsigned long long* stamps = nullptr;    // device [MAX_STAMPS][2]: {min start, max end} of each launch of the current token
	unsigned long long* stamp_acc = nullptr; // device [MAX_STAMPS + 2]: summed durations; [MAX_STAMPS] token span, [MAX_STAMPS + 1] tokens
	int n_stamps = 0;                        // launches with a slot in the current token
	int stamp_stage[MAX_STAMPS] = {};        // launch -> Stage
	double stamp_bytes[MAX_STAMPS] = {};     // algorithmic bytes of that launch (KV bytes use the host copy of kv_len)
	double stage_ms[ST_COUNT] = {};
	double stage_bytes[ST_COUNT] = {};
	long stage_launches[ST_COUNT] = {};
	double token_span_ms = 0;
	int perf_runs = 0;
	cudaEvent_t timer[2] = {nullptr, nullptr};
};

Engine g;

// batched prompt pass (prefill.cuh): buffers for up to `cap` tokens, allocated on first use
struct Prefill {
	int cap = 0;
	float *X = nullptr, *Q = nullptr;
	__half *Nhi = nullptr, *Nlo = nullptr, *Ahi = nullptr, *Alo = nullptr, *Hhi = nullptr, *Hlo = nullptr;
	float2* rope = nullptr;
	int* tokens = nullptr;
	CUtensorMap tmN[2], tmA[2], tmH[2]; // (hi, lo) views of the three activation matrices the GEMMs read
};
Prefill pf;
int g_device_override = -1;
uint64_t g_launches = 0;

void select_device() {
	if (g.device >= 0) return;
	int dev = g_device_override;
	if (dev < 0) {
		const char* e = getenv("CALM_B200_DEVICE");
		dev = e ? atoi(e) : 0;
	}
	int count = 0;
	cudaError_t err = cudaGetDeviceCount(&count);
	if (err != cudaSuccess || count == 0) CALM_FATAL("no CUDA device available (%s); this backend has no CPU fallback", cudaGetErrorString(err));
	if (dev >= count) CALM_FATAL("device %d requested but only %d present", dev, count);
	CUDA_CHECK(cudaSetDevice(dev));
	g.device = dev;
}

void* dev_alloc(size_t bytes) {
	void* p = nullptr;
	CUDA_CHECK(cudaMalloc(&p, bytes ? bytes : 16));
	return p;
}

// opt in to more than 48 KB of dynamic shared memory (once per kernel, with the LARGEST size any launch will use, outside stream capture)
template <typename F>
void smem_optin(F kernel, size_t smem) {
	if (smem > 227 * 1024) CALM_FATAL("kernel needs %zu bytes of shared memory per CTA (limit 227 KB)", smem);
	if (smem > 48 * 1024) CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
}

template <typename F>
int max_ctas(F kernel, int block, size_t smem) {
	int per_sm = 0;
	CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, block, smem));
	if (per_sm < 1) CALM_FATAL("kernel does not fit on an SM (block %d, %zu bytes of shared memory)", block, smem);
	return per_sm * g.sms;
}

int imin(int a, int b) { return a < b ? a : b; }
int cdiv(int a, int b) { return (a + b - 1) / b; }
// grid for `units` equal CTA-sized work items when at most `cap` CTAs are resident: every CTA gets the same
// number of rounds (a 3.03-rounds grid costs 4 rounds on some SMs and idles the rest)
int balanced_grid(int units, int cap) {
	if (units <= cap) return units < 1 ? 1 : units;
	return cdiv(units, cdiv(units, cap));
}

template <int DBITS>
size_t xs_bytes(int n) {
	return (size_t)(32 + xs_all_floats<DBITS>(n)) * sizeof(float);
}


// ---------------------------------------------------------------------------------------------
// NCCL, bound at run time (the library stays loadable and linkable without it; only tensor-parallel runs need it)

struct NcclApi {
	void* lib = nullptr;
	int (*GetUniqueId)(void*) = nullptr;
	int (*CommInitRank)(void**, int, /* ncclUniqueId by value: 128 bytes */ struct Id128, int) = nullptr;
	int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
	int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
	int (*CommDestroy)(void*) = nullptr;
	const char* (*GetErrorString)(int) = nullptr;
};
struct Id128 {
	char bytes[128];
};
NcclApi g_nccl;
Id128 g_tp_id;
bool g_tp_pending = false;
int g_tp_rank = 0, g_tp_world = 1;

void nccl_load() {
	if (g_nccl.lib) return;
	const char* names[] = {"libnccl.so.2", "libnccl.so"};
	for (const char* n : names)
		if ((g_nccl.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL))) break;
	if (!g_nccl.lib) CALM_FATAL("tensor parallelism needs NCCL (libnccl.so.2): %s", dlerror());
	g_nccl.GetUniqueId = (int (*)(void*))dlsym(g_nccl.lib, "ncclGetUniqueId");
	g_nccl.CommInitRank = (int (*)(void**, int, Id128, int))dlsym(g_nccl.lib, "ncclCommInitRank");
	g_nccl.AllReduce = (int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t))dlsym(g_nccl.lib, "ncclAllReduce");
	g_nccl.AllGather = (int (*)(const void*, void*, size_t, int, void*, cudaStream_t))dlsym(g_nccl.lib, "ncclAllGather");
	g_nccl.CommDestroy = (int (*)(void*))dlsym(g_nccl.lib, "ncclCommDestroy");
	g_nccl.GetErrorString = (const char* (*)(int))dlsym(g_nccl.lib, "ncclGetErrorString");
	if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllReduce || !g_nccl.AllGather || !g_nccl.CommDestroy) CALM_FATAL("libnccl lacks the expected entry points");
}

#define NCCL_CHECK(x)                                                                                              \
	do {                                                                                                           \
		int r_ = (x);                                                                                              \
		if (r_ != 0) CALM_FATAL("NCCL error %d (%s) at %s:%d", r_, g_nccl.GetErrorString ? g_nccl.GetErrorString(r_) : "?", __FILE__, __LINE__); \
	} while (0)

// sum over ranks of a float vector, in stream order (captured into the CUDA graph like any kernel)
void tp_allreduce(float* buf, size_t count) {
	NCCL_CHECK(g_nccl.AllReduce(buf, buf, count, /*ncclFloat32*/ 7, /*ncclSum*/ 0, g.tp_comm, g.stream));
}

// Exchange areas for the fused matvec -> all-reduce (stages.cuh TpExchange): one cudaMalloc per rank, mapped into
// every peer with CUDA IPC (one process per GPU); the 64-byte handles travel through an NCCL all-gather.  Falls
// back to ncclAllReduce + k_addvec when peer mapping is unavailable on ANY rank (the ranks agree via an all-reduce).
void tp_setup_exchange() {
	const int W = g.tp_world, dim = g.cfg.dim;
	// cell[slot][src][row] | logits[vocab] | cand_val[W][TP_MAX_CAND] | cand_idx[W][TP_MAX_CAND] | flags[W]
	auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
	g.tp_off_logits = up((size_t)2 * W * dim * sizeof(uint2));
	g.tp_off_cval = g.tp_off_logits + up((size_t)g.cfg.vocab_size * sizeof(float));
	g.tp_off_cidx = g.tp_off_cval + up((size_t)W * TP_MAX_CAND * sizeof(float));
	g.tp_off_flags = g.tp_off_cidx + up((size_t)W * TP_MAX_CAND * sizeof(int));
	const size_t bytes = g.tp_off_flags + up((size_t)W * sizeof(unsigned));
	bool ok = W <= TP_MAX_WORLD && !(getenv("CALM_B200_TP_FUSED") && atoi(getenv("CALM_B200_TP_FUSED")) == 0);
	g.tp_area = dev_alloc(bytes);
	CUDA_CHECK(cudaMemset(g.tp_area, 0, bytes));
	cudaIpcMemHandle_t mine;
	if (cudaIpcGetMemHandle(&mine, g.tp_area) != cudaSuccess) ok = false, (void)cudaGetLastError();
	static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
	char* hdev = (char*)dev_alloc((size_t)W * 64 + sizeof(int));
	CUDA_CHECK(cudaMemcpy(hdev + (size_t)g.tp_rank * 64, &mine, 64, cudaMemcpyHostToDevice));
	NCCL_CHECK(g_nccl.AllGather(hdev + (size_t)g.tp_rank * 64, hdev, 64, /*ncclInt8*/ 0, g.tp_comm, g.stream));
	CUDA_CHECK(cudaStreamSynchronize(g.stream));
	std::vector<cudaIpcMemHandle_t> all(W);
	CUDA_CHECK(cudaMemcpy(all.data(), hdev, (size_t)W * 64, cudaMemcpyDeviceToHost));
	for (int p = 0; p < W && ok; ++p) {
		if (p == g.tp_rank) {
			g.tp_peer[p] = g.tp_area;
			continue;
		}
		if (cudaIpcOpenMemHandle(&g.tp_peer[p], all[p], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
			fprintf(stderr, "calm_b200: rank %d cannot map rank %d's exchange area (%s); using ncclAllReduce\n", g.tp_rank, p, cudaGetErrorString(cudaGetLastError()));
			g.tp_peer[p] = nullptr;
			ok = false;
		}
	}
	// every rank must take the same path: min over ranks of `ok`
	int* okdev = (int*)(hdev + (size_t)W * 64);
	int okh = ok ? 1 : 0;
	CUDA_CHECK(cudaMemcpy(okdev, &okh, sizeof(int), cudaMemcpyHostToDevice));
	NCCL_CHECK(g_nccl.AllReduce(okdev, okdev, 1, /*ncclInt32*/ 2, /*ncclMin*/ 3, g.tp_comm, g.stream));
	CUDA_CHECK(cudaStreamSynchronize(g.stream));
	CUDA_CHECK(cudaMemcpy(&okh, okdev, sizeof(int), cudaMemcpyDeviceToHost));
	CUDA_CHECK(cudaFree(hdev));
	g.tp_fused = okh == 1;
	if (g.tp_fused) {
		CUDA_CHECK(cudaHostAlloc((void**)&g.tp_err, sizeof(int), cudaHostAllocMapped));
		*g.tp_err = 0;
	}
}

void tp_fill(TpExchange& t, int idx) {
	t.world = g.tp_world, t.rank = g.tp_rank, t.idx = (unsigned)idx, t.stride = 2u * g.cfg.n_layers, t.tp = g.tp, t.err = g.tp_err;
	for (int p = 0; p < g.tp_world; ++p) t.cell[p] = (uint2*)g.tp_peer[p];
}

// Launch on the library's stream with programmatic stream serialization (PDL), so that consecutive kernels
// of a token overlap their launch latency (the kernels order themselves with griddepcontrol.wait).
// One L1 / shared-memory split for every kernel of the token (env CALM_B200_CARVEOUT = percent of shared memory, unset:
// the driver picks per kernel): kernels whose preferred splits differ cannot be co-resident on an SM, which serialises
// exactly the hand-over that programmatic dependent launch is there to overlap.
void same_carveout(const void* kernel) {
	if (g.carveout < 0) return;
	static std::vector<const void*> done;
	for (const void* k : done)
		if (k == kernel) return;
	done.push_back(kernel);
	CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, g.carveout));
}

template <typename... KArgs, typename... Args>
void launch_pdl(void (*kernel)(KArgs...), int grid, int block, size_t smem, Args... args) {
	same_carveout((const void*)kernel);
	cudaLaunchConfig_t cfg = {};
	cfg.gridDim = dim3(grid), cfg.blockDim = dim3(block), cfg.dynamicSmemBytes = smem, cfg.stream = g.stream;
	cudaLaunchAttribute at[1];
	at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
	at[0].val.programmaticStreamSerializationAllowed = g.use_pdl ? 1 : 0;
	cfg.attrs = at, cfg.numAttrs = 1;
	CUDA_CHECK(cudaLaunchKernelEx(&cfg, kernel, args...));
}

template <typename... KArgs, typename... Args>
void launch_pdl_grid(void (*kernel)(KArgs...), dim3 grid, int block, Args... args) {
	same_carveout((const void*)kernel);
	cudaLaunchConfig_t cfg = {};
	cfg.gridDim = grid, cfg.blockDim = dim3(block), cfg.dynamicSmemBytes = 0, cfg.stream = g.stream;
	cudaLaunchAttribute at[1];
	at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
	at[0].val.programmaticStreamSerializationAllowed = g.use_pdl ? 1 : 0;
	cfg.attrs = at, cfg.numAttrs = 1;
	CUDA_CHECK(cudaLaunchKernelEx(&cfg, kernel, args...));
}

// ---------------------------------------------------------------------------------------------
// one token = this sequence of launches

// A stage launch: hands out the stamp slot when the profiling graph is being built (NULL in the production graph) and,
// under CALM_B200_DEBUG=1, synchronises after the launch to name the stage that faults or hangs.
struct StageScope {
	Stage st;
	unsigned long long* slot = nullptr;
	StageScope(Stage s, double bytes) : st(s) {
		if (g.perf && g.n_stamps < MAX_STAMPS) {
			g.stamp_stage[g.n_stamps] = s, g.stamp_bytes[g.n_stamps] = bytes;
			slot = g.stamps + 2 * (size_t)g.n_stamps++;
		}
	}
	~StageScope() {
		if (g.debug) {
			cudaError_t e = cudaStreamSynchronize(g.stream);
			fprintf(stderr, "calm_b200: stage %s -> %s\n", kStageNames[st], cudaGetErrorName(e));
		}
	}
};

// end of a profiled token: fold the launch stamps into the running sums (one thread per slot)
__global__ void k_stamp_accum(const unsigned long long* stamps, unsigned long long* acc, int n) {
	pdl_enter();
	__shared__ unsigned long long lo[256], hi[256];
	unsigned long long mn = ~0ull, mx = 0;
	for (int i = threadIdx.x; i < n; i += blockDim.x) {
		const unsigned long long b = stamps[2 * i], e = stamps[2 * i + 1];
		if (b != ~0ull && e > b) {
			acc[i] += e - b;
			mn = b < mn ? b : mn, mx = e > mx ? e : mx;
		}
	}
	lo[threadIdx.x] = mn, hi[threadIdx.x] = mx;
	__syncthreads();
	if (threadIdx.x == 0) {
		for (int i = 1; i < (int)blockDim.x; ++i) mn = lo[i] < mn ? lo[i] : mn, mx = hi[i] > mx ? hi[i] : mx;
		if (mx > mn) acc[MAX_STAMPS] += mx - mn;
		acc[MAX_STAMPS + 1] += 1;
	}
}

// shared memory of k_attn<., HG>: the per-warp records of the in-CTA merge, or the coefficient tables of the slice merge
size_t attn_smem(int hg, int head_dim, int nsplit) {
	size_t smem = (size_t)(ATTN_THREADS / 32) * hg * (head_dim + 2) * sizeof(float);
	size_t smem2 = (size_t)(2 * nsplit + 1) * hg * sizeof(float);
	return smem2 > smem ? smem2 : smem;
}

// nl == NULL: only opt in to the shared-memory size (prepare time, outside stream capture; head_dim 256 with 8 query heads
// per kv head needs 66 KB)
template <typename KVT, int HG>
void launch_attn(const AttnArgs& a, int nunits, int* nl) {
	const size_t smem = attn_smem(HG, a.head_dim, a.nsplit);
	if (!nl) {
		smem_optin(k_attn<KVT, HG>, smem);
		return;
	}
	launch_pdl(k_attn<KVT, HG>, nunits * a.nsplit, ATTN_THREADS, smem, a);
	++*nl;
}

template <typename KVT, int HG, int LPP>
void launch_attn2(const AttnArgs& a, int nunits, int* nl) {
	if (!nl) { // prepare time: opt-ins, and whether the cluster form can be scheduled at all
		smem_optin(k_attn2<KVT, HG, LPP, false>, g.attn2_smem);
		{ // the cell fold polls its peers: the whole grid must fit on the device at once
			int per_sm = 0;
			CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_attn2<KVT, HG, LPP, false>, ATTN_THREADS, g.attn2_smem));
			if (per_sm * g.sms < nunits * a.nsplit) g.attn2 = false; // k_attn (global partials, last-CTA fold) has no such requirement
		}
		if (g.attn2_cluster) {
			smem_optin(k_attn2<KVT, HG, LPP, true>, g.attn2_smem);
			if (a.nsplit > 8) CUDA_CHECK(cudaFuncSetAttribute(k_attn2<KVT, HG, LPP, true>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
			cudaLaunchConfig_t cfg = {};
			cfg.gridDim = dim3(nunits * a.nsplit), cfg.blockDim = dim3(ATTN_THREADS), cfg.dynamicSmemBytes = g.attn2_smem;
			cudaLaunchAttribute at[1];
			at[0].id = cudaLaunchAttributeClusterDimension;
			at[0].val.clusterDim.x = a.nsplit, at[0].val.clusterDim.y = 1, at[0].val.clusterDim.z = 1;
			cfg.attrs = at, cfg.numAttrs = 1;
			int nclusters = 0;
			if (cudaOccupancyMaxActiveClusters(&nclusters, k_attn2<KVT, HG, LPP, true>, &cfg) != cudaSuccess || nclusters < 1) {
				(void)cudaGetLastError();
				g.attn2_cluster = false; // e.g. no GPC with nsplit free SMs: fold the slices through global partials instead
			}
		}
		return;
	}
	if (g.attn2_cluster) {
		same_carveout((const void*)k_attn2<KVT, HG, LPP, true>);
		cudaLaunchConfig_t cfg = {};
		cfg.gridDim = dim3(nunits * a.nsplit), cfg.blockDim = dim3(ATTN_THREADS), cfg.dynamicSmemBytes = g.attn2_smem, cfg.stream = g.stream;
		cudaLaunchAttribute at[2];
		at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
		at[0].val.programmaticStreamSerializationAllowed = g.use_pdl ? 1 : 0;
		at[1].id = cudaLaunchAttributeClusterDimension;
		at[1].val.clusterDim.x = a.nsplit, at[1].val.clusterDim.y = 1, at[1].val.clusterDim.z = 1;
		cfg.attrs = at, cfg.numAttrs = 2;
		CUDA_CHECK(cudaLaunchKernelEx(&cfg, k_attn2<KVT, HG, LPP, true>, a));
	} else {
		launch_pdl(k_attn2<KVT, HG, LPP, false>, nunits * a.nsplit, ATTN_THREADS, g.attn2_smem, a);
	}
	++*nl;
}

template <typename KVT>
void launch_attn_mma(const AttnArgs& a, int nunits, int* nl) {
	if (!nl) { // prepare time: opt-in, and the cell fold's co-residency requirement (as k_attn2)
		smem_optin(k_attn_mma<KVT>, g.attn_mma_smem);
		int per_sm = 0;
		CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_attn_mma<KVT>, ATTN_THREADS, g.attn_mma_smem));
		if (per_sm * g.sms < nunits * a.nsplit) g.attn_mma = false;
		return;
	}
	launch_pdl(k_attn_mma<KVT>, nunits * a.nsplit, ATTN_THREADS, g.attn_mma_smem, a);
	++*nl;
}

// shapes k_attn2 is instantiated for: head_dim 128 with 4 or 8 query heads per kv head, head_dim 64 with 2, 4 or 8
bool attn2_shape_ok(int hg, int lpp, int head_dim) {
	return head_dim == lpp * 8 && ((lpp == 16 && (hg == 4 || hg == 8)) || (lpp == 8 && (hg == 2 || hg == 4 || hg == 8)));
}

template <typename KVT>
void dispatch_attn(const AttnArgs& a, int nunits, int* nl) {
	if (g.attn_mma) {
		launch_attn_mma<KVT>(a, nunits, nl);
		if (nl) return; // (at prepare time k_attn2 is set up as well: the co-residency check may have turned k_attn_mma off)
	}
	if (g.attn2) {
		switch (g.attn_lpp * 100 + g.attn_hg) {
		case 1604: launch_attn2<KVT, 4, 16>(a, nunits, nl); return;
		case 1608: launch_attn2<KVT, 8, 16>(a, nunits, nl); return;
		case 802: launch_attn2<KVT, 2, 8>(a, nunits, nl); return;
		case 804: launch_attn2<KVT, 4, 8>(a, nunits, nl); return;
		case 808: launch_attn2<KVT, 8, 8>(a, nunits, nl); return;
		}
	}
	switch (g.attn_hg) {
	case 1: launch_attn<KVT, 1>(a, nunits, nl); break;
	case 2: launch_attn<KVT, 2>(a, nunits, nl); break;
	case 3: launch_attn<KVT, 3>(a, nunits, nl); break;
	case 4: launch_attn<KVT, 4>(a, nunits, nl); break;
	case 5: launch_attn<KVT, 5>(a, nunits, nl); break;
	case 6: launch_attn<KVT, 6>(a, nunits, nl); break;
	case 7: launch_attn<KVT, 7>(a, nunits, nl); break;
	default: launch_attn<KVT, 8>(a, nunits, nl); break;
	}
}

// ring kernels are instantiated for U in {2, 4} (1 KB / 2 KB per row and chunk) and NS in {2, 3, 4}
template <int DBITS, int U, int NS>
void ring_up_launch(const FfnUpArgs& a, bool attr_only) {
	if (attr_only) return smem_optin(k_ffn_up_ring<DBITS, U, NS>, g.smem_up_ring);
	launch_pdl(k_ffn_up_ring<DBITS, U, NS>, g.grid_up_ring, 256, g.smem_up_ring, a);
}
template <int DBITS, int U, int NS>
void ring_res_launch(const MatResArgs& a, int S, int grid, size_t smem, bool attr_only) {
	if (attr_only) return smem_optin(k_matres_ring<DBITS, U, NS>, smem);
	launch_pdl(k_matres_ring<DBITS, U, NS>, grid, g.ring_res_warps * 32, smem, a, S);
}
template <int DBITS>
void ring_up_dispatch(const FfnUpArgs& a, bool attr_only) {
	switch (g.ring_up_u * 10 + g.ring_up_ns) {
	case 22: return ring_up_launch<DBITS, 2, 2>(a, attr_only);
	case 23: return ring_up_launch<DBITS, 2, 3>(a, attr_only);
	case 24: return ring_up_launch<DBITS, 2, 4>(a, attr_only);
	case 42: return ring_up_launch<DBITS, 4, 2>(a, attr_only);
	case 43: return ring_up_launch<DBITS, 4, 3>(a, attr_only);
	default: return ring_up_launch<DBITS, 4, 4>(a, attr_only);
	}
}
template <int DBITS>
void ring_res_dispatch(const MatResArgs& a, int u, int S, int grid, size_t smem, bool attr_only) {
	switch (u * 10 + g.ring_res_ns) {
	case 22: return ring_res_launch<DBITS, 2, 2>(a, S, grid, smem, attr_only);
	case 23: return ring_res_launch<DBITS, 2, 3>(a, S, grid, smem, attr_only);
	case 24: return ring_res_launch<DBITS, 2, 4>(a, S, grid, smem, attr_only);
	case 42: return ring_res_launch<DBITS, 4, 2>(a, S, grid, smem, attr_only);
	case 43: return ring_res_launch<DBITS, 4, 3>(a, S, grid, smem, attr_only);
	default: return ring_res_launch<DBITS, 4, 4>(a, S, grid, smem, attr_only);
	}
}

// first `budget` bytes of the (w1, w3) row interleave that k_ffn_up walks: half from each matrix (row prefixes)
static void pf_up_prefix(Prefetch& pf, int slot, const void* w1, const void* w3, size_t skip, size_t budget, size_t matrix_bytes) {
	size_t off = (skip / 2) & ~(size_t)15, len = (budget / 2) & ~(size_t)15;
	if (off >= matrix_bytes) return;
	if (off + len > matrix_bytes) len = matrix_bytes - off;
	pf.p[slot] = (const char*)w1 + off, pf.bytes[slot] = len;
	pf.p[slot + 1] = (const char*)w3 + off, pf.bytes[slot + 1] = len;
}

// mode: 0 kv only, 1 logits -> host, 2 logits -> device + advance (greedy loop), 3 logits -> host + argmax, 4 logits -> device + min-p sample + advance
template <int DBITS, typename KVT>
int run_token(int mode) {
	const Config& c = g.cfg;
	const Weights& w = g.w;
	const int dim = c.dim, hidden = c.hidden_dim, hd = c.head_dim;
	const size_t wb = (size_t)DBITS; // bits per weight
	int nl = 0;
	g.n_stamps = 0;
	const size_t kv_layer = (size_t)c.n_kv_heads * c.seq_len * hd; // elements per layer
	const size_t qkv_bytes[3] = {(size_t)g.q_dim * dim * wb / 8, (size_t)g.kv_dim * dim * wb / 8, (size_t)g.kv_dim * dim * wb / 8};
	const size_t wo_bytes = (size_t)dim * g.q_dim * wb / 8, up_bytes = (size_t)hidden * dim * wb / 8 /* per matrix (and expert) */, down_bytes = up_bytes;
	const bool dense = c.n_experts == 0;
	auto kv_prefix = [&](Prefetch& pf, int l) {
		pf.kc = (KVT*)g.kc + l * kv_layer, pf.vc = (KVT*)g.vc + l * kv_layer;
		pf.kv_rowbytes = hd * (int)sizeof(KVT), pf.kv_heads = c.n_kv_heads, pf.kv_head_stride = (unsigned long long)c.seq_len * hd * sizeof(KVT);
	};
	auto qkv_weights = [&](Prefetch& pf, int l) {
		pf.p[0] = w.wq[l], pf.bytes[0] = qkv_bytes[0], pf.p[1] = w.wk[l], pf.bytes[1] = qkv_bytes[1], pf.p[2] = w.wv[l], pf.bytes[2] = qkv_bytes[2];
	};

	{
		StageScope t(ST_EMBED, 0);
		EmbedArgs<KVT> a = {};
		a.x = g.x, a.table = w.token_embedding_table, a.tp = g.tp, a.dim = dim;
		a.embed_blocks = cdiv(dim, 256);
		a.key_cache = (KVT*)g.kc, a.rope_freq = g.rope_freq, a.rope_cs = g.rope_cs;
		a.n_layers = c.n_layers, a.n_kv_heads = c.n_kv_heads, a.head_dim = hd, a.seq_len = c.seq_len;
		a.stamp = nullptr, a.stamp_reset = g.perf ? g.stamps : nullptr, a.n_stamps = MAX_STAMPS + 8; // + the 16 debug stamps
		if (g.pf_down_qkv) qkv_weights(a.pf, 0);
		launch_pdl(k_embed<DBITS, KVT>, a.embed_blocks + 8, 256, 0, a);
		++nl;
	}

	for (int l = 0; l < c.n_layers; ++l) {
		{
			StageScope t(ST_QKV, (double)(g.q_dim + 2 * g.kv_dim) * dim * wb / 8);
			QkvArgs<KVT> a = {};
			a.x = g.x, a.normw = w.rms_att_weight[l], a.wq = w.wq[l], a.wk = w.wk[l], a.wv = w.wv[l], a.bias = w.bqkv[l];
			a.q_out = g.q, a.kc = (KVT*)g.kc + l * kv_layer, a.vc = (KVT*)g.vc + l * kv_layer;
			a.rope_cs = g.rope_cs, a.xb_out = c.norm_par ? g.xb : nullptr, a.tp = g.tp;
			a.dim = dim, a.q_dim = g.q_dim, a.kv_dim = g.kv_dim, a.head_dim = hd, a.seq_len = c.seq_len;
			a.eps = c.norm_eps, a.clip = c.qkv_clip, a.ln = c.norm_ln;
			a.stamp = t.slot;
			if (g.pf_kv && (l == 0 || !g.pf_down_qkv)) kv_prefix(a.pf, l); // later layers: requested by the previous w2 kernel
			launch_pdl(k_qkv<DBITS, KVT>, g.grid_qkv, QKV_THREADS, g.smem_dim, a);
			++nl;
		}
		{
			StageScope t(ST_ATTN, -1.0); // bytes depend on the position: accounted per token in launch_token()
			AttnArgs a = {};
			a.q = g.q, a.kc = (KVT*)g.kc + l * kv_layer, a.vc = (KVT*)g.vc + l * kv_layer;
			a.partial = g.attn_partial, a.counter = g.attn_counter, a.out = g.att, a.tp = g.tp;
			a.head_dim = hd, a.seq_len = c.seq_len, a.nsplit = g.attn_nsplit, a.lpp = g.attn_lpp;
			a.kv_mul = g.kv_mul, a.qgroups = g.attn_qgroups;
			a.inv_sqrt_hd = 1.0f / sqrtf((float)hd);
			a.nbmax = g.attn_nbmax;
			a.cells = g.attn_cells, a.epoch_stride = (unsigned)c.n_layers + 1, a.epoch_idx = (unsigned)l + 1, a.err = g.dev_err;
			a.dbg = (g.perf && l == c.n_layers / 2) ? g.stamps + 2 * (size_t)MAX_STAMPS : nullptr;
			a.stamp = t.slot;
			if (g.pf_attn_wo) a.pf.p[0] = w.wo[l], a.pf.bytes[0] = wo_bytes;
			if (dense && g.pf_attn_up) pf_up_prefix(a.pf, 1, w.w1[l], w.w3[l], 0, g.pf_attn_up, up_bytes);
			dispatch_attn<KVT>(a, c.n_kv_heads * g.attn_qgroups, &nl);
		}
		{
			StageScope t(ST_WO, (double)dim * g.q_dim * wb / 8);
			MatResArgs a = {};
			a.xin = g.att, a.w = w.wo[l], a.y = g.x, a.sel = nullptr, a.n = g.q_dim, a.d = dim, a.nact = 1, a.accumulate = 1, a.tp = g.tp;
			a.stamp = t.slot;
			if (dense && g.pf_wo_up) pf_up_prefix(a.pf, 0, w.w1[l], w.w3[l], g.pf_attn_up, g.pf_wo_up, up_bytes);
			if (g.tp_fused) tp_fill(a.tpx, 2 * l); // partial over this rank's heads, summed over the ranks in the kernel
			else if (g.tp_world > 1) a.y = g.xpart, a.accumulate = 0;
			if (g.ring_wo_u) ring_res_dispatch<DBITS>(a, g.ring_wo_u, g.ring_wo_s, g.grid_wo_ring, g.smem_wo_ring, false);
			else launch_pdl(k_matres<DBITS>, g.grid_wo, 256, g.smem_qdim, a);
			++nl;
			if (g.tp_world > 1 && !g.tp_fused) {
				tp_allreduce(g.xpart, dim);
				launch_pdl(k_addvec, cdiv(dim, 256), 256, 0, g.x, (const float*)g.xpart, dim);
				++nl;
			}
		}
		{
			StageScope t(ST_FFN_UP, (double)2 * g.nact * hidden * dim * wb / 8);
			FfnUpArgs a = {};
			a.x = (c.norm_par ? g.xb : g.x), a.normw = c.norm_par ? nullptr : w.rms_ffn_weight[l];
			a.gate = c.n_experts ? w.moegate[l] : nullptr, a.w1 = w.w1[l], a.w3 = w.w3[l], a.hb = g.hb, a.sel = g.moe_sel;
			a.dim = dim, a.hidden = hidden, a.n_experts = c.n_experts, a.nact = g.nact;
			a.eps = c.norm_eps, a.ln = c.norm_ln, a.gelu = c.act_gelu;
			a.expert_stride = g.up_expert_stride;
			a.stamp = t.slot;
			if (dense && g.pf_up_down) a.pf.p[0] = w.w2[l], a.pf.bytes[0] = (g.pf_up_down < down_bytes ? g.pf_up_down : down_bytes) & ~(size_t)15;
			bool done = false;
			if (g.ring_up_u) ring_up_dispatch<DBITS>(a, false), done = true;
			if (!done) launch_pdl(k_ffn_up<DBITS>, g.grid_up, 256, g.smem_dim, a);
			++nl;
		}
		{
			StageScope t(ST_FFN_DOWN, (double)g.nact * hidden * dim * wb / 8);
			MatResArgs a = {};
			a.xin = g.hb, a.w = w.w2[l], a.y = g.x, a.sel = c.n_experts ? g.moe_sel : nullptr;
			a.n = hidden, a.d = dim, a.nact = g.nact, a.accumulate = 1, a.tp = g.tp;
			a.stamp = t.slot;
			if (l + 1 < c.n_layers && g.pf_down_qkv) {
				qkv_weights(a.pf, l + 1);
				if (g.pf_kv) kv_prefix(a.pf, l + 1);
			}
			if (g.tp_fused) tp_fill(a.tpx, 2 * l + 1); // partial over this rank's FFN rows
			else if (g.tp_world > 1) a.y = g.xpart, a.accumulate = 0;
			if (g.ring_down_u) ring_res_dispatch<DBITS>(a, g.ring_down_u, g.ring_down_s, g.grid_down_ring, g.smem_down_ring, false);
			else launch_pdl(k_matres<DBITS>, g.grid_down, 256, g.smem_hidden, a);
			++nl;
			if (g.tp_world > 1 && !g.tp_fused) {
				tp_allreduce(g.xpart, dim);
				launch_pdl(k_addvec, cdiv(dim, 256), 256, 0, g.x, (const float*)g.xpart, dim);
				++nl;
			}
		}
	}

	if (mode != 0) {
		StageScope t(ST_OUTPUT, (double)c.vocab_size * dim * wb / 8);
		OutputArgs a = {};
		a.x = g.x, a.normw = w.rms_final_weight, a.wcls = w.wcls;
		a.logits = (mode == 2 || mode == 4) ? g.logits_dev : g.logits_host;
		a.cand_val = (mode >= 2) ? g.cand_val : nullptr, a.cand_idx = g.cand_idx;
		a.dim = dim, a.vocab = c.vocab_size, a.eps = c.norm_eps, a.ln = c.norm_ln;
		a.stamp = t.slot;
		int grid = g.grid_out;
		const bool split = g.tp_fused; // classifier rows divided over the ranks, slices pushed into every rank's gather area
		int ncand = grid;
		const float* cand_val = g.cand_val;
		const int* cand_idx = g.cand_idx;
		if (split) {
			a.row0 = g.out_row0, a.row1 = g.out_row1, a.world = g.tp_world, a.rank = g.tp_rank;
			for (int p = 0; p < g.tp_world; ++p) {
				char* area = (char*)g.tp_peer[p];
				a.peer_logits[p] = (float*)(area + g.tp_off_logits), a.peer_cand_val[p] = (float*)(area + g.tp_off_cval), a.peer_cand_idx[p] = (int*)(area + g.tp_off_cidx);
			}
			ncand = grid * g.tp_world;
			cand_val = (const float*)((char*)g.tp_area + g.tp_off_cval), cand_idx = (const int*)((char*)g.tp_area + g.tp_off_cidx);
		}
		launch_pdl(k_output<DBITS>, grid, 256, g.smem_dim, a);
		++nl;
		if (split) {
			TpGatherArgs ga = {};
			ga.world = g.tp_world, ga.rank = g.tp_rank, ga.tp = g.tp, ga.err = g.tp_err;
			for (int p = 0; p < g.tp_world; ++p) ga.flags[p] = (unsigned*)((char*)g.tp_peer[p] + g.tp_off_flags);
			ga.src = (const float*)((char*)g.tp_area + g.tp_off_logits), ga.dst = a.logits, ga.n = c.vocab_size;
			launch_pdl(k_tp_gather, 32, 256, 0, ga);
			++nl;
		}
		if (mode == 4) { // min-p sampling on the device (reference sampler.c:44-90), then the bookkeeping of k_advance
			SampleArgs sa;
			sa.logits = g.logits_dev, sa.cand_val = cand_val, sa.ncand = ncand, sa.vocab = c.vocab_size, sa.nchunks = g.sample_chunks;
			sa.st = g.sample_state, sa.count = g.sample_count, sa.csum = g.sample_csum, sa.sidx = g.sample_idx, sa.sprob = g.sample_prob;
			launch_pdl(k_sample_scan, g.sample_chunks, 256, 0, sa);
			launch_pdl(k_sample_pick, 1, 256, 0, sa, g.sample_state, g.tp, g.out_tokens, g.last_token, 1);
			nl += 2;
		} else if (mode >= 2) {
			launch_pdl(k_advance, 1, 256, 0, cand_val, cand_idx, ncand, g.tp, g.out_tokens, g.last_token, (int)(mode == 2), c.vocab_size);
			++nl;
		}
	}
	if (g.perf) {
		launch_pdl(k_stamp_accum, 1, 256, 0, (const unsigned long long*)g.stamps, g.stamp_acc, g.n_stamps);
		++nl;
	}
	return nl;
}


// Tensor-parallel view of the model for rank r of N (Megatron split; SURVEY.md s.8e): query/kv heads and FFN rows
// are divided, so wq/wk/wv/w1/w3 shards are contiguous row ranges of the uploaded tensors (no copy), while wo and w2
// need their COLUMN range, packed once into a contiguous (dim x n/N) matrix.  Embedding, norms and the classifier
// are replicated.  After this the engine runs unchanged on the "local" shapes; the two partial projections per layer
// are summed with one all-reduce each.
void tp_shard_model() {
	Config& c = g.cfg;
	Weights& w = g.w;
	const int N = g.tp_world, r = g.tp_rank;
	const int ne = c.n_experts ? c.n_experts : 1; // MoE: the same split inside every expert (all ranks serve both active experts)
	if (c.n_heads % N || c.n_kv_heads % N || c.hidden_dim % (32 * N)) CALM_FATAL("tensor parallelism: %d ranks do not divide heads %d/%d or hidden %d", N, c.n_heads, c.n_kv_heads, c.hidden_dim);
	const size_t wb = (size_t)w.dbits;
	const int q_dim = c.head_dim * c.n_heads, kv_dim = c.head_dim * c.n_kv_heads;
	const int ql = q_dim / N, kl = kv_dim / N, hl = c.hidden_dim / N;
	auto rows = [&](void* base, size_t row0, size_t cols) { return (void*)((char*)base + row0 * cols * wb / 8); };
	auto col_slice = [&](const void* base, int nrows, size_t cols, size_t col0, size_t ncols) {
		void* dst = dev_alloc((size_t)nrows * ncols * wb / 8);
		CUDA_CHECK(cudaMemcpy2D(dst, ncols * wb / 8, (const char*)base + col0 * wb / 8, cols * wb / 8, ncols * wb / 8, nrows, cudaMemcpyDeviceToDevice));
		g.tp_owned.push_back(dst);
		return dst;
	};
	for (int l = 0; l < c.n_layers; ++l) {
		w.wq[l] = rows(w.wq[l], (size_t)r * ql, c.dim);
		w.wk[l] = rows(w.wk[l], (size_t)r * kl, c.dim);
		w.wv[l] = rows(w.wv[l], (size_t)r * kl, c.dim);
		w.w1[l] = rows(w.w1[l], (size_t)r * hl, c.dim); // expert e's rows start e * (full hidden) rows further: up_expert_stride
		w.w3[l] = rows(w.w3[l], (size_t)r * hl, c.dim);
		w.wo[l] = col_slice(w.wo[l], c.dim, q_dim, (size_t)r * ql, ql);
		w.w2[l] = col_slice(w.w2[l], ne * c.dim, c.hidden_dim, (size_t)r * hl, hl); // [expert][dim][hl], packed
		if (w.bqkv[l]) { // [q | k | v] -> this rank's [q_r | k_r | v_r]
			float* b = (float*)dev_alloc((size_t)(ql + 2 * kl) * sizeof(float));
			CUDA_CHECK(cudaMemcpy(b, w.bqkv[l] + (size_t)r * ql, ql * sizeof(float), cudaMemcpyDeviceToDevice));
			CUDA_CHECK(cudaMemcpy(b + ql, w.bqkv[l] + q_dim + (size_t)r * kl, kl * sizeof(float), cudaMemcpyDeviceToDevice));
			CUDA_CHECK(cudaMemcpy(b + ql + kl, w.bqkv[l] + q_dim + kv_dim + (size_t)r * kl, kl * sizeof(float), cudaMemcpyDeviceToDevice));
			g.tp_owned.push_back(b);
			w.bqkv[l] = b;
		}
	}
	if (c.n_experts) g.up_expert_stride = (size_t)c.hidden_dim * c.dim * wb / 8 / 16;
	c.n_heads /= N, c.n_kv_heads /= N, c.hidden_dim = hl;
}

// Fix grid sizes and shared-memory opt-ins for this model (called once from prepare_cuda).
template <int DBITS, typename KVT>
void make_plan() {
	const Config& c = g.cfg;
	g.smem_dim = xs_bytes<DBITS>(c.dim);
	g.smem_qdim = xs_bytes<DBITS>(g.q_dim);
	g.smem_hidden = xs_bytes<DBITS>(c.hidden_dim);
	size_t smem_res = g.smem_qdim > g.smem_hidden ? g.smem_qdim : g.smem_hidden;
	if (smem_res > 227 * 1024 || g.smem_dim > 227 * 1024) CALM_FATAL("activation vector does not fit in shared memory (dim %d, hidden %d)", c.dim, c.hidden_dim);
	smem_optin(k_qkv<DBITS, KVT>, g.smem_dim), smem_optin(k_ffn_up<DBITS>, g.smem_dim), smem_optin(k_output<DBITS>, g.smem_dim);
	smem_optin(k_matres<DBITS>, smem_res); // ONE attribute per kernel: the larger of its two launch shapes (wo, w2)
	{
		// k_attn2 when the shape is instantiated and the CTA's share of the context fits in shared memory
		g.attn_nbmax = cdiv(cdiv(c.seq_len, ATTN2_BP), g.attn_nsplit);
		g.attn2_smem = attn2_smem_bytes<KVT>(g.attn_hg, c.head_dim, g.attn_nbmax, g.attn_nsplit);
		const bool want = !(getenv("CALM_B200_ATTN2") && atoi(getenv("CALM_B200_ATTN2")) == 0);
		g.attn2 = want && attn2_shape_ok(g.attn_hg, g.attn_lpp, c.head_dim) && g.attn_nbmax <= ATTN2_MAXB && g.attn2_smem <= 200 * 1024;
		g.attn2_cluster = g.attn2 && g.attn_nsplit <= ATTN2_MAX_CLUSTER && getenv("CALM_B200_ATTN_CLUSTER") && atoi(getenv("CALM_B200_ATTN_CLUSTER")) != 0;
		// k_attn_mma where it applies (CALM_B200_ATTN_MMA=0: k_attn2, for A/B runs in one build)
		g.attn_mma_smem = attn_mma_smem_bytes<KVT>(g.attn_nbmax);
		const bool want_mma = !(getenv("CALM_B200_ATTN_MMA") && atoi(getenv("CALM_B200_ATTN_MMA")) == 0);
		g.attn_mma = want_mma && g.attn2 && !g.attn2_cluster && g.attn_hg == ATTN_MMA_HG && c.head_dim == ATTN_MMA_HD && g.attn_mma_smem <= 200 * 1024;
		AttnArgs aa = {};
		aa.head_dim = c.head_dim, aa.nsplit = g.attn_nsplit;
		dispatch_attn<KVT>(aa, c.n_kv_heads * g.attn_qgroups, nullptr);
	}
	g.grid_qkv = balanced_grid(cdiv((g.q_dim + 2 * g.kv_dim) / 2, 8), max_ctas(k_qkv<DBITS, KVT>, QKV_THREADS, g.smem_dim));
	g.grid_wo = balanced_grid(cdiv(c.dim / 2, 8), max_ctas(k_matres<DBITS>, 256, g.smem_qdim));
	g.grid_down = balanced_grid(cdiv(c.dim / 2, 8), max_ctas(k_matres<DBITS>, 256, g.smem_hidden));
	if (g.tp_fused) { // the in-kernel exchange needs co-resident grids (they are: balanced_grid stays under the cap) within its tables
		for (int grid : {g.grid_wo, g.grid_down})
			if (cdiv(c.dim / 2, grid * 8) > TP_MAX_ITERS) CALM_FATAL("tensor parallelism: grid %d outside the exchange tables for dim %d", grid, c.dim);
	}
	// (measured: for the long FFN-up stage a full 4-CTA/SM grid with uneven rounds beats a balanced 3-CTA/SM one)
	g.grid_up = imin(max_ctas(k_ffn_up<DBITS>, 256, g.smem_dim), cdiv(g.nact * c.hidden_dim, 8));
	// TMA-ring kernels for the dense single-GPU stages whose rows are whole 1 KB / 2 KB chunks (ring.cuh)
	g.ring_up_u = g.ring_wo_u = g.ring_down_u = 0;
	{ // weights are read once per token: L2::evict_first on the ring's bulk copies measured 2 % faster than the default policy
		const int hint = getenv("CALM_B200_RING_HINT") ? atoi(getenv("CALM_B200_RING_HINT")) : 1;
		CUDA_CHECK(cudaMemcpyToSymbol(d_ring_l2_hint, &hint, sizeof(int)));
	}
	if (const char* e = getenv("CALM_B200_RING")) sscanf(e, "%d,%d,%d,%d", &g.ring_up_ns, &g.ring_up_cps, &g.ring_res_ns, &g.ring_res_warps); // 0 slots: stage not ring-fed
	const bool ring_ok = c.n_experts == 0; // MoE: the expert rows are known only after the router
	const bool ring_up_on = ring_ok && g.ring_up_ns >= 2 && g.ring_up_ns <= RING_MAX_NS; // (row shards of w1 / w3 under tensor parallelism are fine)
	const bool ring_res_on = ring_ok && (g.tp_world == 1 || g.tp_fused) /* the ring kernels carry the in-kernel exchange too */ && g.ring_res_ns >= 2 && g.ring_res_ns <= RING_MAX_NS && (g.ring_res_warps == 8 || g.ring_res_warps == 16); // (gf4 too: 2.384 vs 2.467 ms per Mistral-7B token, profiles/r02_sweep_gf4_rows_per_slot.jsonl)
	auto chunk_units = [](size_t rowbytes) { return rowbytes % 2048 == 0 ? 4 : (rowbytes % 1024 == 0 ? 2 : 0); };
	if (ring_up_on) {
		const int u = chunk_units((size_t)c.dim * DBITS / 8);
		if (u) {
			g.smem_up_ring = ring_smem_bytes<DBITS>(c.dim, u, g.ring_up_ns, 8);
			if (g.smem_up_ring <= 200 * 1024) {
				g.ring_up_u = u;
				g.grid_up_ring = imin(g.sms * imin(g.ring_up_cps, (int)(220 * 1024 / g.smem_up_ring)), c.hidden_dim);
				if (g.grid_up_ring < 1) g.grid_up_ring = 1;
				FfnUpArgs fa = {};
				ring_up_dispatch<DBITS>(fa, true);
			}
		}
	}
	if (ring_res_on) {
		auto plan_res = [&](int n, int& u_out, int& s_out, int& grid_out, size_t& smem_out) {
			const size_t rowbytes = (size_t)n * DBITS / 8;
			int u = chunk_units(rowbytes);
			if (u == 4 && getenv("CALM_B200_RING_RES_U") && atoi(getenv("CALM_B200_RING_RES_U")) == 2) u = 2; // (experiments) 1 KB chunks
			if (!u) return;
			size_t smem = ring_smem_bytes<DBITS>(n, u, g.ring_res_ns, g.ring_res_warps);
			if (smem > 220 * 1024 && u == 4) u = 2, smem = ring_smem_bytes<DBITS>(n, u, g.ring_res_ns, g.ring_res_warps); // long activation vectors (70B w2: 112 KB): 1 KB chunks
			if (smem > 220 * 1024) return;
			const int grid = imin(g.sms * imin(16 / g.ring_res_warps, (int)(224 * 1024 / smem)), c.dim / 2);
			const int cpt = (int)(rowbytes / (u * 512));
			if (g.tp_world > 1 && cdiv(c.dim / 2, grid) + 1 > RING_MAX_PAIRS) return; // the exchange keeps a CTA's rows in shared memory
			const bool split = cdiv(c.dim / 2, grid) + 1 <= RING_MAX_PAIRS && cpt <= RING_MAX_SLICES; // K-slices of one chunk, folded in shared memory
			u_out = u, s_out = split ? 1 : cpt, grid_out = grid < 1 ? 1 : grid, smem_out = smem;
			MatResArgs ma = {};
			ring_res_dispatch<DBITS>(ma, u, s_out, grid_out, smem, true);
		};
		// ONE shared-memory attribute per kernel instantiation: wo and w2 may share one (same U): opt in to the larger first
		int uw = 0, ud = 0, sw = 1, sd = 1, gw = 0, gd = 0;
		size_t mw = 0, md = 0;
		plan_res(g.q_dim, uw, sw, gw, mw);
		plan_res(c.hidden_dim, ud, sd, gd, md);
		if (uw && ud && uw == ud) { // same instantiation: its attribute must cover both launches
			MatResArgs ma = {};
			ring_res_dispatch<DBITS>(ma, uw, 1, 1, mw > md ? mw : md, true);
		}
		g.ring_wo_u = uw, g.ring_wo_s = sw, g.grid_wo_ring = gw, g.smem_wo_ring = mw;
		g.ring_down_u = ud, g.ring_down_s = sd, g.grid_down_ring = gd, g.smem_down_ring = md;
	}
	g.out_row0 = 0, g.out_row1 = c.vocab_size;
	if (g.tp_fused) { // vocabulary split: equal slices of whole 32-row CTA iterations (the last rank's may be short)
		const int per = cdiv(cdiv(c.vocab_size, g.tp_world), 32) * 32;
		g.out_row0 = imin(c.vocab_size, g.tp_rank * per), g.out_row1 = imin(c.vocab_size, g.out_row0 + per);
		g.grid_out = balanced_grid(cdiv(per, 32), max_ctas(k_output<DBITS>, 256, g.smem_dim)); // the same grid on every rank
		if (g.grid_out > TP_MAX_CAND) CALM_FATAL("tensor parallelism: %d classifier CTAs exceed the gather area", g.grid_out);
	} else {
		g.grid_out = balanced_grid(cdiv(c.vocab_size, 32), max_ctas(k_output<DBITS>, 256, g.smem_dim));
	}
	g.ncand = g.grid_out;
}

template <int DBITS>
void make_plan_kv() {
	g.kvbits == 8 ? make_plan<DBITS, uint8_t>() : make_plan<DBITS, __half>();
}

template <int DBITS>
int run_token_kv(int mode) {
	return g.kvbits == 8 ? run_token<DBITS, uint8_t>(mode) : run_token<DBITS, __half>(mode);
}

int run_token_any(int mode) {
	switch (g.w.dbits) {
	case 16: return run_token_kv<16>(mode);
	case 8: return run_token_kv<8>(mode);
	default: return run_token_kv<4>(mode);
	}
}


void launch_token(int mode) {
	const int pv = g.perf ? 1 : 0; // the profiling variant is the same graph with stamp slots
	if (!g.use_graph) {
		g_launches += run_token_any(mode);
		CUDA_CHECK(cudaGetLastError());
	} else {
		if (!g.graph[pv][mode]) {
			cudaGraph_t graph;
			CUDA_CHECK(cudaStreamBeginCapture(g.stream, cudaStreamCaptureModeThreadLocal));
			g.graph_launches[pv][mode] = run_token_any(mode);
			CUDA_CHECK(cudaStreamEndCapture(g.stream, &graph));
			CUDA_CHECK(cudaGraphInstantiate(&g.graph[pv][mode], graph, 0));
			CUDA_CHECK(cudaGraphDestroy(graph));
		}
		CUDA_CHECK(cudaGraphLaunch(g.graph[pv][mode], g.stream));
		g_launches += g.graph_launches[pv][mode];
	}
	if (g.perf) { // algorithmic bytes of this token per stage (the reference's accounting, infer.cu:683-699)
		const int n = g.cfg.n_layers * 5 + (mode != 0 ? 1 : 0) + 1;
		for (int i = 0; i < n && i < MAX_STAMPS; ++i) {
			const int st = g.stamp_stage[i];
			g.stage_bytes[st] += g.stamp_bytes[i] >= 0 ? g.stamp_bytes[i] : 2.0 * g.kv_dim * g.cur_kv_len * (g.kvbits / 8);
			g.stage_launches[st] += 1;
		}
		++g.perf_runs;
	}
}

void set_params(int token, int pos, int step) {
	g.cur_kv_len = pos >= g.cfg.seq_len ? g.cfg.seq_len : pos + 1;
	g.cur_pos = pos;
	same_carveout((const void*)k_set_params);
	k_set_params<<<1, 1, 0, g.stream>>>(g.tp, token, pos, g.cfg.seq_len, step);
	++g_launches;
}

} // namespace

// =================================================================================================
// C ABI

extern "C" int calm_b200_abi_version(void) {
	return CALM_B200_ABI_VERSION;
}

extern "C" void calm_b200_set_device(int device) {
	g_device_override = device;
}

extern "C" void* upload_cuda(void* host, size_t size) {
	select_device();
	void* dev = dev_alloc(size);
	CUDA_CHECK(cudaMemcpyAsync(dev, host, size, cudaMemcpyHostToDevice));
	return dev;
}

extern "C" void calm_b200_free(void* device_ptr) {
	if (device_ptr) CUDA_CHECK(cudaFree(device_ptr));
}

extern "C" void prepare_cuda(struct Transformer* transformer) {
	select_device();
	if (g.ready) CALM_FATAL("prepare_cuda called twice; call calm_b200_release() first (one model per process, as in the reference)");

	Config c = transformer->config; // copies: under tensor parallelism they become this rank's shard view
	Weights w = transformer->weights;
	RunState* s = &transformer->state;

	cudaDeviceProp prop;
	CUDA_CHECK(cudaGetDeviceProperties(&prop, g.device));
	if (prop.major != 10) CALM_FATAL("device %s is sm_%d%d; this library contains sm_100a code only and has no fallback", prop.name, prop.major, prop.minor);
	g.sms = prop.multiProcessorCount;
	if (!getenv("CALM_B200_QUIET"))
		printf("# CUDA: %s, compute %d.%d, %d SMs, %.1f GiB, peak bandwidth %.0f GB/s (ECC %d)\n", prop.name, prop.major, prop.minor, prop.multiProcessorCount,
		       (double)prop.totalGlobalMem / (1024 * 1024 * 1024), (double)prop.memoryClockRate * (prop.memoryBusWidth / 8) * 2 / 1e6, prop.ECCEnabled);

	// configuration checks (the reference asserts the same alignment, infer.cu:670, 755)
	if (w.dbits != 4 && w.dbits != 8 && w.dbits != 16) CALM_FATAL("unsupported dbits %d: must be 4, 8 or 16", w.dbits);
	if (s->kvbits != 8 && s->kvbits != 16) CALM_FATAL("unsupported kvbits %d: must be 8 or 16", s->kvbits);
	int q_dim = c.head_dim * c.n_heads, kv_dim = c.head_dim * c.n_kv_heads;
	if (c.dim % 32 || kv_dim % 32 || c.hidden_dim % 32 || q_dim % 32) CALM_FATAL("dim, q_dim, kv_dim and hidden_dim must be multiples of 32");
	if (c.head_dim % 8 || c.head_dim > 256) CALM_FATAL("head_dim %d unsupported (multiple of 8, <= 256)", c.head_dim);
	if (c.n_heads % c.n_kv_heads) CALM_FATAL("n_heads must be a multiple of n_kv_heads");
	if (c.n_layers > MAX_LAYERS) CALM_FATAL("too many layers");
	if (c.n_experts > MAX_EXPERTS || c.n_experts_ac > CALM_MAX_ACTIVE) CALM_FATAL("too many experts (%d, %d active)", c.n_experts, c.n_experts_ac);
	if (c.seq_len <= KV_SINKS) CALM_FATAL("seq_len too small");

	g.cfg = c;
	g.w = w;
	g.kvbits = s->kvbits;
	g.nact = c.n_experts ? c.n_experts_ac : 1;
	g.tp_rank = g_tp_rank, g.tp_world = g_tp_world;
	if (g.tp_world > 1) {
		nccl_load();
		NCCL_CHECK(g_nccl.CommInitRank(&g.tp_comm, g.tp_world, g_tp_id, g.tp_rank));
		tp_shard_model(); // g.cfg / g.w now describe this rank's shard
		c = g.cfg, w = g.w;
		q_dim = c.head_dim * c.n_heads, kv_dim = c.head_dim * c.n_kv_heads;
		if (kv_dim % 32 || c.hidden_dim % 32 || q_dim % 32) CALM_FATAL("tensor parallelism: per-rank q_dim, kv_dim and hidden_dim must be multiples of 32");
		g.xpart = (float*)dev_alloc(c.dim * sizeof(float));
	}
	g.q_dim = q_dim, g.kv_dim = kv_dim, g.kv_mul = g.cfg.n_heads / g.cfg.n_kv_heads;
	g.use_graph = !(getenv("CALM_B200_GRAPH") && atoi(getenv("CALM_B200_GRAPH")) == 0);
	g.use_pdl = !(getenv("CALM_B200_PDL") && atoi(getenv("CALM_B200_PDL")) == 0);
	g.carveout = getenv("CALM_B200_CARVEOUT") ? atoi(getenv("CALM_B200_CARVEOUT")) : -1;
	g.debug = getenv("CALM_B200_DEBUG") && atoi(getenv("CALM_B200_DEBUG"));
	if (g.debug) g.use_graph = false;
	g.perf = (getenv("CALM_B200_PERF") && atoi(getenv("CALM_B200_PERF"))) || getenv("CUDA_INJECTION64_PATH");
	if (getenv("CALM_B200_PERF") && atoi(getenv("CALM_B200_PERF"))) { // the reference driver only calls perf_cuda under a CUPTI injection (run.c:630): print at exit
		static bool registered = false;
		if (!registered) atexit(perf_cuda), registered = true;
	}
	if (const char* e = getenv("CALM_B200_PF")) { // kv,attn_wo,attn_up_MB,wo_up_MB,up_down_MB,down_qkv  (experiments; defaults in struct Engine)
		int kv = 0, awo = 0, aup = 0, wup = 0, ud = 0, dq = 0;
		sscanf(e, "%d,%d,%d,%d,%d,%d", &kv, &awo, &aup, &wup, &ud, &dq);
		g.pf_kv = kv != 0, g.pf_attn_wo = awo != 0, g.pf_attn_up = (size_t)aup << 20, g.pf_wo_up = (size_t)wup << 20, g.pf_up_down = (size_t)ud << 20, g.pf_down_qkv = dq != 0;
	}

	CUDA_CHECK(cudaStreamCreateWithFlags(&g.stream, cudaStreamNonBlocking));
	for (int i = 0; i < 2; ++i) CUDA_CHECK(cudaEventCreate(&g.timer[i]));
	g.stamps = (unsigned long long*)dev_alloc((size_t)(MAX_STAMPS * 2 + 16) * sizeof(unsigned long long));
	g.stamp_acc = (unsigned long long*)dev_alloc((size_t)(MAX_STAMPS + 2) * sizeof(unsigned long long));
	CUDA_CHECK(cudaMemset(g.stamps, 0, (size_t)(MAX_STAMPS * 2 + 16) * sizeof(unsigned long long)));
	CUDA_CHECK(cudaMemset(g.stamp_acc, 0, (size_t)(MAX_STAMPS + 2) * sizeof(unsigned long long)));
	if (g.tp_world > 1) { // first collective outside any graph capture: NCCL sets up its channels and buffers here
		CUDA_CHECK(cudaMemsetAsync(g.xpart, 0, c.dim * sizeof(float), g.stream));
		tp_allreduce(g.xpart, c.dim);
		CUDA_CHECK(cudaStreamSynchronize(g.stream));
		tp_setup_exchange();
	}

	g.x = (float*)dev_alloc(c.dim * sizeof(float));
	g.xb = (float*)dev_alloc(c.dim * sizeof(float));
	g.q = (float*)dev_alloc(q_dim * sizeof(float));
	g.att = (float*)dev_alloc(q_dim * sizeof(float));
	g.hb = (float*)dev_alloc((size_t)g.nact * c.hidden_dim * sizeof(float));
	g.logits_dev = (float*)dev_alloc((size_t)c.vocab_size * sizeof(float));
	CUDA_CHECK(cudaHostAlloc((void**)&g.logits_host, (size_t)c.vocab_size * sizeof(float), cudaHostAllocMapped));
	CUDA_CHECK(cudaHostAlloc((void**)&g.last_token, sizeof(int), cudaHostAllocMapped));
	memset(g.logits_host, 0, (size_t)c.vocab_size * sizeof(float));

	size_t kvbytes = (size_t)c.n_layers * c.seq_len * kv_dim * (g.kvbits / 8);
	g.kc = dev_alloc(kvbytes);
	g.vc = dev_alloc(kvbytes);
	CUDA_CHECK(cudaMemsetAsync(g.kc, 0, kvbytes, g.stream));
	CUDA_CHECK(cudaMemsetAsync(g.vc, 0, kvbytes, g.stream));

	// RoPE frequencies with the host libm, exactly as the CPU reference forms them (infer.c:225-226)
	std::vector<float> freq(c.head_dim / 2);
	for (int i = 0; i < c.head_dim; i += 2) freq[i / 2] = i >= c.rotary_dim ? 0.f : 1.0f / powf(c.rope_theta, (float)i / (float)c.rotary_dim);
	g.rope_cs = (float2*)dev_alloc(freq.size() * sizeof(float2));
	g.rope_freq = (float*)dev_alloc(freq.size() * sizeof(float));
	CUDA_CHECK(cudaMemcpyAsync(g.rope_freq, freq.data(), freq.size() * sizeof(float), cudaMemcpyHostToDevice, g.stream));
	CUDA_CHECK(cudaStreamSynchronize(g.stream)); // freq is a local

	// attention shape: query-head group per CTA (largest divisor of kv_mul <= 8), lanes per position, slices
	g.attn_hg = 1;
	for (int h = 8; h >= 1; --h)
		if (g.kv_mul % h == 0) {
			g.attn_hg = h;
			break;
		}
	g.attn_qgroups = g.kv_mul / g.attn_hg;
	g.attn_lpp = 1;
	while (g.attn_lpp * 8 < c.head_dim) g.attn_lpp *= 2;
	int units = c.n_kv_heads * g.attn_qgroups;
	const int split_mul = getenv("CALM_B200_ATTN_SPLIT_MUL") ? atoi(getenv("CALM_B200_ATTN_SPLIT_MUL")) : 1; // CTAs per SM (experiments)
	int want = (split_mul > 1 ? split_mul : 1) * g.sms / units; // about one 256-thread CTA per SM
	int maxsplit = cdiv(c.seq_len, 64);                 // at least 64 positions per slice at full context
	g.attn_nsplit = want < 1 ? 1 : (want > maxsplit ? maxsplit : want);
	// (measured 9 us per launch SLOWER than the global-partial fold: a 16-CTA cluster needs 16 SMs of one GPC at once, which the
	// still-resident q/k/v CTAs delay; kept selectable for the record -- profiles/r02_sweep_ring_and_attention_variants.jsonl)
	if (g.attn_nsplit > ATTN2_MAXB + 4) g.attn_nsplit = ATTN2_MAXB + 4; // k_attn2 keeps one (m, l) pair per slice in static shared memory
	const bool want_cluster = getenv("CALM_B200_ATTN_CLUSTER") && atoi(getenv("CALM_B200_ATTN_CLUSTER")) != 0;
	if (want_cluster && attn2_shape_ok(g.attn_hg, g.attn_lpp, c.head_dim) && !(getenv("CALM_B200_ATTN2") && atoi(getenv("CALM_B200_ATTN2")) == 0)) {
		int ns = 1; // the slices of a unit will be one thread-block cluster: a power of two, at most 16 CTAs
		while (ns * 2 <= g.attn_nsplit && ns * 2 <= ATTN2_MAX_CLUSTER) ns *= 2;
		g.attn_nsplit = ns;
	}
	g.attn_partial = (float*)dev_alloc((size_t)units * g.attn_nsplit * g.attn_hg * (c.head_dim + 2) * sizeof(float));
	{
		const size_t cell_bytes = (size_t)units * (g.sms / units > g.attn_nsplit ? g.sms / units : g.attn_nsplit) * g.attn_hg * (c.head_dim + 2) * sizeof(unsigned long long);
		// (the attention grid must be co-resident for the cell fold: units * nsplit CTAs of <= 1/2 SM each)
		g.attn_cells = (unsigned long long*)dev_alloc(cell_bytes);
		CUDA_CHECK(cudaMemset(g.attn_cells, 0, cell_bytes));
		CUDA_CHECK(cudaHostAlloc((void**)&g.dev_err, sizeof(int), cudaHostAllocMapped));
		*g.dev_err = 0;
	}
	g.attn_counter = (unsigned*)dev_alloc(units * sizeof(unsigned));
	CUDA_CHECK(cudaMemset(g.attn_counter, 0, units * sizeof(unsigned)));

	g.attn_nsplit_cap = g.attn_nsplit; // the partial buffer below is sized for this many slices
	if (g.sms / units > g.attn_nsplit_cap) {
		g.attn_nsplit_cap = g.sms / units;
		CUDA_CHECK(cudaFree(g.attn_partial));
		g.attn_partial = (float*)dev_alloc((size_t)units * g.attn_nsplit_cap * g.attn_hg * (c.head_dim + 2) * sizeof(float));
	}
	g.moe_sel = (MoeSel*)dev_alloc(sizeof(MoeSel));
	CUDA_CHECK(cudaMemset(g.moe_sel, 0, sizeof(MoeSel)));
	g.tp = (TokenParams*)dev_alloc(sizeof(TokenParams));
	CUDA_CHECK(cudaMemset(g.tp, 0, sizeof(TokenParams)));

	switch (w.dbits) {
	case 16: make_plan_kv<16>(); break;
	case 8: make_plan_kv<8>(); break;
	default: make_plan_kv<4>(); break;
	}
	g.cand_val = (float*)dev_alloc(g.ncand * sizeof(float));
	g.cand_idx = (int*)dev_alloc(g.ncand * sizeof(int));
	g.out_tokens_cap = 1 << 16;
	g.out_tokens = (int*)dev_alloc(g.out_tokens_cap * sizeof(int));
	g.sample_chunks = cdiv(c.vocab_size, SAMPLE_CHUNK);
	g.sample_state = (SampleState*)dev_alloc(sizeof(SampleState));
	g.sample_count = (int*)dev_alloc(g.sample_chunks * sizeof(int));
	g.sample_csum = (float*)dev_alloc(g.sample_chunks * sizeof(float));
	g.sample_idx = (int*)dev_alloc((size_t)g.sample_chunks * SAMPLE_CHUNK * sizeof(int));
	g.sample_prob = (float*)dev_alloc((size_t)g.sample_chunks * SAMPLE_CHUNK * sizeof(float));

	// what the reference backend publishes in RunState (infer.cu:99-112)
	s->x = g.x, s->hb = g.hb, s->he = g.hb, s->q = g.q, s->att = g.att;
	s->key_cache = g.kc, s->value_cache = g.vc;
	s->logits = g.logits_host;

	g.ready = true;
	CUDA_CHECK(cudaDeviceSynchronize());
}

extern "C" void calm_b200_tp_unique_id(void* out128) {
	select_device();
	nccl_load();
	Id128 id;
	memset(&id, 0, sizeof(id));
	NCCL_CHECK(g_nccl.GetUniqueId(&id));
	memcpy(out128, &id, sizeof(id));
}

extern "C" void calm_b200_tp_init(int rank, int world, const void* id128) {
	if (g.ready) CALM_FATAL("calm_b200_tp_init must precede prepare_cuda");
	if (world < 1 || rank < 0 || rank >= world) CALM_FATAL("calm_b200_tp_init: bad rank %d of %d", rank, world);
	g_tp_rank = rank, g_tp_world = world;
	if (world > 1) memcpy(&g_tp_id, id128, sizeof(g_tp_id));
}

extern "C" int calm_b200_tp_world(void) {
	return g.ready ? g.tp_world : g_tp_world;
}

extern "C" int calm_b200_tp_mode(void) {
	return !g.ready || g.tp_world <= 1 ? 0 : (g.tp_fused ? 2 : 1);
}

extern "C" void calm_b200_release(struct Transformer* transformer) {
	if (!g.ready) return;
	CUDA_CHECK(cudaDeviceSynchronize());
	for (int v = 0; v < 2; ++v)
		for (int i = 0; i < 5; ++i)
			if (g.graph[v][i]) CUDA_CHECK(cudaGraphExecDestroy(g.graph[v][i]));
	cudaFree(g.stamps), cudaFree(g.stamp_acc), cudaFree(g.attn_cells);
	if (g.dev_err) cudaFreeHost(g.dev_err);
	if (pf.cap) {
		cudaFree(pf.X), cudaFree(pf.Q), cudaFree(pf.Nhi), cudaFree(pf.Nlo), cudaFree(pf.Ahi), cudaFree(pf.Alo), cudaFree(pf.Hhi), cudaFree(pf.Hlo), cudaFree(pf.rope), cudaFree(pf.tokens);
		pf = Prefill();
	}
	cudaFree(g.x), cudaFree(g.xb), cudaFree(g.q), cudaFree(g.att), cudaFree(g.hb), cudaFree(g.logits_dev);
	cudaFreeHost(g.logits_host), cudaFreeHost(g.last_token);
	cudaFree(g.kc), cudaFree(g.vc), cudaFree(g.rope_freq), cudaFree(g.rope_cs), cudaFree(g.attn_partial), cudaFree(g.attn_counter);
	cudaFree(g.moe_sel), cudaFree(g.tp), cudaFree(g.cand_val), cudaFree(g.cand_idx), cudaFree(g.out_tokens);
	for (int p = 0; p < TP_MAX_WORLD; ++p)
		if (g.tp_peer[p] && g.tp_peer[p] != g.tp_area) cudaIpcCloseMemHandle(g.tp_peer[p]);
	if (g.tp_area) cudaFree(g.tp_area);
	if (g.tp_err) cudaFreeHost(g.tp_err);
	cudaFree(g.sample_state), cudaFree(g.sample_count), cudaFree(g.sample_csum), cudaFree(g.sample_idx), cudaFree(g.sample_prob);
	if (g.tp_comm) g_nccl.CommDestroy(g.tp_comm);
	if (g.xpart) cudaFree(g.xpart);
	for (void* p : g.tp_owned) cudaFree(p);
	g_tp_world = 1, g_tp_rank = 0; // a new communicator needs a new calm_b200_tp_init
	for (int i = 0; i < 2; ++i) cudaEventDestroy(g.timer[i]);
	cudaStreamDestroy(g.stream);
	int dev = g.device;
	g = Engine();
	g.device = dev;
	if (transformer) {
		int kvbits = transformer->state.kvbits;
		memset(&transformer->state, 0, sizeof(transformer->state));
		transformer->state.kvbits = kvbits;
	}
}

static void sync_stream() {
	cudaError_t e = cudaStreamSynchronize(g.stream);
	if (e != cudaSuccess) {
		int code = g.tp_err ? *(volatile int*)g.tp_err : 0; // 9000 + the rank never heard from
		if (!code && g.dev_err) code = *(volatile int*)g.dev_err; // 9200: a slice of the attention fold never arrived
		fprintf(stderr, "calm_b200: device failure: %s (%s); watchdog code %d\n", cudaGetErrorString(e), cudaGetErrorName(e), code);
		abort();
	}
}

static void check_call(struct Transformer* transformer, int token, int pos) {
	if (!g.ready) CALM_FATAL("forward before prepare_cuda");
	(void)transformer;
	if (token < 0 || token >= g.cfg.vocab_size) CALM_FATAL("token %d out of range", token);
	if (pos < 0) CALM_FATAL("negative position");
}

extern "C" float* forward_cuda(struct Transformer* transformer, int token, int pos, unsigned flags) {
	check_call(transformer, token, pos);
	set_params(token, pos, 0);
	if (flags & FF_UPDATE_KV_ONLY) {
		launch_token(0);
		return NULL; // no synchronisation: prompt tokens pipeline (reference infer.cu:724-727)
	}
	launch_token(1);
	sync_stream();
	CUDA_CHECK(cudaGetLastError());
	return g.logits_host;
}

extern "C" int calm_b200_forward_argmax(struct Transformer* transformer, int token, int pos) {
	check_call(transformer, token, pos);
	set_params(token, pos, 0);
	launch_token(3);
	sync_stream();
	return *(volatile int*)g.last_token;
}

extern "C" void calm_b200_decode_greedy(struct Transformer* transformer, int token0, int pos0, int n_tokens, int* out_tokens) {
	check_call(transformer, token0, pos0);
	if (n_tokens > g.out_tokens_cap) CALM_FATAL("decode_greedy: at most %d tokens per call", g.out_tokens_cap);
	set_params(token0, pos0, 0);
	for (int i = 0; i < n_tokens; ++i) {
		g.cur_pos = pos0 + i, g.cur_kv_len = g.cur_pos >= g.cfg.seq_len ? g.cfg.seq_len : g.cur_pos + 1;
		launch_token(2);
	}
	sync_stream();
	CUDA_CHECK(cudaMemcpy(out_tokens, g.out_tokens, n_tokens * sizeof(int), cudaMemcpyDeviceToHost));
}

// min-p / temperature sampling without a host round trip per token (reference sample(), sampler.c:80-90)
extern "C" void calm_b200_decode_sample(struct Transformer* transformer, int token0, int pos0, int n_tokens, float temperature, float minp,
                                        unsigned long long* rng_state, int* out_tokens) {
	if (temperature == 0.0f || minp >= 1.0f) { // greedy: the reference does not touch the generator either
		calm_b200_decode_greedy(transformer, token0, pos0, n_tokens, out_tokens);
		return;
	}
	check_call(transformer, token0, pos0);
	if (n_tokens > g.out_tokens_cap) CALM_FATAL("decode_sample: at most %d tokens per call", g.out_tokens_cap);
	SampleState st;
	st.rng = *rng_state, st.temperature = temperature, st.cut_delta = logf(minp) * temperature;
	CUDA_CHECK(cudaMemcpyAsync(g.sample_state, &st, sizeof(st), cudaMemcpyHostToDevice, g.stream));
	set_params(token0, pos0, 0);
	for (int i = 0; i < n_tokens; ++i) {
		g.cur_pos = pos0 + i, g.cur_kv_len = g.cur_pos >= g.cfg.seq_len ? g.cfg.seq_len : g.cur_pos + 1;
		launch_token(4);
	}
	sync_stream();
	CUDA_CHECK(cudaMemcpy(out_tokens, g.out_tokens, n_tokens * sizeof(int), cudaMemcpyDeviceToHost));
	CUDA_CHECK(cudaMemcpy(&st, g.sample_state, sizeof(st), cudaMemcpyDeviceToHost));
	*rng_state = st.rng;
}

extern "C" int calm_b200_forward_sample(struct Transformer* transformer, int token, int pos, float temperature, float minp, unsigned long long* rng_state) {
	int tok = 0;
	calm_b200_decode_sample(transformer, token, pos, 1, temperature, minp, rng_state, &tok);
	return tok;
}

// The device sampler on its own: logits given by the host, any vocabulary size; returns the token and advances *rng_state.
// Same kernels as the decode loop (k_sample_scan + k_sample_pick); device_us (optional) receives their mean duration.
extern "C" int calm_b200_sample_logits(const float* logits_host, int vocab, float temperature, float minp, unsigned long long* rng_state, float* device_us) {
	select_device();
	if (vocab <= 0) CALM_FATAL("sample_logits: empty vocabulary");
	if (temperature == 0.0f || minp >= 1.0f) { // greedy, first maximum (sampler.c:34-42); the generator is not touched
		int best = 0;
		for (int i = 1; i < vocab; ++i)
			if (logits_host[i] > logits_host[best]) best = i;
		if (device_us) *device_us = 0.f;
		return best;
	}
	const int nchunks = cdiv(vocab, SAMPLE_CHUNK);
	cudaStream_t st;
	CUDA_CHECK(cudaStreamCreate(&st));
	float* logits = (float*)dev_alloc((size_t)vocab * sizeof(float));
	float* cmax = (float*)dev_alloc(nchunks * sizeof(float));
	SampleState* sst = (SampleState*)dev_alloc(sizeof(SampleState));
	int* count = (int*)dev_alloc(nchunks * sizeof(int));
	float* csum = (float*)dev_alloc(nchunks * sizeof(float));
	int* sidx = (int*)dev_alloc((size_t)nchunks * SAMPLE_CHUNK * sizeof(int));
	float* sprob = (float*)dev_alloc((size_t)nchunks * SAMPLE_CHUNK * sizeof(float));
	int* tok = (int*)dev_alloc(sizeof(int));
	TokenParams* tp = (TokenParams*)dev_alloc(sizeof(TokenParams));
	CUDA_CHECK(cudaMemcpyAsync(logits, logits_host, (size_t)vocab * sizeof(float), cudaMemcpyHostToDevice, st));
	SampleState hs;
	hs.rng = *rng_state, hs.temperature = temperature, hs.cut_delta = logf(minp) * temperature;
	SampleArgs sa;
	sa.logits = logits, sa.cand_val = cmax, sa.ncand = nchunks, sa.vocab = vocab, sa.nchunks = nchunks;
	sa.st = sst, sa.count = count, sa.csum = csum, sa.sidx = sidx, sa.sprob = sprob;
	cudaEvent_t e0, e1;
	CUDA_CHECK(cudaEventCreate(&e0));
	CUDA_CHECK(cudaEventCreate(&e1));
	const int reps = device_us ? 5 : 1;
	float ms = 0;
	for (int r = 0; r < reps; ++r) { // every repetition restarts from the caller's generator state: same draw
		CUDA_CHECK(cudaMemcpyAsync(sst, &hs, sizeof(hs), cudaMemcpyHostToDevice, st));
		k_chunk_max<<<nchunks, 256, 0, st>>>(logits, vocab, cmax);
		CUDA_CHECK(cudaEventRecord(e0, st));
		k_sample_scan<<<nchunks, 256, 0, st>>>(sa);
		k_sample_pick<<<1, 256, 0, st>>>(sa, sst, tp, nullptr, tok, 0);
		CUDA_CHECK(cudaEventRecord(e1, st));
		CUDA_CHECK(cudaEventSynchronize(e1));
		CUDA_CHECK(cudaGetLastError());
		CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
		g_launches += 3;
	}
	if (device_us) *device_us = ms * 1e3f;
	int htok = 0;
	CUDA_CHECK(cudaMemcpy(&htok, tok, sizeof(int), cudaMemcpyDeviceToHost));
	CUDA_CHECK(cudaMemcpy(&hs, sst, sizeof(hs), cudaMemcpyDeviceToHost));
	*rng_state = hs.rng;
	cudaFree(logits), cudaFree(cmax), cudaFree(sst), cudaFree(count), cudaFree(csum), cudaFree(sidx), cudaFree(sprob), cudaFree(tok), cudaFree(tp);
	cudaEventDestroy(e0), cudaEventDestroy(e1), cudaStreamDestroy(st);
	return htok;
}

// ---------------------------------------------------------------------------------------------
// forward_prefill_cuda: the prompt as one batched pass (SURVEY.md s.8b "additive entry points"; reference run.c:206-209 calls
// forward(..., FF_UPDATE_KV_ONLY) once per prompt token).

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static void pf_make_map(CUtensorMap* map, void* base, int rows, int cols) { // f16 [rows][cols], box = 128 rows x 64 columns, 128-byte swizzle
	static EncodeTiledFn encode = nullptr;
	if (!encode) {
		cudaDriverEntryPointQueryResult qres;
		void* fn = nullptr;
		CUDA_CHECK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
		if (!fn || qres != cudaDriverEntryPointSuccess) CALM_FATAL("cuTensorMapEncodeTiled is not available from this driver");
		encode = (EncodeTiledFn)fn;
	}
	const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
	const cuuint64_t strides[1] = {(cuuint64_t)cols * sizeof(__half)};
	const cuuint32_t box[2] = {PF_BK, PF_BN}, estr[2] = {1, 1};
	CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
	                    CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
	if (r != CUDA_SUCCESS) CALM_FATAL("cuTensorMapEncodeTiled failed (%d) for a %d x %d f16 matrix", (int)r, rows, cols);
}

static void pf_reserve(int n) {
	const Config& c = g.cfg;
	int cap = cdiv(n, PF_BN) * PF_BN;
	if (cap <= pf.cap) return;
	if (pf.cap) {
		CUDA_CHECK(cudaStreamSynchronize(g.stream));
		cudaFree(pf.X), cudaFree(pf.Q), cudaFree(pf.Nhi), cudaFree(pf.Nlo), cudaFree(pf.Ahi), cudaFree(pf.Alo), cudaFree(pf.Hhi), cudaFree(pf.Hlo), cudaFree(pf.rope), cudaFree(pf.tokens);
	}
	pf.cap = cap;
	auto zalloc = [&](size_t bytes) {
		void* p = dev_alloc(bytes);
		CUDA_CHECK(cudaMemset(p, 0, bytes)); // padding rows of a partial token tile stay zero
		return p;
	};
	pf.X = (float*)zalloc((size_t)cap * c.dim * sizeof(float));
	pf.Q = (float*)zalloc((size_t)cap * g.q_dim * sizeof(float));
	pf.Nhi = (__half*)zalloc((size_t)cap * c.dim * sizeof(__half)), pf.Nlo = (__half*)zalloc((size_t)cap * c.dim * sizeof(__half));
	pf.Ahi = (__half*)zalloc((size_t)cap * g.q_dim * sizeof(__half)), pf.Alo = (__half*)zalloc((size_t)cap * g.q_dim * sizeof(__half));
	pf.Hhi = (__half*)zalloc((size_t)cap * c.hidden_dim * sizeof(__half)), pf.Hlo = (__half*)zalloc((size_t)cap * c.hidden_dim * sizeof(__half));
	pf.rope = (float2*)zalloc((size_t)cap * (c.head_dim / 2) * sizeof(float2));
	pf.tokens = (int*)zalloc((size_t)cap * sizeof(int));
	pf_make_map(&pf.tmN[0], pf.Nhi, cap, c.dim), pf_make_map(&pf.tmN[1], pf.Nlo, cap, c.dim);
	pf_make_map(&pf.tmA[0], pf.Ahi, cap, g.q_dim), pf_make_map(&pf.tmA[1], pf.Alo, cap, g.q_dim);
	pf_make_map(&pf.tmH[0], pf.Hhi, cap, c.hidden_dim), pf_make_map(&pf.tmH[1], pf.Hlo, cap, c.hidden_dim);
}

// which models the tensor-core pass serves; everything else is fed token by token (still on the GPU)
static bool pf_supported() {
	const Config& c = g.cfg;
	return c.n_experts == 0 && g.tp_world == 1 && c.dim % PF_BM == 0 && g.q_dim % PF_BM == 0 && g.kv_dim % PF_BM == 0 && c.hidden_dim % PF_BM == 0 &&
	       (c.head_dim == 64 || c.head_dim == 128) && !(getenv("CALM_B200_PREFILL") && atoi(getenv("CALM_B200_PREFILL")) == 0);
}

template <int MODE, int DBITS, typename KVT>
static void pf_gemm(const CUtensorMap* tm, const PfGemmArgs& a, int rows, int n) {
	static bool opted = false;
	if (!opted) smem_optin(k_pf_gemm<MODE, DBITS, KVT>, pf_smem_bytes<MODE>()), opted = true;
	same_carveout((const void*)k_pf_gemm<MODE, DBITS, KVT>);
	cudaLaunchConfig_t cfg = {};
	cfg.gridDim = dim3(rows / PF_BM, cdiv(n, PF_BN)), cfg.blockDim = dim3(PF_THREADS), cfg.dynamicSmemBytes = pf_smem_bytes<MODE>(), cfg.stream = g.stream;
	cudaLaunchAttribute at[1];
	at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
	at[0].val.programmaticStreamSerializationAllowed = g.use_pdl ? 1 : 0;
	cfg.attrs = at, cfg.numAttrs = 1;
	CUDA_CHECK(cudaLaunchKernelEx(&cfg, k_pf_gemm<MODE, DBITS, KVT>, tm[0], tm[1], a));
	++g_launches;
}

template <typename KVT, int HD>
static void pf_attn(const PfAttnArgs& a, int n) {
	const dim3 grid(cdiv(n, PFA_WARPS), g.cfg.n_kv_heads);
	if (g.kv_mul % 4 == 0) launch_pdl_grid(k_pf_attn<KVT, HD, 4>, grid, PFA_WARPS * 32, a);
	else if (g.kv_mul % 2 == 0) launch_pdl_grid(k_pf_attn<KVT, HD, 2>, grid, PFA_WARPS * 32, a);
	else launch_pdl_grid(k_pf_attn<KVT, HD, 1>, grid, PFA_WARPS * 32, a);
	++g_launches;
}

template <int DBITS, typename KVT>
static void pf_run(int n, int pos0) {
	const Config& c = g.cfg;
	const Weights& w = g.w;
	const size_t kv_layer = (size_t)c.n_kv_heads * c.seq_len * c.head_dim;
	launch_pdl(k_pf_embed<DBITS>, n, 256, 0, pf.X, (const void*)w.token_embedding_table, (const int*)pf.tokens, n, c.dim);
	launch_pdl(k_pf_rope, cdiv(n * (c.head_dim / 2), 256), 256, 0, pf.rope, (const float*)g.rope_freq, n, c.head_dim / 2, pos0);
	g_launches += 2;
	for (int l = 0; l < c.n_layers; ++l) {
		launch_pdl(k_pf_norm, n, 256, 0, (const float*)pf.X, (const float*)w.rms_att_weight[l], pf.Nhi, pf.Nlo, n, c.dim, c.norm_eps, (int)c.norm_ln);
		++g_launches;
		PfGemmArgs a = {};
		a.n_tokens = n;
		a.w[0] = w.wq[l], a.w[1] = w.wk[l], a.w[2] = w.wv[l], a.K = c.dim;
		a.Q = pf.Q, a.q_dim = g.q_dim, a.kv_dim = g.kv_dim, a.head_dim = c.head_dim, a.seq_len = c.seq_len, a.pos0 = pos0;
		a.bias = w.bqkv[l], a.clip = c.qkv_clip, a.rope = pf.rope;
		a.kc = (KVT*)g.kc + l * kv_layer, a.vc = (KVT*)g.vc + l * kv_layer;
		pf_gemm<PF_QKV, DBITS, KVT>(pf.tmN, a, g.q_dim + 2 * g.kv_dim, n);

		PfAttnArgs aa = {};
		aa.Q = pf.Q, aa.kc = a.kc, aa.vc = a.vc, aa.Ohi = pf.Ahi, aa.Olo = pf.Alo;
		aa.n_tokens = n, aa.pos0 = pos0, aa.seq_len = c.seq_len, aa.q_dim = g.q_dim, aa.kv_mul = g.kv_mul, aa.inv_sqrt_hd = 1.0f / sqrtf((float)c.head_dim);
		if (c.head_dim == 128) pf_attn<KVT, 128>(aa, n);
		else pf_attn<KVT, 64>(aa, n);

		PfGemmArgs b = {};
		b.n_tokens = n, b.w[0] = w.wo[l], b.K = g.q_dim, b.X = pf.X, b.dim = c.dim;
		pf_gemm<PF_WO, DBITS, KVT>(pf.tmA, b, c.dim, n);

		if (!c.norm_par) { // (parallel-norm models reuse the attention-norm output, reference infer.c:417-420)
			launch_pdl(k_pf_norm, n, 256, 0, (const float*)pf.X, (const float*)w.rms_ffn_weight[l], pf.Nhi, pf.Nlo, n, c.dim, c.norm_eps, (int)c.norm_ln);
			++g_launches;
		}
		PfGemmArgs u = {};
		u.n_tokens = n, u.w[0] = w.w1[l], u.w[1] = w.w3[l], u.K = c.dim, u.Hhi = pf.Hhi, u.Hlo = pf.Hlo, u.hidden = c.hidden_dim, u.gelu = c.act_gelu;
		pf_gemm<PF_UP, DBITS, KVT>(pf.tmN, u, c.hidden_dim, n);

		PfGemmArgs d = {};
		d.n_tokens = n, d.w[0] = w.w2[l], d.K = c.hidden_dim, d.X = pf.X, d.dim = c.dim;
		pf_gemm<PF_DOWN, DBITS, KVT>(pf.tmH, d, c.dim, n);
	}
}

// Feed `n` prompt tokens at positions pos0 .. pos0 + n - 1: the KV cache afterwards is what n calls of
// forward_cuda(token, pos, FF_UPDATE_KV_ONLY) leave (within the stated tolerance); no logits, no synchronisation.
// Returns 1 when the tensor-core pass ran, 0 when the tokens were fed one by one (unsupported model shape, MoE, tensor
// parallelism, or a block that would roll the cache over).
extern "C" int forward_prefill_cuda(struct Transformer* transformer, const int* tokens, int n, int pos0) {
	if (n <= 0) return 1;
	check_call(transformer, tokens[0], pos0);
	for (int i = 0; i < n; ++i)
		if (tokens[i] < 0 || tokens[i] >= g.cfg.vocab_size) CALM_FATAL("token %d out of range", tokens[i]);
	if (!pf_supported() || pos0 + n > g.cfg.seq_len) {
		for (int i = 0; i < n; ++i) {
			set_params(tokens[i], pos0 + i, 0);
			launch_token(0);
		}
		return 0;
	}
	const int chunk_cap = 2048;
	for (int o = 0; o < n; o += chunk_cap) {
		const int m = n - o < chunk_cap ? n - o : chunk_cap;
		pf_reserve(m);
		CUDA_CHECK(cudaMemcpyAsync(pf.tokens, tokens + o, (size_t)m * sizeof(int), cudaMemcpyHostToDevice, g.stream));
		const int key = g.w.dbits * 100 + g.kvbits;
		switch (key) {
		case 1616: pf_run<16, __half>(m, pos0 + o); break;
		case 1608: pf_run<16, uint8_t>(m, pos0 + o); break;
		case 816: pf_run<8, __half>(m, pos0 + o); break;
		case 808: pf_run<8, uint8_t>(m, pos0 + o); break;
		case 416: pf_run<4, __half>(m, pos0 + o); break;
		default: pf_run<4, uint8_t>(m, pos0 + o); break;
		}
		CUDA_CHECK(cudaStreamSynchronize(g.stream)); // `tokens` is the caller's memory (pageable): the copy above must have left it
	}
	CUDA_CHECK(cudaGetLastError());
	return 1;
}

// the logits of the last device-resident step (decode_greedy / decode_sample keep them in HBM): copy for tests
extern "C" void calm_b200_read_device_logits(float* out) {
	CUDA_CHECK(cudaMemcpy(out, g.logits_dev, (size_t)g.cfg.vocab_size * sizeof(float), cudaMemcpyDeviceToHost));
}

extern "C" void calm_b200_timer_start(void) {
	CUDA_CHECK(cudaEventRecord(g.timer[0], g.stream));
}

extern "C" float calm_b200_timer_stop(void) {
	CUDA_CHECK(cudaEventRecord(g.timer[1], g.stream));
	CUDA_CHECK(cudaEventSynchronize(g.timer[1]));
	float ms = 0;
	CUDA_CHECK(cudaEventElapsedTime(&ms, g.timer[0], g.timer[1]));
	return ms;
}

extern "C" void* calm_b200_stream(void) {
	return (void*)g.stream;
}

extern "C" uint64_t calm_b200_launch_count(void) {
	return g_launches;
}

extern "C" void calm_b200_read_kv(struct Transformer* transformer, int layer, int kv_pos, float* k_out, float* v_out) {
	(void)transformer;
	const Config& c = g.cfg;
	CUDA_CHECK(cudaStreamSynchronize(g.stream));
	size_t es = g.kvbits / 8;
	std::vector<unsigned char> kb(c.head_dim * es), vb(c.head_dim * es);
	for (int h = 0; h < c.n_kv_heads; ++h) {
		size_t off = (((size_t)layer * c.n_kv_heads + h) * c.seq_len + kv_pos) * c.head_dim * es;
		CUDA_CHECK(cudaMemcpy(kb.data(), (char*)g.kc + off, kb.size(), cudaMemcpyDeviceToHost));
		CUDA_CHECK(cudaMemcpy(vb.data(), (char*)g.vc + off, vb.size(), cudaMemcpyDeviceToHost));
		for (int d = 0; d < c.head_dim; ++d) {
			float kf, vf;
			if (es == 2) {
				kf = __half2float(((__half*)kb.data())[d]);
				vf = __half2float(((__half*)vb.data())[d]);
			} else {
				kf = __half2float(__ushort_as_half((unsigned short)(kb[d] << 8)));
				vf = __half2float(__ushort_as_half((unsigned short)(vb[d] << 8)));
			}
			k_out[h * c.head_dim + d] = kf;
			v_out[h * c.head_dim + d] = vf;
		}
	}
}

extern "C" void calm_b200_fill_kv(struct Transformer* transformer, int n_pos, uint64_t seed) {
	(void)transformer;
	const Config& c = g.cfg;
	size_t lh = (size_t)c.n_layers * c.n_kv_heads;
	if (n_pos > c.seq_len) n_pos = c.seq_len;
	if (g.kvbits == 8)
		k_fill_kv<uint8_t><<<g.sms * 4, 256, 0, g.stream>>>((uint8_t*)g.kc, (uint8_t*)g.vc, lh, c.seq_len, c.head_dim, n_pos, seed);
	else
		k_fill_kv<__half><<<g.sms * 4, 256, 0, g.stream>>>((__half*)g.kc, (__half*)g.vc, lh, c.seq_len, c.head_dim, n_pos, seed);
	++g_launches;
	CUDA_CHECK(cudaStreamSynchronize(g.stream));
}

template <int DBITS>
static float matvec_impl(const void* w_device, const float* x_host, float* y_host, int n, int d, int warmup, int iters) {
	cudaStream_t st;
	CUDA_CHECK(cudaStreamCreate(&st));
	float *x, *y;
	CUDA_CHECK(cudaMalloc(&x, n * sizeof(float)));
	CUDA_CHECK(cudaMalloc(&y, d * sizeof(float)));
	CUDA_CHECK(cudaMemcpy(x, x_host, n * sizeof(float), cudaMemcpyHostToDevice));
	cudaDeviceProp prop;
	CUDA_CHECK(cudaGetDeviceProperties(&prop, g.device));
	g.sms = prop.multiProcessorCount;
	size_t smem = xs_bytes<DBITS>(n);
	smem_optin(k_matvec<DBITS>, smem);
	int cap = max_ctas(k_matvec<DBITS>, 256, smem);
	int grid = imin(cap, cdiv((d + 1) / 2, 8));
	MatvecArgs a{x, w_device, y, n, d};
	cudaEvent_t e0, e1;
	CUDA_CHECK(cudaEventCreate(&e0));
	CUDA_CHECK(cudaEventCreate(&e1));
	for (int i = 0; i < warmup; ++i) k_matvec<DBITS><<<grid, 256, smem, st>>>(a);
	CUDA_CHECK(cudaEventRecord(e0, st));
	for (int i = 0; i < iters; ++i) k_matvec<DBITS><<<grid, 256, smem, st>>>(a);
	CUDA_CHECK(cudaEventRecord(e1, st));
	CUDA_CHECK(cudaEventSynchronize(e1));
	CUDA_CHECK(cudaGetLastError());
	g_launches += warmup + iters;
	float ms = 0;
	CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
	CUDA_CHECK(cudaMemcpy(y_host, y, d * sizeof(float), cudaMemcpyDeviceToHost));
	cudaFree(x), cudaFree(y), cudaEventDestroy(e0), cudaEventDestroy(e1), cudaStreamDestroy(st);
	return iters > 0 ? ms / iters : 0.f;
}

extern "C" float calm_b200_matvec(int dbits, const void* w_device, const float* x_host, float* y_host, int n, int d, int warmup, int iters) {
	select_device();
	if (n % 32) CALM_FATAL("matvec: n must be a multiple of 32");
	switch (dbits) {
	case 16: return matvec_impl<16>(w_device, x_host, y_host, n, d, warmup, iters);
	case 8: return matvec_impl<8>(w_device, x_host, y_host, n, d, warmup, iters);
	case 4: return matvec_impl<4>(w_device, x_host, y_host, n, d, warmup, iters);
	}
	CALM_FATAL("matvec: unsupported dbits %d", dbits);
	return 0.f;
}

// Pull the in-kernel launch stamps (summed on the device by k_stamp_accum) into the per-stage tables.
static void perf_collect() {
	if (!g.stamp_acc) return;
	CUDA_CHECK(cudaStreamSynchronize(g.stream));
	std::vector<unsigned long long> acc(MAX_STAMPS + 2);
	CUDA_CHECK(cudaMemcpy(acc.data(), g.stamp_acc, acc.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
	for (int i = 0; i < ST_COUNT; ++i) g.stage_ms[i] = 0;
	for (int i = 0; i < MAX_STAMPS; ++i) g.stage_ms[g.stamp_stage[i]] += (double)acc[i] / 1e6;
	g.token_span_ms = (double)acc[MAX_STAMPS] / 1e6;
}

extern "C" void calm_b200_set_perf(int on) {
	if (!g.ready) return;
	if (!on) perf_collect();
	g.perf = on != 0;
	if (!on) return;
	CUDA_CHECK(cudaStreamSynchronize(g.stream));
	CUDA_CHECK(cudaMemset(g.stamp_acc, 0, (size_t)(MAX_STAMPS + 2) * sizeof(unsigned long long)));
	for (int i = 0; i < ST_COUNT; ++i) g.stage_ms[i] = 0, g.stage_bytes[i] = 0, g.stage_launches[i] = 0;
	g.perf_runs = 0, g.token_span_ms = 0;
}

extern "C" int calm_b200_stage_stats(int stage, char* name, int name_cap, double* ms_total, double* bytes_total, long* launches) {
	if (stage < 0 || stage >= ST_COUNT) return 0;
	if (name && name_cap > 0) {
		strncpy(name, kStageNames[stage], name_cap - 1);
		name[name_cap - 1] = 0;
	}
	if (g.perf) perf_collect();
	*ms_total = g.stage_ms[stage], *bytes_total = g.stage_bytes[stage], *launches = g.stage_launches[stage];
	return 1;
}

// (debug) the 16 in-kernel timestamps the middle layer's attention kernel left during the last profiled token
extern "C" void calm_b200_debug_stamps(unsigned long long* out16) {
	CUDA_CHECK(cudaStreamSynchronize(g.stream));
	CUDA_CHECK(cudaMemcpy(out16, g.stamps + 2 * (size_t)MAX_STAMPS, 16 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
}

extern "C" double calm_b200_perf_token_ms(void) {
	if (g.perf) perf_collect();
	return g.perf_runs ? g.token_span_ms / g.perf_runs : 0.0;
}

extern "C" void perf_cuda(void) {
	if (!g.ready || !g.perf || g.perf_runs == 0) return;
	perf_collect();
	double total = 0;
	for (int i = 0; i < ST_COUNT; ++i) total += g.stage_ms[i];
	if (total <= 0) return;
	// same shape as the reference's table (infer.cu:761-801); times are first-CTA-start to last-CTA-end of every launch of
	// the production CUDA graph, read from %globaltimer inside the kernels
	printf("\nforward breakdown (over %d runs, avg %.1f usec/run; token span %.1f usec):\n", g.perf_runs, total / g.perf_runs * 1e3, g.token_span_ms / g.perf_runs * 1e3);
	for (int i = 0; i < ST_COUNT; ++i) {
		if (g.stage_ms[i] == 0) continue;
		printf("\t[%d] %16s: %4.1f%%; %8.1f usec/run, %6.1f GB/s\n", i, kStageNames[i], g.stage_ms[i] / total * 100, g.stage_ms[i] / g.perf_runs * 1e3,
		       g.stage_bytes[i] / 1e9 / (g.stage_ms[i] / 1e3));
	}
	fflush(stdout);
}
