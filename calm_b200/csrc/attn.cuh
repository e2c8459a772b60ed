// attn.cuh -- k_attn2: flash-decoding with the KV slice brought into shared memory by bulk TMA copies that are issued
// BEFORE the dependency wait.
//
// Why: the cache prefix of a layer is immutable while k_qkv of the same layer runs (k_qkv only writes slot kv_pos), so the
// attention kernel -- resident early thanks to programmatic dependent launch -- can request its whole K/V slice while the
// q/k/v matvec is still streaming weights.  When the dependency wait returns, the 16.8 MB a Llama-3-8B layer reads at
// position 4095 are already on chip, and what remains on the critical path is q -> scores -> softmax -> values out of
// shared memory (no DRAM round trips) plus the slice merge of stages.cuh (attn_tail).
//
// Work split: unit = kv head x group of HG query heads (as k_attn); the positions of a unit are cut into blocks of
// ATTN2_BP = 16 positions and dealt round-robin to the unit's `nsplit` CTAs (block b belongs to CTA b % nsplit), so the
// split is balanced for every kv_len and does NOT depend on kv_len -- which the pre-wait code only knows as a hint
// (TokenParams may still be about to be rewritten by the previous token's tail; the hint decides what to request early,
// never what is computed).  One mbarrier per block; a 16-position K block and V block are one bulk copy each
// ([position][head_dim] is contiguous per (layer, kv head)).  The slot written this step and the attention sinks that
// k_embed re-rotates are read from global memory after the wait instead of from the early copy.
//
// Lane layout and arithmetic are k_attn's transposing score path: LPP = head_dim / 8 lanes own a position (8 dims per
// lane), P = LPP / HG positions per lane group and step, so the HG * P partial dot products of a step transpose onto the
// LPP lanes of the group (one complete score per lane), the two exponentials are evaluated once per lane, and the
// probabilities are broadcast back for the value accumulation.  Reference arithmetic: infer.c:238-267.
#pragma once

#include "stages.cuh"

#define ATTN2_BP 16   // positions per block (one bulk copy of K, one of V)
#define ATTN2_MAXB 32 // blocks per CTA

// ---- thread-block cluster helpers (the CTAs of a unit form one cluster when CLUSTER: nsplit <= 16)
__device__ __forceinline__ void cluster_sync_all() { // every thread of every CTA of the cluster; release / acquire at cluster scope
	asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
	asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ float ld_dsmem(const float* local_ptr, uint32_t cta_rank) { // the same shared-memory location in CTA `cta_rank` of this cluster
	uint32_t raddr;
	float v;
	asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(raddr) : "r"(smem_u32(local_ptr)), "r"(cta_rank));
	asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(raddr) : "memory");
	return v;
}

#define ATTN2_MAX_CLUSTER 16

// shared memory: K blocks | V blocks | q [HG][head_dim] | merge scratch | this CTA's merged record [HG][head_dim + 2]
template <typename KVT>
__host__ __device__ inline size_t attn2_smem_bytes(int hg, int head_dim, int nbmax, int nsplit) {
	size_t kv = (size_t)2 * nbmax * ATTN2_BP * head_dim * sizeof(KVT);
	size_t scratch = (size_t)(ATTN_THREADS / 32) * hg * (head_dim + 2);
	size_t scratch2 = (size_t)(2 * nsplit + 1) * hg;
	if (scratch2 > scratch) scratch = scratch2;
	return kv + ((size_t)hg * head_dim + scratch + (size_t)hg * (head_dim + 2)) * sizeof(float);
}

// How the slices of a unit are folded (measured on the in-kernel timeline, profiles/README.md round 2: with global partials,
// a grid-scope fence, an atomic counter and a last-CTA pass the fold cost the last CTA 5.5 us of a 15 us kernel):
//   CLUSTER = false (default): every CTA publishes its record as 8-byte {value, epoch} cells -- no fence, no atomic: a reader
//     that sees the epoch sees the value -- and then normalises 1/nsplit of the unit's outputs itself, polling the cells
//     of its peers (all CTAs of the grid are resident, so every cell arrives; a watchdog traps instead of hanging).
//   CLUSTER = true: the nsplit CTAs of a unit are one thread-block cluster and read each other's records through
//     distributed shared memory (measured slower: a 16-CTA cluster waits for 16 free SMs of one GPC; kept selectable).
__device__ __forceinline__ float attn_cell_wait(const unsigned long long* cell, unsigned epoch, int* err) {
	unsigned long long v;
	unsigned spins = 0;
	unsigned long long t0 = 0;
	for (;;) {
		asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(cell) : "memory");
		if ((unsigned)(v >> 32) == epoch) break;
		if ((++spins & 1023) == 0) {
			const unsigned long long now = globaltimer_ns();
			if (!t0) t0 = now;
			if (now - t0 > 5000000000ull) { // 5 s: a slice never arrived -- fail loudly, never hang the GPU
				if (err) *reinterpret_cast<volatile int*>(err) = 9200;
				__threadfence_system();
				__trap();
			}
		}
	}
	return __uint_as_float((unsigned)v);
}

// two adjacent cells (16-byte aligned) with ONE poll: a slice's (m, l)
__device__ __forceinline__ void attn_cell_pair_wait(const unsigned long long* cell, unsigned epoch, int* err, float& v0, float& v1) {
	unsigned long long c0, c1;
	unsigned spins = 0;
	unsigned long long t0 = 0;
	for (;;) {
		asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(c0), "=l"(c1) : "l"(cell) : "memory");
		if ((unsigned)(c0 >> 32) == epoch && (unsigned)(c1 >> 32) == epoch) break;
		if ((++spins & 1023) == 0) {
			const unsigned long long now = globaltimer_ns();
			if (!t0) t0 = now;
			if (now - t0 > 5000000000ull) {
				if (err) *reinterpret_cast<volatile int*>(err) = 9201;
				__threadfence_system();
				__trap();
			}
		}
	}
	v0 = __uint_as_float((unsigned)c0), v1 = __uint_as_float((unsigned)c1);
}

// in-kernel timeline of CTA 0 (first layer only, tools/sweep.py): 0 entry, 1 dependency wait returned, 2 q loaded,
// 3 first block ready, 4 position loop done, 5 record published, 6 every slice's (m, l) in and coefficients formed, 7 outputs
#define ATTN_DBG(i)                                                                    \
	do {                                                                               \
		if (a.dbg && blockIdx.x == 0 && threadIdx.x == 0) a.dbg[i] = globaltimer_ns(); \
	} while (0)

// The fold across the nsplit CTAs of a unit, after this CTA published its record (m, l, acc[HG][HD]) as {value, epoch}
// cells: wait for every slice's (m, l), form one coefficient exp(m_s - M) per (slice, head), and normalise 1/nsplit of
// the unit's outputs.  `myrec` [HG][HD + 2] is this CTA's own record in shared memory, complete before the call.
template <int HG, int HD>
__device__ __forceinline__ void attn_cell_fold(const AttnArgs& a, int unit, int split, int hbase, unsigned epoch, const float* myrec) {
	constexpr int REC = HD + 2;
	__shared__ float mls[ATTN2_MAXB + 4][HG][2]; // (m, l) of every slice, then the coefficient in place  (nsplit <= 36)
	__shared__ float invl[HG];
	const int tid = threadIdx.x, nsplit = a.nsplit;
	const unsigned long long* cells = a.cells + (size_t)unit * nsplit * HG * REC;
	for (int i = tid; i < nsplit * HG; i += ATTN_THREADS) {
		const int s = i / HG, h = i % HG;
		const unsigned long long* c = cells + (size_t)s * HG * REC + h * REC + HD;
		if (s == split) mls[s][h][0] = myrec[h * REC + HD], mls[s][h][1] = myrec[h * REC + HD + 1];
		else attn_cell_pair_wait(c, epoch, a.err, mls[s][h][0], mls[s][h][1]); // (REC and HD are even: the pair is 16-byte aligned)
	}
	__syncthreads();
	__shared__ float cfs[ATTN2_MAXB + 4][HG]; // exp(m_s - M): one exponential per (slice, head), in parallel
	for (int i = tid; i < nsplit * HG; i += ATTN_THREADS) {
		const int s = i / HG, h = i % HG;
		float M = -FLT_MAX;
		for (int s2 = 0; s2 < nsplit; ++s2) M = fmaxf(M, mls[s2][h][0]);
		cfs[s][h] = expf(mls[s][h][0] - M);
	}
	__syncthreads();
	if (tid < HG) {
		float L = 0.f;
		for (int s = 0; s < nsplit; ++s) L = fmaf(mls[s][tid][1], cfs[s][tid], L); // slice order: deterministic
		invl[tid] = 1.0f / L;
	}
	for (int i = tid; i < nsplit * HG; i += ATTN_THREADS) mls[i / HG][i % HG][0] = cfs[i / HG][i % HG]; // the output loop reads the coefficient from mls
	__syncthreads();
	ATTN_DBG(6);
	// CTA `split` normalises outputs [split * per, (split + 1) * per): 8 adjacent lanes share an output, each sums every 8th slice
	const int nout = HG * HD, per = (nout + nsplit - 1) / nsplit;
	const int o_end = min(nout, (split + 1) * per);
	for (int o0 = split * per; o0 < o_end; o0 += ATTN_THREADS / 8) {
		const int o = o0 + tid / 8, sg = tid & 7;
		float v = 0.f;
		if (o < o_end) {
			const int h = o / HD, e = o % HD;
			// all of this lane's cells are requested before the first is looked at (their slices' (m, l) have been seen: they are
			// almost always there) -- one L2 round trip instead of one per slice; a cell that is not there yet is polled as before
			constexpr int NS8 = (ATTN2_MAXB + 4 + 7) / 8;
			unsigned long long c[NS8];
#pragma unroll
			for (int k = 0; k < NS8; ++k) {
				const int s = sg + 8 * k;
				c[k] = 0;
				if (s < nsplit && s != split) asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(c[k]) : "l"(cells + (size_t)s * HG * REC + h * REC + e) : "memory");
			}
#pragma unroll
			for (int k = 0; k < NS8; ++k) {
				const int s = sg + 8 * k;
				if (s < nsplit) {
					float x;
					if (s == split) x = myrec[h * REC + e];
					else if ((unsigned)(c[k] >> 32) == epoch) x = __uint_as_float((unsigned)c[k]);
					else x = attn_cell_wait(cells + (size_t)s * HG * REC + h * REC + e, epoch, a.err);
					v = fmaf(x, mls[s][h][0], v); // slice order per lane: deterministic
				}
			}
		}
		v += __shfl_xor_sync(0xffffffffu, v, 1), v += __shfl_xor_sync(0xffffffffu, v, 2), v += __shfl_xor_sync(0xffffffffu, v, 4);
		if (o < o_end && sg == 0) __stcg(a.out + (size_t)hbase * HD + o, v * invl[o / HD]);
	}
}

template <typename KVT, int HG, int LPP, bool CLUSTER>
__global__ void __launch_bounds__(ATTN_THREADS) k_attn2(const AttnArgs a) {
	typedef typename KvRaw<KVT>::type raw_t;
	constexpr int HD = LPP * 8, P = LPP / HG, G = 32 / LPP, NW = ATTN_THREADS / 32, NC = LPP;
	static_assert(HG * P == LPP && P >= 1 && P <= 4 && ATTN2_BP % P == 0, "unsupported head grouping");
	extern __shared__ __align__(128) unsigned char smem_raw[];
	__shared__ __align__(8) uint64_t bars[ATTN2_MAXB];
	__shared__ int flag;
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const int nbmax = a.nbmax, nsplit = a.nsplit;
	const int unit = blockIdx.x / nsplit, split = blockIdx.x % nsplit;
	const int kvh = unit / a.qgroups;
	const int hbase = kvh * a.kv_mul + (unit % a.qgroups) * HG;
	constexpr uint32_t BLK = ATTN2_BP * HD * sizeof(KVT); // bytes of a whole block
	KVT* Ks = reinterpret_cast<KVT*>(smem_raw);
	KVT* Vs = Ks + (size_t)nbmax * ATTN2_BP * HD;
	float* qs = reinterpret_cast<float*>(Vs + (size_t)nbmax * ATTN2_BP * HD);
	float* scratch = qs + HG * HD;
	float* myrec = scratch + max(NW * HG * (HD + 2), (2 * nsplit + 1) * HG); // [HG][HD + 2]
	const KVT* kglob = reinterpret_cast<const KVT*>(a.kc) + (size_t)kvh * a.seq_len * HD;
	const KVT* vglob = reinterpret_cast<const KVT*>(a.vc) + (size_t)kvh * a.seq_len * HD;

	ATTN_DBG(0);
	pdl_launch_next();
	if (tid == 0) {
		for (int j = 0; j < nbmax; ++j) mbar_init(&bars[j], 1);
		mbar_init_fence();
	}
	__syncthreads();
	// request the slice while the previous kernel (k_qkv of this layer) is still running: thread j owns block j
	bool issued = false;
	auto request = [&](int j) {
		const int b = split + j * nsplit;
		const uint32_t bytes = (uint32_t)min(ATTN2_BP, a.seq_len - b * ATTN2_BP) * HD * sizeof(KVT);
		mbar_expect_tx(&bars[j], 2 * bytes);
		tma_load_1d(Ks + (size_t)j * ATTN2_BP * HD, kglob + (size_t)b * ATTN2_BP * HD, bytes, &bars[j]);
		tma_load_1d(Vs + (size_t)j * ATTN2_BP * HD, vglob + (size_t)b * ATTN2_BP * HD, bytes, &bars[j]);
	};
	if (tid < nbmax) {
		const int hint = min(*reinterpret_cast<const volatile int*>(&a.tp->kv_len), a.seq_len);
		if ((split + tid * nsplit) * ATTN2_BP < hint) request(tid), issued = true;
	}
	pdl_wait_prev();
	stamp_begin(a.stamp);
	ATTN_DBG(1);
	if (a.dbg && tid == 0) atomicMin(a.dbg + 10, globaltimer_ns());
	// q and the token parameters are requested together (one L2 round trip, not two)
	constexpr int QPT = (HG * HD + ATTN_THREADS - 1) / ATTN_THREADS;
	float qreg[QPT];
#pragma unroll
	for (int i = 0; i < QPT; ++i) qreg[i] = (tid + i * ATTN_THREADS < HG * HD) ? __ldcg(a.q + (size_t)hbase * HD + tid + i * ATTN_THREADS) : 0.f;
	const int kv_len = a.tp->kv_len, kv_pos = a.tp->kv_pos, kv_sink = a.tp->kv_sink;
	const unsigned epoch = (unsigned)a.tp->tp_seq * a.epoch_stride + a.epoch_idx;
	if (tid < nbmax && !issued && (split + tid * nsplit) * ATTN2_BP < kv_len) request(tid), issued = true;
#pragma unroll
	for (int i = 0; i < QPT; ++i)
		if (tid + i * ATTN_THREADS < HG * HD) qs[tid + i * ATTN_THREADS] = qreg[i];
	__syncthreads();
	ATTN_DBG(2);

	// blocks of this CTA that hold cached positions
	const int nblk = (kv_len + ATTN2_BP - 1) / ATTN2_BP;
	const int nb = nblk > split ? (nblk - split + nsplit - 1) / nsplit : 0;
	const int nslots = nb * ATTN2_BP;
	const int grp = lane / LPP, li = lane % LPP;

	float acc[HG][8], m[HG], l[HG];
#pragma unroll
	for (int h = 0; h < HG; ++h) {
		m[h] = -FLT_MAX, l[h] = 0.f;
#pragma unroll
		for (int d = 0; d < 8; ++d) acc[h][d] = 0.f;
	}
	float mh = -FLT_MAX, lh = 0.f; // running max / sum of THIS lane's head (li / P)

	// Steps are taken SC at a time: first ALL scores of the chunk (independent dot products and transposing reductions: no
	// serial softmax state between them), then one max / exp / sum for the chunk, then the value pass.  With 8 warps per SM
	// the per-step online softmax was a latency chain (5 us for 4 steps on the in-kernel timeline); this form rescales the
	// accumulators once per chunk.
	constexpr int SC = 4, STEP = NW * G * P;
	const int gbase = grp * LPP;
	auto slot_of = [&](int s0, int& j, int& o, int& t0) {
		j = s0 / ATTN2_BP, o = s0 % ATTN2_BP;
		t0 = (split + j * nsplit) * ATTN2_BP + o;
	};
	for (int sb = (warp * G + grp) * P; sb - grp * P < nslots; sb += SC * STEP) { // warp-uniform trip count (full-warp shuffles inside)
		float sc[SC];
		bool val[SC], fast[SC];
#pragma unroll
		for (int c = 0; c < SC; ++c) {
			const int s0 = sb + c * STEP;
			const bool inr = s0 < nslots;
			int j = 0, o = 0, t0 = 0;
			if (inr) slot_of(s0, j, o, t0);
			if (inr) mbar_wait(&bars[j], 0);
			if (s0 == 0) ATTN_DBG(3);
			// the common case for a whole warp -- P cached positions, none of them written during this token -- needs no per-position tests
			fast[c] = __all_sync(0xffffffffu, inr && t0 + P <= kv_len && (kv_pos < t0 || kv_pos >= t0 + P) && t0 >= kv_sink);
			float part[NC]; // combo h * P + i: partial dot product of this lane's 8 dims
			{
				float kf[P][8];
				if (fast[c]) {
					const KVT* kp = Ks + ((size_t)j * ATTN2_BP + o) * HD + li * 8;
#pragma unroll
					for (int i = 0; i < P; ++i) KvRaw<KVT>::unpack(*reinterpret_cast<const raw_t*>(kp + i * HD), kf[i]);
				} else {
#pragma unroll
					for (int i = 0; i < P; ++i) {
						const int t = t0 + i;
						raw_t kr = KvRaw<KVT>::zero();
						if (inr && t < kv_len)
							kr = (t == kv_pos || t < kv_sink) ? KvRaw<KVT>::load(kglob + (size_t)t * HD + li * 8) // written during this token: not in the early copy
							                                  : *reinterpret_cast<const raw_t*>(Ks + ((size_t)j * ATTN2_BP + o + i) * HD + li * 8);
						KvRaw<KVT>::unpack(kr, kf[i]);
					}
				}
#pragma unroll
				for (int h = 0; h < HG; ++h) {
					const float4 q0 = *reinterpret_cast<const float4*>(qs + h * HD + li * 8), q1 = *reinterpret_cast<const float4*>(qs + h * HD + li * 8 + 4);
#pragma unroll
					for (int i = 0; i < P; ++i) {
						float d = q0.x * kf[i][0];
						d = fmaf(q0.y, kf[i][1], d), d = fmaf(q0.z, kf[i][2], d), d = fmaf(q0.w, kf[i][3], d);
						d = fmaf(q1.x, kf[i][4], d), d = fmaf(q1.y, kf[i][5], d), d = fmaf(q1.z, kf[i][6], d), d = fmaf(q1.w, kf[i][7], d);
						part[h * P + i] = d;
					}
				}
			}
			// transposing reduction over the LPP lanes of the group: after the step with stride s a lane keeps the half selected by bit s
#pragma unroll
			for (int s_ = NC / 2; s_ >= 1; s_ >>= 1) {
				const bool up = li & s_;
#pragma unroll
				for (int k = 0; k < s_; ++k) {
					float send = up ? part[k] : part[k + s_];
					float recv = __shfl_xor_sync(0xffffffffu, send, s_);
					part[k] = (up ? part[k + s_] : part[k]) + recv;
				}
			}
			// lane li owns combo li: head li / P, position li % P
			val[c] = inr && (t0 + li % P) < kv_len;
			sc[c] = val[c] ? part[0] * a.inv_sqrt_hd : -FLT_MAX;
		}
		float gmax = sc[0];
#pragma unroll
		for (int c = 1; c < SC; ++c) gmax = fmaxf(gmax, sc[c]);
#pragma unroll
		for (int o2 = 1; o2 < P; o2 <<= 1) gmax = fmaxf(gmax, __shfl_xor_sync(0xffffffffu, gmax, o2));
		const float mnew = fmaxf(mh, gmax);
		const float corr = __expf(mh - mnew);
		float pr[SC], ps = 0.f;
#pragma unroll
		for (int c = 0; c < SC; ++c) pr[c] = val[c] ? __expf(sc[c] - mnew) : 0.f, ps += pr[c];
#pragma unroll
		for (int o2 = 1; o2 < P; o2 <<= 1) ps += __shfl_xor_sync(0xffffffffu, ps, o2);
		lh = fmaf(lh, corr, ps);
		mh = mnew;
#pragma unroll
		for (int h = 0; h < HG; ++h) {
			const float ch = __shfl_sync(0xffffffffu, corr, gbase + h * P);
#pragma unroll
			for (int e = 0; e < 8; ++e) acc[h][e] *= ch;
		}
#pragma unroll
		for (int c = 0; c < SC; ++c) {
			const int s0 = sb + c * STEP;
			const bool inr = s0 < nslots;
			int j = 0, o = 0, t0 = 0;
			if (inr) slot_of(s0, j, o, t0);
			float vf[P][8];
			if (fast[c]) {
				const KVT* vp = Vs + ((size_t)j * ATTN2_BP + o) * HD + li * 8;
#pragma unroll
				for (int i = 0; i < P; ++i) KvRaw<KVT>::unpack(*reinterpret_cast<const raw_t*>(vp + i * HD), vf[i]);
			} else {
#pragma unroll
				for (int i = 0; i < P; ++i) {
					const int t = t0 + i;
					raw_t vr = KvRaw<KVT>::zero();
					if (inr && t < kv_len)
						vr = (t == kv_pos || t < kv_sink) ? KvRaw<KVT>::load(vglob + (size_t)t * HD + li * 8)
						                                  : *reinterpret_cast<const raw_t*>(Vs + ((size_t)j * ATTN2_BP + o + i) * HD + li * 8);
					KvRaw<KVT>::unpack(vr, vf[i]);
				}
			}
#pragma unroll
			for (int h = 0; h < HG; ++h) {
				float pw[P];
#pragma unroll
				for (int i = 0; i < P; ++i) pw[i] = __shfl_sync(0xffffffffu, pr[c], gbase + h * P + i);
#pragma unroll
				for (int e = 0; e < 8; ++e) {
					float v = acc[h][e];
#pragma unroll
					for (int i = 0; i < P; ++i) v = fmaf(pw[i], vf[i][e], v);
					acc[h][e] = v;
				}
			}
		}
	}
	ATTN_DBG(4);
#pragma unroll
	for (int h = 0; h < HG; ++h) { // running max / sum live in the lanes that own the head: hand them to every lane of the group
		m[h] = __shfl_sync(0xffffffffu, mh, grp * LPP + h * P);
		l[h] = __shfl_sync(0xffffffffu, lh, grp * LPP + h * P);
	}
	if constexpr (CLUSTER) {
		constexpr int REC = HD + 2;
		__shared__ float mls[ATTN2_MAX_CLUSTER][HG][2]; // (m, l) of every slice, then (coefficient, -) in place
		__shared__ float invl[HG];
		attn_cta_merge<HG>(a, HG, 0, HG, warp, NW, m, l, acc, scratch, myrec);
		cluster_sync_all(); // every CTA's record is complete and visible cluster-wide
		for (int i = tid; i < nsplit * HG; i += ATTN_THREADS) {
			const int s = i / HG, h = i % HG;
			mls[s][h][0] = ld_dsmem(myrec + h * REC + HD, s), mls[s][h][1] = ld_dsmem(myrec + h * REC + HD + 1, s);
		}
		__syncthreads();
		if (tid < HG) {
			float M = -FLT_MAX;
			for (int s = 0; s < nsplit; ++s) M = fmaxf(M, mls[s][tid][0]);
			float L = 0.f;
			for (int s = 0; s < nsplit; ++s) {
				const float c = expf(mls[s][tid][0] - M);
				L = fmaf(mls[s][tid][1], c, L);
				mls[s][tid][0] = c;
			}
			invl[tid] = 1.0f / L;
		}
		__syncthreads();
		// CTA `split` normalises outputs [split * per, (split + 1) * per): 8 adjacent lanes share an output, each sums every 8th slice
		const int nout = HG * HD, per = (nout + nsplit - 1) / nsplit;
		const int o_end = min(nout, (split + 1) * per);
		for (int o0 = split * per; o0 < o_end; o0 += ATTN_THREADS / 8) {
			const int o = o0 + tid / 8, sg = tid & 7;
			float v = 0.f;
			if (o < o_end) {
				const int h = o / HD, e = o % HD;
				for (int s = sg; s < nsplit; s += 8) v = fmaf(ld_dsmem(myrec + h * REC + e, s), mls[s][h][0], v);
			}
			v += __shfl_xor_sync(0xffffffffu, v, 1), v += __shfl_xor_sync(0xffffffffu, v, 2), v += __shfl_xor_sync(0xffffffffu, v, 4);
			if (o < o_end && sg == 0) __stcg(a.out + (size_t)hbase * HD + o, v * invl[o / HD]);
		}
		cluster_sync_all(); // no CTA may exit (and free its shared memory) while a peer still reads its record
	} else {
		constexpr int REC = HD + 2;
		(void)flag;
		attn_cta_merge<HG>(a, HG, 0, HG, warp, NW, m, l, acc, scratch, myrec);
		__syncthreads();
		ATTN_DBG(5);
		unsigned long long* cells = a.cells + (size_t)unit * nsplit * HG * REC;
		for (int i = tid; i < HG * REC; i += ATTN_THREADS) { // publish: ONE 8-byte store per value
			const unsigned long long c = ((unsigned long long)epoch << 32) | __float_as_uint(myrec[i]);
			asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(cells + (size_t)split * HG * REC + i), "l"(c) : "memory");
		}
		attn_cell_fold<HG, HD>(a, unit, split, hbase, epoch, myrec);
	}
	// no bulk copy may still be in flight into this CTA's shared memory when it exits (a block requested on a stale hint)
	if (tid < nbmax && issued) mbar_wait(&bars[tid], 0);
	ATTN_DBG(7);
	if (a.dbg && tid == 0) atomicMax(a.dbg + 9, globaltimer_ns());
	stamp_end(a.stamp);
}

// ---------------------------------------------------------------------------------------------------------------------
// k_attn_mma: the same units, slices, early bulk copies and cell fold as k_attn2, for head_dim 128 with 4 query heads per
// kv head; scores and values on mma.sync.m16n8k16 (f16 in, f32 accumulate), softmax once per CTA.
//
//   scores  S = K.Q per 16-position block: A = 16 positions x 16 dims of K (f16; e5m2 is the high byte of an f16, so one
//           PRMT makes a pair exact), B = 16 dims x 8 columns {hi, lo} of the 4 query heads, q * 2^e = hi + lo in f16 with
//           a power of two per head that puts max |q| at [2^14, 2^15).  f16 x f16 products are exact in f32, so what
//           differs from the SIMT path is the summation order and q carried to 22 bits.  Warps take the CTA's blocks.
//   softmax every score of the CTA lands in shared memory; m and l per head over all of them, p = exp(s - m) as f16
//           hi + lo (p to 22 bits; the sum l is taken in f32).
//   values  warp w owns dims [16w, 16w + 16) over all of the CTA's positions: out^T = V^T.P with A = V^T (16 dims x 16
//           positions) and B = P (16 positions x {hi, lo} of the 4 heads).  The CTA's record (m, l, acc[4][128]) is then
//           two values per thread, published straight into the cells: no merge of per-warp records.
//
// Shared-memory banks: a K or V row is 256 B (fp16), so eight rows of one block at the same dims fall on the same four
// banks and every fragment load would conflict 8 ways.  Each row is therefore its own bulk copy into a row stride of
// 256 + 16 B (e5m2: 128 + 16 B): eight consecutive rows then cover all 32 banks for ldmatrix (fp16 K and V, e5m2 K) and
// for the 16-bit loads of e5m2 V.
//
// Fragment layouts (lane = 4 g + t): with e5m2 K, ldmatrix returns 4 consecutive dims of one row per lane, so the 16
// dims of a k-step are taken in the order {4t, 4t+1 | 4t+2, 4t+3} instead of {2t, 2t+1 | 2t+8, 2t+9}; q is loaded in
// the same order and the dot product does not see it.  With e5m2 V, output row g / g + 8 of a warp's tile is dim 2g /
// 2g + 1 (fp16: g / g + 8).
#define ATTN_MMA_HG 4
#define ATTN_MMA_HD 128

template <typename KVT>
struct AttnMmaShape {
	static constexpr int ROWB = ATTN_MMA_HD * (int)sizeof(KVT); // bytes of one cached row
	static constexpr int KST = ROWB + 16;                         // its stride in shared memory
};

// shared memory: K blocks | V blocks | scores [HG][sst] | probabilities [2 HG][pst] (f16 pairs) | this CTA's record [HG][HD + 2]
__host__ __device__ inline int attn_mma_sst(int nbmax) { return (nbmax * ATTN2_BP + 31) / 32 * 32 + 8; }     // == 8 mod 32: score stores conflict-free
__host__ __device__ inline int attn_mma_pst(int nbmax) { return (nbmax * ATTN2_BP / 2 + 31) / 32 * 32 + 4; } // == 4 mod 32: B fragments conflict-free
template <typename KVT>
__host__ __device__ inline size_t attn_mma_smem_bytes(int nbmax) {
	return (size_t)2 * nbmax * ATTN2_BP * AttnMmaShape<KVT>::KST +
	       ((size_t)ATTN_MMA_HG * attn_mma_sst(nbmax) + (size_t)2 * ATTN_MMA_HG * attn_mma_pst(nbmax) + (size_t)ATTN_MMA_HG * (ATTN_MMA_HD + 2)) * sizeof(float);
}

__device__ __forceinline__ void mma_f16_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
	asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
	             : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
	             : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], const void* p) {
	asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(smem_u32(p)));
}
__device__ __forceinline__ void ldsm_x4_trans(uint32_t (&r)[4], const void* p) {
	asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(smem_u32(p)));
}
__device__ __forceinline__ uint32_t pack_half2(__half lo, __half hi) {
	return (uint32_t)__half_as_ushort(lo) | ((uint32_t)__half_as_ushort(hi) << 16);
}

template <typename KVT>
__global__ void __launch_bounds__(ATTN_THREADS, 1) k_attn_mma(const AttnArgs a) {
	constexpr int HG = ATTN_MMA_HG, HD = ATTN_MMA_HD, BP = ATTN2_BP, NW = ATTN_THREADS / 32, REC = HD + 2;
	constexpr bool F16 = sizeof(KVT) == 2;
	constexpr int ROWB = AttnMmaShape<KVT>::ROWB, KST = AttnMmaShape<KVT>::KST;
	static_assert(NW * 16 == HD, "one warp per 16 output dims");
	extern __shared__ __align__(128) unsigned char smem_raw[];
	__shared__ __align__(8) uint64_t bars[ATTN2_MAXB];
	__shared__ int s_hint;
	__shared__ float s_m[HG], s_l[NW];
	__shared__ __align__(16) float s_q[HG * HD];
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
	const int nbmax = a.nbmax, nsplit = a.nsplit, seq_len = a.seq_len;
	const int unit = blockIdx.x / nsplit, split = blockIdx.x % nsplit;
	const int kvh = unit / a.qgroups;
	const int hbase = kvh * a.kv_mul + (unit % a.qgroups) * HG;
	const int sst = attn_mma_sst(nbmax), pst = attn_mma_pst(nbmax);
	unsigned char* Ks = smem_raw;
	unsigned char* Vs = Ks + (size_t)nbmax * BP * KST;
	float* sc = reinterpret_cast<float*>(Vs + (size_t)nbmax * BP * KST); // [HG][sst]
	uint32_t* ph = reinterpret_cast<uint32_t*>(sc + HG * sst);           // [2 HG][pst]: column 2h = hi, 2h + 1 = lo halves of p, position pairs
	float* myrec = reinterpret_cast<float*>(ph + 2 * HG * pst);          // [HG][REC]
	const unsigned char* kglob = reinterpret_cast<const unsigned char*>(a.kc) + (size_t)kvh * seq_len * ROWB;
	const unsigned char* vglob = reinterpret_cast<const unsigned char*>(a.vc) + (size_t)kvh * seq_len * ROWB;

	ATTN_DBG(0);
	pdl_launch_next();
	if (tid == 0) {
		for (int j = 0; j < nbmax; ++j) mbar_init(&bars[j], 1);
		mbar_init_fence();
		s_hint = min(*reinterpret_cast<const volatile int*>(&a.tp->kv_len), seq_len); // ONE read: every thread of a block agrees on it
	}
	__syncthreads();
	// block j (cache block split + j * nsplit) is 16 row copies of K and 16 of V; thread (j, r) issues row r
	auto request_row = [&](int j, int r) {
		const int b = split + j * nsplit;
		const int rows = min(BP, seq_len - b * BP);
		if (r == 0) mbar_expect_tx(&bars[j], (uint32_t)(2 * rows * ROWB));
		if (r < rows) {
			const size_t src = ((size_t)b * BP + r) * ROWB, dst = ((size_t)j * BP + r) * KST;
			tma_load_1d(Ks + dst, kglob + src, ROWB, &bars[j]);
			tma_load_1d(Vs + dst, vglob + src, ROWB, &bars[j]);
		}
	};
	const int hint = s_hint;
	auto early = [&](int j) { return (split + j * nsplit) * BP < hint; };
	for (int i = tid; i < nbmax * BP; i += ATTN_THREADS)
		if (early(i / BP)) request_row(i / BP, i % BP);
	pdl_wait_prev();
	stamp_begin(a.stamp);
	ATTN_DBG(1);
	if (a.dbg && tid == 0) atomicMin(a.dbg + 10, globaltimer_ns());

	// the CTA's 4 query heads (one coalesced 8-byte load per thread: every q line is read once per CTA, not once per warp),
	// requested with the token parameters
	static_assert(HG * HD == 2 * ATTN_THREADS, "one float2 of q per thread");
	const float2 qg = __ldcg(reinterpret_cast<const float2*>(a.q + (size_t)hbase * HD) + tid);
	const int kv_len = a.tp->kv_len, kv_pos = a.tp->kv_pos, kv_sink = a.tp->kv_sink;
	const unsigned epoch = (unsigned)a.tp->tp_seq * a.epoch_stride + a.epoch_idx;
	auto needed = [&](int j) { return (split + j * nsplit) * BP < kv_len; };
	for (int i = tid; i < nbmax * BP; i += ATTN_THREADS)
		if (!early(i / BP) && needed(i / BP)) request_row(i / BP, i % BP);
	reinterpret_cast<float2*>(s_q)[tid] = qg;
	__syncthreads();
	// q as B fragments (column g: head g / 2, hi or lo half by g & 1)
	const int qh = g >> 1;
	float2 qv[8][2];
#pragma unroll
	for (int kk = 0; kk < 8; ++kk) {
		const int d0 = F16 ? 16 * kk + 2 * t : 16 * kk + 4 * t, d1 = F16 ? d0 + 8 : d0 + 2;
		qv[kk][0] = *reinterpret_cast<const float2*>(s_q + qh * HD + d0);
		qv[kk][1] = *reinterpret_cast<const float2*>(s_q + qh * HD + d1);
	}
	uint32_t qb[8][2];
	int qexp; // max |q of this head| = f * 2^qexp, f in [0.5, 1): q * 2^(15 - qexp) is below 2^15
	{
		float mx = 0.f;
#pragma unroll
		for (int kk = 0; kk < 8; ++kk)
			mx = fmaxf(mx, fmaxf(fmaxf(fabsf(qv[kk][0].x), fabsf(qv[kk][0].y)), fmaxf(fabsf(qv[kk][1].x), fabsf(qv[kk][1].y))));
		mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1)), mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2)); // the 4 lanes of column g hold all 128 dims
		frexpf(mx, &qexp);
		qexp = max(-100, min(qexp, 100));
		const float s = ldexpf(1.f, 15 - qexp);
		auto split_q = [&](float x) { // the hi or lo f16 part of x * s
			const float y = x * s;
			const __half hi = __float2half_rn(y);
			return (g & 1) ? __float2half_rn(y - __half2float(hi)) : hi;
		};
#pragma unroll
		for (int kk = 0; kk < 8; ++kk)
#pragma unroll
			for (int i = 0; i < 2; ++i) qb[kk][i] = pack_half2(split_q(qv[kk][i].x), split_q(qv[kk][i].y));
	}
	// score of head t: C * 2^(qexp - 15) (exact) * 1/sqrt(head_dim); column 2t's lanes (g = 2t) hold that head's exponent
	const float sunscale = ldexpf(1.f, __shfl_sync(0xffffffffu, qexp, 8 * t) - 15);
	ATTN_DBG(2);

	const int nblk = (kv_len + BP - 1) / BP;
	const int nb = nblk > split ? (nblk - split + nsplit - 1) / nsplit : 0;
	const int nslots = nb * BP;

	// ---- scores: warp w takes blocks w, w + NW, ...
	for (int j = warp; j < nb; j += NW) {
		mbar_wait(&bars[j], 0);
		if (j == 0) ATTN_DBG(3);
		const int p0 = (split + j * nsplit) * BP;
		unsigned char* kb = Ks + (size_t)j * BP * KST;
		unsigned char* vb = Vs + (size_t)j * BP * KST;
		// rows written during this token (slot kv_pos, the re-rotated sinks) come from global memory; rows past kv_len are
		// zeroed (p = 0 there, and 0 * whatever the row held must stay 0)
		if ((kv_pos >= p0 && kv_pos < p0 + BP) || p0 < kv_sink || p0 + BP > kv_len) {
			for (int o = 0; o < BP; ++o) {
				const int pos = p0 + o;
				const bool fresh = pos < kv_len && (pos == kv_pos || pos < kv_sink), past = pos >= kv_len;
				if ((fresh || past) && lane < ROWB / 16) {
					uint4 kr = make_uint4(0, 0, 0, 0), vr = kr;
					if (fresh) {
						kr = __ldcg(reinterpret_cast<const uint4*>(kglob + (size_t)pos * ROWB) + lane);
						vr = __ldcg(reinterpret_cast<const uint4*>(vglob + (size_t)pos * ROWB) + lane);
					}
					reinterpret_cast<uint4*>(kb + o * KST)[lane] = kr;
					reinterpret_cast<uint4*>(vb + o * KST)[lane] = vr;
				}
			}
			__syncwarp();
		}
		float c[4] = {0.f, 0.f, 0.f, 0.f};
		if constexpr (F16) {
			// matrices: rows 0-7 / 8-15 x dims 16kk + 0-7, then the same rows x dims 16kk + 8-15
			const unsigned char* base = kb + ((lane & 7) + ((lane >> 3) & 1) * 8) * KST + (lane >> 4) * 16;
#pragma unroll
			for (int kk = 0; kk < 8; ++kk) {
				uint32_t af[4];
				ldsm_x4(af, base + kk * 32);
				mma_f16_16816(c, af, qb[kk][0], qb[kk][1]);
			}
		} else {
			// matrices: rows 0-7 / 8-15 x bytes (dims) 16s + 0-15, then the same rows x 16(s + 1) + 0-15: two k-steps
			const unsigned char* base = kb + ((lane & 7) + ((lane >> 3) & 1) * 8) * KST + (lane >> 4) * 16;
#pragma unroll
			for (int s2 = 0; s2 < 4; ++s2) {
				uint32_t r[4];
				ldsm_x4(r, base + s2 * 32);
#pragma unroll
				for (int h = 0; h < 2; ++h) {
					const uint32_t af[4] = {__byte_perm(0u, r[2 * h], 0x5040), __byte_perm(0u, r[2 * h + 1], 0x5040), __byte_perm(0u, r[2 * h], 0x7060),
					                        __byte_perm(0u, r[2 * h + 1], 0x7060)};
					mma_f16_16816(c, af, qb[2 * s2 + h][0], qb[2 * s2 + h][1]);
				}
			}
		}
		// lane (g, t): head t at positions g and g + 8 of the block
#pragma unroll
		for (int i = 0; i < 2; ++i) {
			const int o = g + 8 * i;
			sc[t * sst + j * BP + o] = p0 + o < kv_len ? (c[2 * i] + c[2 * i + 1]) * sunscale * a.inv_sqrt_hd : -FLT_MAX;
		}
	}
	__syncthreads();

	// ---- softmax over the CTA's positions: warps h and h + 4 take head h (both form m, each half of the pairs)
	{
		const int h = warp & 3, half = warp >> 2;
		const float* sh = sc + h * sst;
		float m = -FLT_MAX;
		for (int i = lane; i < nslots; i += 32) m = fmaxf(m, sh[i]);
#pragma unroll
		for (int o = 16; o >= 1; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
		float ls = 0.f;
		for (int i = half * 32 + lane; i < nslots / 2; i += 64) {
			const float2 s2 = *reinterpret_cast<const float2*>(sh + 2 * i);
			const float e0 = __expf(s2.x - m), e1 = __expf(s2.y - m);
			ls += e0 + e1;
			const __half h0 = __float2half_rn(e0), h1 = __float2half_rn(e1);
			ph[(2 * h) * pst + i] = pack_half2(h0, h1);
			ph[(2 * h + 1) * pst + i] = pack_half2(__float2half_rn(e0 - __half2float(h0)), __float2half_rn(e1 - __half2float(h1)));
		}
#pragma unroll
		for (int o = 16; o >= 1; o >>= 1) ls += __shfl_xor_sync(0xffffffffu, ls, o);
		if (lane == 0) {
			s_l[warp] = ls;
			if (half == 0) s_m[h] = m;
		}
	}
	__syncthreads();

	// ---- values: warp w owns dims [16w, 16w + 16); two accumulator chains (even / odd blocks)
	float acc0[4] = {0.f, 0.f, 0.f, 0.f}, acc1[4] = {0.f, 0.f, 0.f, 0.f};
	auto pv = [&](int j, float (&acc)[4]) {
		const unsigned char* vb = Vs + (size_t)j * BP * KST;
		uint32_t af[4];
		if constexpr (F16) {
			// matrices (transposed): positions 0-7 x dims 0-7, 0-7 x 8-15, 8-15 x 0-7, 8-15 x 8-15 of the warp's 16 dims
			ldsm_x4_trans(af, vb + ((lane & 7) + (lane >> 4) * 8) * KST + (16 * warp + ((lane >> 3) & 1) * 8) * 2);
		} else {
			// rows g / g + 8 of the tile are dims 2g / 2g + 1: one 16-bit load per position, two positions per PRMT
			const unsigned char* col = vb + 16 * warp + 2 * g;
			uint32_t x[4];
#pragma unroll
			for (int i = 0; i < 4; ++i) x[i] = *reinterpret_cast<const unsigned short*>(col + (2 * t + (i & 1) + 8 * (i >> 1)) * KST);
			af[0] = __byte_perm(x[0], x[1], 0x4202), af[1] = __byte_perm(x[0], x[1], 0x5212);
			af[2] = __byte_perm(x[2], x[3], 0x4202), af[3] = __byte_perm(x[2], x[3], 0x5212);
		}
		const uint32_t* pb = ph + g * pst + j * (BP / 2) + t;
		mma_f16_16816(acc, af, pb[0], pb[4]);
	};
	for (int j = 0; j < nb; j += 2) {
		pv(j, acc0);
		if (j + 1 < nb) pv(j + 1, acc1);
	}
	ATTN_DBG(4);

	// ---- this CTA's record: head t, dims r0 / r1, published straight into the cells
	{
		const int r0 = F16 ? 16 * warp + g : 16 * warp + 2 * g, r1 = F16 ? r0 + 8 : r0 + 1;
		const float v0 = (acc0[0] + acc0[1]) + (acc1[0] + acc1[1]), v1 = (acc0[2] + acc0[3]) + (acc1[2] + acc1[3]);
		unsigned long long* cell = a.cells + ((size_t)unit * nsplit + split) * HG * REC + t * REC;
		asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(cell + r0), "l"(((unsigned long long)epoch << 32) | __float_as_uint(v0)) : "memory");
		asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(cell + r1), "l"(((unsigned long long)epoch << 32) | __float_as_uint(v1)) : "memory");
		myrec[t * REC + r0] = v0, myrec[t * REC + r1] = v1;
		if (tid < HG) {
			const float m = s_m[tid], l = s_l[tid] + s_l[tid + 4];
			unsigned long long* ml = a.cells + ((size_t)unit * nsplit + split) * HG * REC + tid * REC + HD;
			asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(ml), "l"(((unsigned long long)epoch << 32) | __float_as_uint(m)) : "memory");
			asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(ml + 1), "l"(((unsigned long long)epoch << 32) | __float_as_uint(l)) : "memory");
			myrec[tid * REC + HD] = m, myrec[tid * REC + HD + 1] = l;
		}
	}
	__syncthreads();
	ATTN_DBG(5);
	attn_cell_fold<HG, HD>(a, unit, split, hbase, epoch, myrec);
	// no bulk copy may still be in flight into this CTA's shared memory when it exits (a block requested on a stale hint)
	if (tid < nbmax && (early(tid) || needed(tid))) mbar_wait(&bars[tid], 0);
	ATTN_DBG(7);
	if (a.dbg && tid == 0) atomicMax(a.dbg + 9, globaltimer_ns());
	stamp_end(a.stamp);
}
