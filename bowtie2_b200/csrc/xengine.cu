// xengine.cu -- the exact search policy ON THE DEVICE: the state machine of xengine.cuh as a kernel (one thread per read pair /
// read, state resident in HBM), advanced in WAVES.  A wave = k_xe_step (every unfinished unit runs until it needs a batched
// primitive and appends that request to a device queue; SA-offset resolution, SwDriver::extend and ungapped alignment happen
// inline in the thread) followed by one launch per non-empty queue: seed-extension DP, mate-finding DP (both = the fill + tail
// kernels of dp_kernels.cu over the queued bt2g_dp_problem arrays), 1-mismatch search, (re-)seeding.  exactSweep for every read
// runs once at admission.  The host only reads five queue counters per wave to size the launches.
//
// This replaces the reference's per-thread control loop (multiseedSearchWorker, bt2_search.cpp:3094-4254, driving
// SwDriver::extendSeedsPaired, aligner_sw_driver.cpp:1582-2637) with the same decisions, RNG draws included, made by up to
// hundreds of thousands of reads at once; results are the reference program's (tests/test_xengine_gpu.py, bench.py's parity gate).
#include <new>
#include <mutex>
#include <map>
#include <cstdio>
#include <cstddef>
#include <chrono>
#include <cstring>
#include <string>
#include <vector>
#include "dp_ungapped_device.cuh"
#include "dp_device.cuh"
#include "launch.cuh"
#define XE_HD __device__           // the host twin of the state machine is compiled in xengine_host.cpp
#include "xengine.cuh"
#include "xengine_shared.h"

extern "C" int bt2g_policy_align(const bt2g_policy_backend *, const bt2g_policy_params *, const bt2g_reads *, const char *const *,
                                 bt2g_read_result *, uint8_t *, uint32_t, bt2g_pair_result *, uint64_t *);

namespace {
using namespace xe;

#define XE_MM_MAXHITS 16
#define XE_TEV 96                    // timing marks per DP queue and wave (fill / tail split; chunks beyond that go unsplit)

struct XQueues {                     // per wave, reset before k_xe_step
	uint32_t nDpA, nDpM, nMm, nSeed, nDone, nFallback, nActive, pad1;
	unsigned long long cellsA, cellsM;
};

struct DpOut { bt2g_dp_problem *probs; bt2g_dp_summary *summ; bt2g_dp_cand *cands; bt2g_dp_aln *alns; uint8_t *ops; int maxCands, maxAlns, maxOps; };

struct XDev {                        // everything the step kernel needs (passed by value)
	const uint8_t *seq, *qual; const uint64_t *roff;
	const uint32_t *seeds;
	const uint64_t *packed; const uint32_t *nmask;         // the reads 2 bits per base + N masks (k_pack_reads)
	const uint8_t *mine; const uint64_t *ee;
	const bt2g_mm_hit *mmHits; const int32_t *mmCounts;
	uint32_t *mmSel; int32_t *mmMinsc; uint8_t *mmMask;
	const uint64_t *ranges; const int32_t *nseeds; int maxSeeds;
	int32_t *seedInterval, *seedOffset; uint8_t *seedActive;
	DpOut A, M;
	XQueues *q;
	XUnit *units; uint8_t *status; uint64_t nUnits;
	bt2g_read_result *res; uint8_t *resOps; bt2g_pair_result *pairs; uint32_t resMaxOps;
};

template <typename OFF>
struct DevSvc {
	const DevIndex<OFF> &ix; const bt2g_scoring &sc; const XDev &d;
	__device__ DevSvc(const DevIndex<OFF> &i, const bt2g_scoring &s, const XDev &dd) : ix(i), sc(s), d(dd) {}
	__device__ const uint8_t *codes(int read) const { return d.seq + d.roff[read]; }
	__device__ const uint8_t *quals(int read) const { return d.qual + d.roff[read]; }
	__device__ int rdlen(int read) const { return (int)(d.roff[read + 1] - d.roff[read]); }
	__device__ uint32_t randSeed(int read) const { return d.seeds[read]; }
	__device__ void sweep(int read, int mined[2], uint64_t tb[4]) const {
		mined[0] = d.mine[2 * (size_t)read]; mined[1] = d.mine[2 * (size_t)read + 1];
		for(int j = 0; j < 4; j++) tb[j] = d.ee[4 * (size_t)read + j];
	}
	__device__ int mmMax() const { return XE_MM_MAXHITS; }
	__device__ int mmCount(int slot, int task) const { return d.mmCounts[4 * (size_t)slot + task]; }
	__device__ const bt2g_mm_hit *mmHits(int slot, int task) const { return d.mmHits + (4 * (size_t)slot + task) * XE_MM_MAXHITS; }
	__device__ int nSeeds(int read) const { return d.nseeds[read]; }
	__device__ const uint64_t *seedRange(int read, int strand, int i) const { return d.ranges + (((size_t)read * 2 + strand) * d.maxSeeds + i) * 4; }
	__device__ const DpOut &dq(bool mate) const { return mate ? d.M : d.A; }
	__device__ const bt2g_dp_summary *dpSumm(int slot, bool mate) const { return dq(mate).summ + slot; }
	__device__ const bt2g_dp_cand *dpCands(int slot, bool mate) const { return dq(mate).cands + (size_t)slot * dq(mate).maxCands; }
	__device__ const bt2g_dp_aln *dpAlns(int slot, bool mate) const { return dq(mate).alns + (size_t)slot * dq(mate).maxAlns; }
	__device__ const uint8_t *dpOps(int slot, bool mate, int k) const { const DpOut &o = dq(mate); return o.ops + ((size_t)slot * o.maxAlns + k) * o.maxOps; }
	__device__ int dpMaxAlns() const { return d.A.maxAlns; }
	// GroupWalk2S::advanceElement == Ebwt::getOffset, then Ebwt::joinedToTextOff (k_resolve2, fm_seed2.cu)
	__device__ bool resolve(uint64_t row, int qlen, bool reject, int64_t &tidx, int64_t &toff, int64_t &tlen) const {
		unsigned nside = 0;
		// (a 1-mismatch hit of a unique occurrence arrives as its joined offset: fm_onemm.cu)
		const uint64_t off = (row & BT2G_ROW_IS_OFFSET) ? (row & ~BT2G_ROW_IS_OFFSET) : get_offset<OFF>(ix, row, nside);
		uint64_t ti, to, tl; bool st;
		const bool ok = joined_to_text<OFF>(ix, (uint64_t)qlen, off, reject, ti, to, tl, st);
		tidx = (int64_t)ti; toff = (int64_t)to; tlen = (int64_t)tl;
		return ok;
	}
	// SwDriver::extend (k_extend, fm_kernels.cu): left with the forward index, right with the mirror index
	__device__ void extend(int read, bool fw, int rdoff, int seedlen, const uint64_t rng[4], int &nlex, int &nrex) const {
		const int len = rdlen(read);
		uint32_t nl = 0, nr = 0;
		const uint64_t wb = (d.roff[read] >> 5) + (uint64_t)read;
		extend_hit<OFF>(ix, rng, codes(read), len, fw, rdoff, seedlen < len ? seedlen : len, true, true, nl, nr, d.packed + wb, d.nmask + wb);
		nlex = (int)nl; nrex = (int)nr;
	}
	__device__ int ungapped(int read, bool fw, int64_t tidx, int64_t refoff, int64_t tlen, int64_t minsc, bt2g_ungapped_result &r) const {
		bt2g_ungapped_problem p; p.read_idx = (uint32_t)read; p.fw = fw ? 1u : 0u; p.tidx = (uint64_t)tidx; p.refoff = refoff; p.reflen = (uint64_t)tlen;
		p.minsc = (int32_t)minsc; p.ohang = 0;
		ungapped_one<OFF>(ix, sc, codes(read), quals(read), rdlen(read), p, r, nullptr, 0);
		return r.status;
	}
	mutable RefCursor<OFF> refCur;
	__device__ int refChar(int64_t tidx, int64_t off) const { return refCur.get(ix, (uint64_t)tidx, off); }
};

// genRandSeed (pat.cpp:45-82) for every read; names: rows of nameStride bytes (NUL-terminated) or nullptr = "r<unit index>"
__global__ void k_xe_seeds(const uint8_t *seq, const uint8_t *qual, const uint64_t *roff, uint64_t nReads, const char *names, uint32_t nameStride,
                           int paired, uint32_t seed, uint32_t *out) {
	const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if(i >= nReads) return;
	const uint8_t *c = seq + roff[i], *q = qual + roff[i];
	const int len = (int)(roff[i + 1] - roff[i]);
	uint32_t rseed = (seed + 101u) * 59u * 61u * 67u * 71u * 73u * 79u * 83u;
	for(int k = 0; k < len; k++) rseed ^= (uint32_t)c[k] << ((k & 15) << 1);
	for(int k = 0; k < len; k++) rseed ^= (uint32_t)q[k] << ((k & 3) << 3);
	if(names) {
		const char *nm = names + i * (uint64_t)nameStride;
		for(uint32_t k = 0; k < nameStride && nm[k]; k++) { if(nm[k] == '/') break; rseed ^= (uint32_t)(unsigned char)nm[k] << ((k & 3) << 3); }
	} else {
		char buf[24]; int n = 0;
		uint64_t v = paired ? i >> 1 : i;
		char tmp[20]; int t = 0;
		do { tmp[t++] = (char)('0' + v % 10); v /= 10; } while(v);
		buf[n++] = 'r';
		while(t) buf[n++] = tmp[--t];
		for(int k = 0; k < n; k++) rseed ^= (uint32_t)(unsigned char)buf[k] << ((k & 3) << 3);
	}
	out[i] = rseed;
}

__global__ void k_xe_reset(XUnit *units, uint8_t *status, uint64_t nUnits, int paired) {
	const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if(i >= nUnits) return;
	x_unit_reset(units[i], (uint32_t)i, paired != 0);
	status[i] = 0;
}

// counter += 1 for every calling lane, one atomic per group of lanes that arrive together on the same counter
__device__ __forceinline__ uint32_t agg_inc(uint32_t *ctr) {
	const unsigned act = __activemask();
	const unsigned peers = __match_any_sync(act, (unsigned long long)ctr);
	const int lane = threadIdx.x & 31, leader = __ffs(peers) - 1;
	uint32_t base = 0;
	if(lane == leader) base = atomicAdd(ctr, (uint32_t)__popc(peers));
	base = __shfl_sync(peers, base, leader);
	return base + (uint32_t)__popc(peers & ((1u << lane) - 1u));
}

// status: 0 running, 1 finished, 2 fallback (to be re-run by the coroutine engine).
// The wave runs over the ACTIVE list (activeIn, nAct entries; nullptr = every unit, the first wave): units that wait for an
// answer append themselves to activeOut, so later waves launch as many threads as there are unfinished units -- the long tail
// of a batch (a few thousand repeat-rich pairs going through dozens of DP rounds) then occupies a few warps, not the GPU.
template <typename OFF, int MINB>
__global__ void __launch_bounds__(128, MINB) k_xe_step(DevIndex<OFF> ix, bt2g_scoring sc, XParams P, XDev d, const uint32_t *activeIn, uint32_t *activeOut,
                                                       uint32_t nAct, int spread) {
	// spread = s: one unit per 2^s threads (the others idle).  The state machines of a warp's lanes diverge and serialise, so when
	// a wave has few units (the tail of a batch) one unit per warp finishes sooner than 32.
	const uint64_t tt = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	const uint64_t t = tt >> spread;
	const bool valid = t < nAct && (tt & ((1u << spread) - 1u)) == 0;
	const uint64_t i = valid ? (activeIn ? activeIn[t] : t) : 0;
	int r = XR_DONE;
	if(valid) {
		XUnit &u = d.units[i];
		DevSvc<OFF> svc(ix, sc, d);
		r = x_step(P, u, svc);
		switch(r) {
		case XR_DP: case XR_DP_MATE: {
			const bool mate = r == XR_DP_MATE;
			const uint32_t slot = agg_inc(mate ? &d.q->nDpM : &d.q->nDpA);
			(mate ? d.M : d.A).probs[slot] = u.rqProb;
			u.dpSlot = (int32_t)slot;
			const unsigned long long cells = (unsigned long long)svc.rdlen((int)u.rqProb.read_idx) * (unsigned long long)(u.rqProb.refr - u.rqProb.refl + 1);
			atomicAdd(mate ? &d.q->cellsM : &d.q->cellsA, cells);
			break; }
		case XR_ONE_MM: {
			const uint32_t slot = agg_inc(&d.q->nMm);
			d.mmSel[slot] = (uint32_t)u.rqRead; d.mmMinsc[slot] = u.rqMinsc; d.mmMask[slot] = (uint8_t)((u.rqNofw ? 0 : 1) | (u.rqNorc ? 0 : 2));
			u.dpSlot = (int32_t)slot;
			break; }
		case XR_SEED:
			d.seedActive[u.rqRead] = 1; d.seedInterval[u.rqRead] = u.rqInterval; d.seedOffset[u.rqRead] = u.rqOffset;
			agg_inc(&d.q->nSeed);
			break;
		case XR_DONE: {
			d.status[i] = 1;
			agg_inc(&d.q->nDone);
			const uint64_t r0 = u.paired ? 2 * i : i; const int nr = u.paired ? 2 : 1;
			for(int k = 0; k < nr; k++) x_fill_result(u, k, svc.codes((int)(r0 + k)), d.res[r0 + k], d.resOps + (r0 + k) * (uint64_t)d.resMaxOps, d.resMaxOps);
			if(u.paired) { bt2g_pair_result pr; pr.pair_type = u.pairType; pr.kind = u.pairKind; pr.source = 0; pr.score_sum = (int32_t)u.scoreSum; pr.fraglen = u.fraglen; d.pairs[i] = pr; }
			break; }
		default:
			d.status[i] = 2;
			agg_inc(&d.q->nFallback);
			break;
		}
	}
	// the units of this warp that wait for an answer, appended as ONE run in their order (the active list stays a sequence of
	// ascending runs: neighbouring threads keep working on neighbouring units -- their 44 KB states share TLB entries); no
	// block-wide barrier: a warp retires as soon as its own slowest unit has stepped
	__syncwarp();
	const bool cont = valid && (r == XR_DP || r == XR_DP_MATE || r == XR_ONE_MM || r == XR_SEED);
	const unsigned m = __ballot_sync(0xffffffffu, cont);
	if(m) {
		const int lane = threadIdx.x & 31, leader = __ffs(m) - 1;
		uint32_t base = 0;
		if(lane == leader) base = atomicAdd(&d.q->nActive, (uint32_t)__popc(m));
		base = __shfl_sync(0xffffffffu, base, leader);
		if(cont) activeOut[base + (uint32_t)__popc(m & ((1u << lane) - 1u))] = (uint32_t)i;
	}
}

struct DpWork {                       // workspace of one DP queue (anchor rectangles / mate rectangles)
	DpOut o{}; uint8_t *codes = nullptr; int32_t *lastH = nullptr; uint64_t *rawKeys = nullptr;
	int maxCol = 0, packed = 0, maxRaw = 0; uint64_t codeStride = 0, chunk = 0, numSlots = 0;
};

} // namespace

struct bt2g_xengine {
	bt2g_ctx *ctx = nullptr;
	bt2g_policy_params pp{};
	bt2g_scoring sc{};
	XParams P{}; XTables T;
	uint64_t maxUnits = 0, maxReads = 0, maxBases = 0; int maxLen = 0; uint32_t maxOps = 0;
	std::vector<void *> allocs;
	int32_t *dTabs = nullptr;
	XDev d{};
	DpWork A, M;
	uint64_t *packed = nullptr; uint32_t *nmask = nullptr; unsigned long long *nextTask = nullptr;
	uint32_t *active[2] = {nullptr, nullptr};          // unit indices of the current / the next wave
	uint8_t *dSeq = nullptr, *dQual = nullptr; uint64_t *dOff = nullptr; char *dNames = nullptr; uint32_t nameStrideCap = 0;
	XQueues *hq = nullptr;             // pinned
	uint8_t *hStatus = nullptr;        // pinned
	int sms = 148;
	cudaStream_t stream = nullptr;     // the engine's own stream (bt2g_xengine_align; run_dev when the caller passes none)
	cudaStream_t streamHi = nullptr;   // high-priority twin: the small waves of a batch's tail run here, so that their few blocks are
	                                   // scheduled ahead of the pending blocks of another engine's full waves
	bool ownStreams = false;           // this batch runs on the engine's streams (the caller passed none)
	int debug = 0;                     // BT2G_XE_DEBUG: per-wave log on stderr
	uint64_t stats[8] = {0, 0, 0, 0, 0, 0, 0, 0};     // waves, fallbacks, anchor DPs, mate DPs, anchor cells, mate cells, 1-mm requests, seed requests
	// device time of the last batch per stage (CUDA events on the batch's stream): admission (read seeds, packing, exactSweep),
	// state machine (k_xe_step), 1-mismatch search, seed search, seed-extension DP, mate-finding DP, host fallback (wall), total
	float stageMs[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};   // [8], [9]: DP fill / DP tail kernels of both queues (split of [4] + [5])
	cudaEvent_t tev[2][XE_TEV]; int tevN[2] = {0, 0};
	cudaEvent_t evJoin = nullptr;
	uint64_t launches = 0;             // kernels of this library launched by the last batch
	cudaEvent_t ev[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
};

namespace {

template <typename T> int xalloc(bt2g_xengine *e, T *&ptr, uint64_t count) {
	void *v = nullptr;
	const cudaError_t err = cudaMalloc(&v, (count ? count : 1) * sizeof(T));
	if(err != cudaSuccess) { e->ctx->err = std::string("xengine cudaMalloc: ") + cudaGetErrorString(err); return -2; }
	e->allocs.push_back(v);
	ptr = (T *)v;
	return 0;
}

int setupDp(bt2g_xengine *e, DpWork &w, int maxCol, uint64_t cap, int maxCands, int maxAlns) {
	const bt2g_scoring &sc = e->sc;
	int64_t mn = 0;
	for(int l = 1; l <= e->maxLen; l++) if(e->T.minsc[l] < mn) mn = e->T.minsc[l];
	w.maxCol = maxCol + 1;
	w.packed = sc.local ? 0 : dp_kernel_mode(sc, mn, e->maxLen, e->ctx->dpModeCap);
	w.codeStride = dp_code_stride(w.maxCol, e->maxLen, w.packed);
	w.numSlots = (uint64_t)e->sms * 24;
	int rc = 0;
	// (3 GiB of H-byte workspace per queue: a chunk still holds tens of thousands of problems, and several engines fit one GPU)
	if(w.packed == 3) { w.chunk = dp_chunk_problems(w.codeStride, cap, 3ull << 30); rc |= xalloc(e, w.codes, w.chunk * w.codeStride); }
	else rc |= xalloc(e, w.codes, w.numSlots * w.codeStride * (w.packed ? 2 : 1));
	rc |= xalloc(e, w.lastH, w.numSlots * (uint64_t)w.maxCol);
	w.maxRaw = maxCands * 4 < 1024 ? 1024 : maxCands * 4;
	if(sc.local) rc |= xalloc(e, w.rawKeys, w.numSlots * (uint64_t)w.maxRaw);
	w.o.maxCands = maxCands; w.o.maxAlns = maxAlns; w.o.maxOps = e->maxLen + 80;
	rc |= xalloc(e, w.o.probs, cap); rc |= xalloc(e, w.o.summ, cap); rc |= xalloc(e, w.o.cands, cap * (uint64_t)maxCands);
	rc |= xalloc(e, w.o.alns, cap * (uint64_t)maxAlns); rc |= xalloc(e, w.o.ops, cap * (uint64_t)maxAlns * w.o.maxOps);
	return rc;
}

template <typename OFF>
int launchDp(bt2g_xengine *e, const DpWork &w, uint64_t n, cudaStream_t st) {
	if(n == 0) return 0;
	DpLaunch L;
	L.seq = e->d.seq; L.qual = e->d.qual; L.roff = e->d.roff; L.probs = w.o.probs; L.n = n; L.nDev = nullptr;
	L.numSlots = w.numSlots; L.codes = w.codes; L.lastH = w.lastH; L.rawKeys = w.rawKeys; L.maxRaw = w.rawKeys ? w.maxRaw : 0;
	L.codeStride = w.codeStride; L.maxCol = w.maxCol; L.maxCands = w.o.maxCands; L.maxAlns = w.o.maxAlns; L.maxOps = w.o.maxOps;
	L.chunk = w.chunk; L.packed = w.packed;
	{ const int qi = &w == &e->M ? 1 : 0; e->tevN[qi] = 0; L.tev = e->tev[qi]; L.tevCap = XE_TEV; L.tevN = &e->tevN[qi]; }
	L.summ = w.o.summ; L.cands = w.o.cands; L.alns = w.o.alns; L.ops = w.o.ops;
	const DevIndex<OFF> ix = bt2g_dev_index<OFF>(e->ctx);
	e->launches += (!e->sc.local && w.packed == 3) ? 2 * ((n + w.chunk - 1) / w.chunk) : 1;
	return e->sc.local ? launch_dp_local<OFF>(ix, e->sc, L, e->maxLen, st) : launch_dp_e2e<OFF>(ix, e->sc, L, e->maxLen, st);
}

// the waves of one batch whose reads are in device memory (e->d.seq / qual / roff set)
template <typename OFF>
int runBatch(bt2g_xengine *e, uint64_t nReads, const char *dNames, uint32_t nameStride, cudaStream_t st0) {
	cudaStream_t st = st0;
	bt2g_ctx *ctx = e->ctx;
	const bool paired = e->P.paired != 0;
	const uint64_t nUnits = paired ? nReads / 2 : nReads;
	const DevIndex<OFF> ix = bt2g_dev_index<OFF>(ctx);
	XDev &d = e->d;
	d.nUnits = nUnits;
	d.packed = e->packed; d.nmask = e->nmask;
	const unsigned T = 128;
	auto grid = [&](uint64_t m, unsigned t) { return (unsigned)((m + t - 1) / t); };
	for(int k = 0; k < 8; k++) e->stats[k] = 0;
	for(int k = 0; k < 12; k++) e->stageMs[k] = 0.f;
	e->tevN[0] = e->tevN[1] = 0;
	e->launches = 4;                                   // k_xe_seeds, k_xe_reset, k_pack_reads, k_exact_sweep2
	cudaEvent_t *ev = e->ev;
	auto lap = [&](int a, int b, int stage) { float ms = 0.f; if(cudaEventElapsedTime(&ms, ev[a], ev[b]) == cudaSuccess) e->stageMs[stage] += ms; };
	cudaEventRecord(ev[7], st);
	// admission: read seeds, unit reset, 2-bit packing, exactSweep of every read
	k_xe_seeds<<<grid(nReads, T), T, 0, st>>>(d.seq, d.qual, d.roff, nReads, dNames, nameStride, paired ? 1 : 0, e->P.seed, const_cast<uint32_t *>(d.seeds));
	k_xe_reset<<<grid(nUnits, T), T, 0, st>>>(d.units, d.status, nUnits, paired ? 1 : 0);
	launch_pack_reads(d.seq, d.roff, nReads, e->maxLen, e->packed, e->nmask, st);
	launch_exact_sweep2<OFF>(ix, d.roff, nReads, 0, 0, const_cast<uint8_t *>(d.mine), const_cast<uint64_t *>(d.ee), e->packed, e->nmask, e->nextTask, e->sms, st, nullptr,
	                         ix.extText ? 2 : 0 /* unique ranges continue in the text */);
	BT2G_CUDA_TRY(ctx, cudaMemsetAsync(d.seedActive, 0, nReads, st));
	BT2G_CUDA_TRY(ctx, cudaGetLastError());
	uint64_t done = 0;
	uint32_t nActive = 0;
	cudaEventRecord(ev[0], st);
	for(uint64_t wave = 0;; wave++) {
		BT2G_CUDA_TRY(ctx, cudaMemsetAsync(d.q, 0, sizeof(XQueues), st));
		{
			const uint32_t nAct = wave == 0 ? (uint32_t)nUnits : nActive;
			const uint32_t *in = wave == 0 ? nullptr : e->active[wave & 1];
			uint32_t *out = e->active[(wave + 1) & 1];
			const int spread = (uint64_t)nAct * 32 <= (uint64_t)e->sms * 2048 * 4 ? 5 : 0;       // few units: one per warp
			const uint64_t nThr = (uint64_t)nAct << spread;
			k_xe_step<OFF, 4><<<grid(nThr, 128), 128, 0, st>>>(ix, e->sc, e->P, d, in, out, nAct, spread);
		}
		cudaEventRecord(ev[1], st);
		e->launches++;
		BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(e->hq, d.q, sizeof(XQueues), cudaMemcpyDeviceToHost, st));
		BT2G_CUDA_TRY(ctx, cudaStreamSynchronize(st));
		// everything recorded before this synchronisation has completed: the primitives of the previous wave and this step
		if(wave == 0) lap(7, 0, 0); else { lap(2, 3, 2); lap(3, 4, 3); lap(4, 5, 4); lap(5, 0, 5); }
		for(int qi = 0; qi < 2; qi++) {                   // fill / tail split of the DP launches of the previous wave
			for(int k = 0; k + 1 < e->tevN[qi]; k++) { float ms = 0.f; if(cudaEventElapsedTime(&ms, e->tev[qi][k], e->tev[qi][k + 1]) == cudaSuccess) e->stageMs[8 + (k & 1)] += ms; }
			e->tevN[qi] = 0;
		}
		lap(0, 1, 1);
		const XQueues q = *e->hq;
		if(e->debug) {
			float ms = 0.f; cudaEventElapsedTime(&ms, ev[0], ev[1]);
			fprintf(stderr, "[xengine] wave %llu: step %.3f ms; done %u fallback %u | dpA %u dpM %u mm %u seed %u\n", (unsigned long long)wave, ms, q.nDone, q.nFallback,
			        q.nDpA, q.nDpM, q.nMm, q.nSeed);
		}
		e->stats[0]++; e->stats[1] += q.nFallback; e->stats[2] += q.nDpA; e->stats[3] += q.nDpM; e->stats[4] += q.cellsA; e->stats[5] += q.cellsM;
		e->stats[6] += q.nMm; e->stats[7] += q.nSeed;
		e->launches += (q.nMm ? 1 : 0) + (q.nSeed ? 1 : 0);
		done += q.nDone + q.nFallback;
		nActive = q.nActive;
		if(done >= nUnits) break;
		// everything launched so far has completed (the synchronisation above): the primitives of this wave and the next step may
		// run on another stream -- the high-priority one when few units are left
		if(e->ownStreams) st = (uint64_t)nActive * 32 <= (uint64_t)e->sms * 2048 * 4 ? e->streamHi : e->stream;
		if(q.nDpA + q.nDpM + q.nMm + q.nSeed == 0) { ctx->err = "xengine: units neither finished nor waiting"; return -5; }
		cudaEventRecord(ev[2], st);
		if(q.nMm) launch_one_mm_sel<OFF>(ix, d.seq, d.qual, d.roff, q.nMm, d.mmSel, d.mmMinsc, d.mmMask, e->sc, XE_MM_MAXHITS, const_cast<bt2g_mm_hit *>(d.mmHits), const_cast<int32_t *>(d.mmCounts), st,
		                                      ix.extText != 0);
		cudaEventRecord(ev[3], st);
		if(q.nSeed) {
			launch_seed_search_active<OFF>(ix, d.roff, nReads, e->P.seedLen, d.maxSeeds, d.seedInterval, d.seedOffset, d.seedActive, const_cast<uint64_t *>(d.ranges),
			                               const_cast<int32_t *>(d.nseeds), e->packed, e->nmask, e->nextTask, e->sms, st);
			BT2G_CUDA_TRY(ctx, cudaMemsetAsync(d.seedActive, 0, nReads, st));
		}
		cudaEventRecord(ev[4], st);
		// small waves (the tail of a batch): the two DP queues hold a few thousand problems each, so their fill / tail launches run
		// side by side on the engine's two streams instead of one after the other (everything before this point has completed)
		const bool sideBySide = e->ownStreams && q.nDpA && q.nDpM && (uint64_t)(q.nDpA + q.nDpM) * 16 <= (uint64_t)e->sms * 2048;
		cudaStream_t stM = sideBySide ? (st == e->stream ? e->streamHi : e->stream) : st;
		if(launchDp<OFF>(e, e->A, q.nDpA, st)) { ctx->err = "xengine: DP launch rejected"; return -1; }
		cudaEventRecord(ev[5], st);
		if(launchDp<OFF>(e, e->M, q.nDpM, stM)) { ctx->err = "xengine: DP launch rejected"; return -1; }
		if(sideBySide) { cudaEventRecord(e->evJoin, stM); cudaStreamWaitEvent(st, e->evJoin, 0); }
		cudaEventRecord(ev[0], st);
		BT2G_CUDA_TRY(ctx, cudaGetLastError());
	}
	lap(7, 1, 7);
	return 0;
}

} // namespace

extern "C" {

int bt2g_xengine_create(bt2g_ctx *ctx, const bt2g_policy_params *pp, uint64_t maxUnits, uint32_t maxLen, bt2g_xengine **out) {
	if(!ctx || !pp || !out || maxUnits == 0 || maxLen == 0) return -1;
	*out = nullptr;
	if(!ctx->loaded) { ctx->err = "no index loaded"; return -1; }
	if(!ctx->info.has_bw || !ctx->info.has_ref) { ctx->err = "xengine: needs the mirror index and the packed reference"; return -1; }
	if(maxLen > XE_MAX_LEN) { ctx->err = "xengine: reads longer than 512 are not supported"; return -1; }
	if(pp->all_hits || pp->khits > 1) { ctx->err = "xengine: -k / -a are served by bt2g_policy_align_k"; return -1; }
	BT2G_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
	bt2g_xengine *e = new(std::nothrow) bt2g_xengine();
	if(!e) return -4;
	e->ctx = ctx; e->pp = *pp; e->maxLen = (int)maxLen; e->maxUnits = maxUnits;
	e->maxReads = pp->paired ? 2 * maxUnits : maxUnits; e->maxBases = e->maxReads * (uint64_t)maxLen;
	e->maxOps = maxLen + 80;
	cudaDeviceGetAttribute(&e->sms, cudaDevAttrMultiProcessorCount, ctx->device);
	if(getenv("BT2G_XE_DEBUG")) e->debug = 1;
	// the kernels score with the scheme the policy reasons about (one source: the policy parameters)
	scoringFromParams(pp, &e->sc);
	ctx->scoring = e->sc;
	buildParams(pp, ctx->info.off_size, (int)maxLen, e->P, e->T);
	int rc = 0;
	const uint64_t nR = e->maxReads, nU = maxUnits;
	rc |= xalloc(e, e->dTabs, 4ull * (maxLen + 1));
	XDev &d = e->d;
	rc |= xalloc(e, e->dSeq, e->maxBases); rc |= xalloc(e, e->dQual, e->maxBases); rc |= xalloc(e, e->dOff, nR + 1);
	uint32_t *seeds; uint8_t *mine; uint64_t *ee;
	rc |= xalloc(e, seeds, nR); rc |= xalloc(e, mine, nR * 2); rc |= xalloc(e, ee, nR * 4);
	d.seeds = seeds; d.mine = mine; d.ee = ee;
	bt2g_mm_hit *mmHits; int32_t *mmCounts;
	rc |= xalloc(e, mmHits, nU * 4 * XE_MM_MAXHITS); rc |= xalloc(e, mmCounts, nU * 4);
	d.mmHits = mmHits; d.mmCounts = mmCounts;
	rc |= xalloc(e, d.mmSel, nU); rc |= xalloc(e, d.mmMinsc, nU); rc |= xalloc(e, d.mmMask, nU);
	{
		int minIval = 1 << 30;
		for(int l = 1; l <= (int)maxLen; l++) { minIval = std::min(minIval, std::min(e->T.ivalOne[l], e->T.ivalBoth[l])); }
		int ms = 1 + ((int)maxLen - std::min<int>(pp->seed_len, (int)maxLen)) / std::max(1, minIval) + 1;
		if(ms > XE_MAX_SEEDS) ms = XE_MAX_SEEDS + 1;          // reads with more seeds fall back
		d.maxSeeds = ms;
	}
	uint64_t *ranges; int32_t *nseeds;
	rc |= xalloc(e, ranges, nR * 2ull * d.maxSeeds * 4); rc |= xalloc(e, nseeds, nR);
	d.ranges = ranges; d.nseeds = nseeds;
	rc |= xalloc(e, d.seedInterval, nR); rc |= xalloc(e, d.seedOffset, nR); rc |= xalloc(e, d.seedActive, nR);
	rc |= xalloc(e, e->packed, (e->maxBases >> 5) + nR + 2); rc |= xalloc(e, e->nmask, (e->maxBases >> 5) + nR + 2); rc |= xalloc(e, e->nextTask, 1);
	rc |= xalloc(e, d.q, 1); rc |= xalloc(e, d.units, nU); rc |= xalloc(e, d.status, nU);
	rc |= xalloc(e, e->active[0], nU); rc |= xalloc(e, e->active[1], nU);
	rc |= xalloc(e, d.res, nR); rc |= xalloc(e, d.resOps, nR * (uint64_t)e->maxOps); rc |= xalloc(e, d.pairs, nU);
	d.resMaxOps = e->maxOps;
	if(!rc) {
		// anchor rectangles: rdlen + 4 * min(maxgap, 15) columns; mate rectangles: the fragment window plus the mate and its gaps
		const int maxColA = (int)maxLen + 4 * 15 + 4;
		int gapMax = 15;
		for(int l = 1; l <= (int)maxLen; l++) { gapMax = std::max(gapMax, std::max(e->P.maxReadGaps(e->T.minsc[l], l), e->P.maxRefGaps(e->T.minsc[l], l))); }
		if(gapMax > 512) gapMax = 512;
		const uint64_t maxfrag = std::max<uint64_t>(pp->pe.maxfrag, maxLen);
		int maxColM = (int)std::min<uint64_t>(maxfrag + 2ull * maxLen + 2ull * gapMax + 16, 8000);
		// (local mode: a 300 bp read has thousands of candidate cells and tens of distinct successful backtraces per rectangle;
		// a problem that overflows either list sends its unit to the host fallback)
		const int maxCands = e->sc.local ? 16384 : 256, maxAlns = e->sc.local ? 32 : 8;
		rc |= setupDp(e, e->A, maxColA, nU, maxCands, maxAlns);
		if(pp->paired) rc |= setupDp(e, e->M, maxColM, nU, maxCands, maxAlns);
		else e->M = e->A;
		d.A = e->A.o; d.M = e->M.o;
	}
	cudaError_t err = cudaSuccess;
	if(!rc) {
		std::vector<int32_t> tabs(4ull * (maxLen + 1));
		for(uint32_t l = 0; l <= maxLen; l++) { tabs[l] = e->T.minsc[l]; tabs[(maxLen + 1) + l] = e->T.nceilRaw[l]; tabs[2 * (maxLen + 1) + l] = e->T.ivalOne[l]; tabs[3 * (maxLen + 1) + l] = e->T.ivalBoth[l]; }
		err = cudaMemcpy(e->dTabs, tabs.data(), tabs.size() * 4, cudaMemcpyHostToDevice);
		e->P.minscTab = e->dTabs; e->P.nceilRawTab = e->dTabs + (maxLen + 1); e->P.ivalOneTab = e->dTabs + 2 * (maxLen + 1); e->P.ivalBothTab = e->dTabs + 3 * (maxLen + 1);
		if(err == cudaSuccess) err = cudaHostAlloc((void **)&e->hq, sizeof(XQueues), cudaHostAllocDefault);
		if(err == cudaSuccess) err = cudaHostAlloc((void **)&e->hStatus, nU, cudaHostAllocDefault);
		for(int k = 0; k < 8 && err == cudaSuccess; k++) err = cudaEventCreate(&e->ev[k]);
		for(int k = 0; k < 2 * XE_TEV && err == cudaSuccess; k++) err = cudaEventCreate(&e->tev[k / XE_TEV][k % XE_TEV]);
		if(err == cudaSuccess) err = cudaEventCreateWithFlags(&e->evJoin, cudaEventDisableTiming);
		if(err == cudaSuccess) err = cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking);
		if(err == cudaSuccess) { int lo = 0, hi = 0; cudaDeviceGetStreamPriorityRange(&lo, &hi); err = cudaStreamCreateWithPriority(&e->streamHi, cudaStreamNonBlocking, hi); }
	}
	if(rc || err != cudaSuccess) {
		if(err != cudaSuccess) ctx->err = std::string("xengine setup: ") + cudaGetErrorString(err);
		bt2g_xengine_destroy(e);
		return -2;
	}
	*out = e;
	return 0;
}

void bt2g_xengine_destroy(bt2g_xengine *e) {
	if(!e) return;
	cudaSetDevice(e->ctx->device);
	for(void *v : e->allocs) cudaFree(v);
	if(e->hq) cudaFreeHost(e->hq);
	if(e->hStatus) cudaFreeHost(e->hStatus);
	for(int k = 0; k < 8; k++) if(e->ev[k]) cudaEventDestroy(e->ev[k]);
	for(int k = 0; k < 2 * XE_TEV; k++) if(e->tev[k / XE_TEV][k % XE_TEV]) cudaEventDestroy(e->tev[k / XE_TEV][k % XE_TEV]);
	if(e->evJoin) cudaEventDestroy(e->evJoin);
	if(e->stream) cudaStreamDestroy(e->stream);
	if(e->streamHi) cudaStreamDestroy(e->streamHi);
	delete e;
}

// reads already in device memory; results stay on the device (bt2g_xengine_results_dev).  Units that fall back are re-run
// by the coroutine engine over this library's entry points and patched into the device result arrays.
int bt2g_xengine_run_dev(bt2g_xengine *e, const uint8_t *dSeq, const uint8_t *dQual, const uint64_t *dOff, uint64_t nReads,
                         const char *dNames, uint32_t nameStride, void *stream, uint64_t *stats) {
	if(!e || !dSeq || !dQual || !dOff) return -1;
	bt2g_ctx *ctx = e->ctx;
	if(nReads > e->maxReads || (e->P.paired && (nReads & 1))) { ctx->err = "xengine: batch larger than the engine was created for"; return -1; }
	if(nReads == 0) return 0;
	BT2G_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
	cudaStream_t st = stream ? (cudaStream_t)stream : e->stream;
	e->ownStreams = stream == nullptr;
	ctx->scoring = e->sc;
	e->d.seq = dSeq; e->d.qual = dQual; e->d.roff = dOff;
	const int rc = ctx->info.off_size == 4 ? runBatch<uint32_t>(e, nReads, dNames, nameStride, st) : runBatch<uint64_t>(e, nReads, dNames, nameStride, st);
	if(rc) return rc;
	if(e->stats[1]) {
		// fallback units: their reads come back to the host, the coroutine engine answers them through the C ABI
		// (the coroutine engine drives the context's own entry points and scratch buffers: one fallback at a time per process)
		static std::mutex fbMutex;
		std::lock_guard<std::mutex> fbLock(fbMutex);
		const auto tFb = std::chrono::steady_clock::now();
		const bool paired = e->P.paired != 0;
		const uint64_t nUnits = paired ? nReads / 2 : nReads, per = paired ? 2 : 1;
		BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(e->hStatus, e->d.status, nUnits, cudaMemcpyDeviceToHost, st));
		std::vector<uint64_t> off(nReads + 1);
		BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(off.data(), dOff, (nReads + 1) * 8, cudaMemcpyDeviceToHost, st));
		BT2G_CUDA_TRY(ctx, cudaStreamSynchronize(st));
		std::vector<uint64_t> ids;
		for(uint64_t i = 0; i < nUnits; i++) if(e->hStatus[i] == 2) ids.push_back(i);
		if(getenv("BT2G_XE_DEBUG")) {                     // which capacity stopped the units (source lines of xengine.cuh)
			std::map<uint32_t, uint64_t> hist;
			for(uint64_t id : ids) { uint32_t ln = 0; cudaMemcpy(&ln, reinterpret_cast<const char *>(e->d.units + id) + offsetof(XUnit, fbLine), 4, cudaMemcpyDeviceToHost); hist[ln]++; }
			fprintf(stderr, "[xengine] %zu fallback units of %llu; by xengine.cuh line:", ids.size(), (unsigned long long)nUnits);
			for(auto &kv : hist) fprintf(stderr, " %u:%llu", kv.first, (unsigned long long)kv.second);
			fprintf(stderr, "\n");
		}
		std::vector<uint8_t> seq, qual; std::vector<uint64_t> soff{0}; std::vector<char> names; std::vector<const char *> nptr;
		for(uint64_t id : ids) for(uint64_t k = 0; k < per; k++) {
			const uint64_t r = id * per + k, a = off[r], b = off[r + 1];
			const size_t o = seq.size();
			seq.resize(o + (b - a)); qual.resize(o + (b - a));
			BT2G_CUDA_TRY(ctx, cudaMemcpy(seq.data() + o, dSeq + a, b - a, cudaMemcpyDeviceToHost));
			BT2G_CUDA_TRY(ctx, cudaMemcpy(qual.data() + o, dQual + a, b - a, cudaMemcpyDeviceToHost));
			soff.push_back(seq.size());
		}
		const uint32_t ns = dNames ? nameStride : 24;
		names.assign(ids.size() * per * (size_t)ns, 0);
		for(size_t j = 0; j < ids.size() * per; j++) {
			const uint64_t r = ids[j / per] * per + (j % per);
			if(dNames) { BT2G_CUDA_TRY(ctx, cudaMemcpy(names.data() + j * ns, dNames + r * (uint64_t)nameStride, nameStride, cudaMemcpyDeviceToHost)); names[j * ns + ns - 1] = 0; }
			else snprintf(names.data() + j * ns, ns, "r%llu", (unsigned long long)(paired ? r >> 1 : r));
		}
		for(size_t j = 0; j < ids.size() * per; j++) nptr.push_back(names.data() + j * ns);
		bt2g_reads sub; sub.n_reads = ids.size() * per; sub.seq = seq.data(); sub.qual = qual.data(); sub.off = soff.data();
		std::vector<bt2g_read_result> res(sub.n_reads); std::vector<uint8_t> ops(sub.n_reads * (size_t)e->maxOps); std::vector<bt2g_pair_result> prs(ids.size());
		bt2g_policy_backend be; bt2g_policy_backend_gpu(ctx, &be);
		bt2g_policy_params pp = e->pp; pp.host_threads = 8;
		const int rc2 = bt2g_policy_align(&be, &pp, &sub, nptr.data(), res.data(), ops.data(), e->maxOps, paired ? prs.data() : nullptr, nullptr);
		if(rc2 < 0) { ctx->err = "xengine: fallback engine failed"; return rc2; }
		for(size_t j = 0; j < ids.size(); j++) {
			const uint64_t r0 = ids[j] * per;
			BT2G_CUDA_TRY(ctx, cudaMemcpy(e->d.res + r0, res.data() + j * per, per * sizeof(bt2g_read_result), cudaMemcpyHostToDevice));
			BT2G_CUDA_TRY(ctx, cudaMemcpy(e->d.resOps + r0 * (uint64_t)e->maxOps, ops.data() + j * per * (size_t)e->maxOps, per * (size_t)e->maxOps, cudaMemcpyHostToDevice));
			if(paired) BT2G_CUDA_TRY(ctx, cudaMemcpy(e->d.pairs + ids[j], prs.data() + j, sizeof(bt2g_pair_result), cudaMemcpyHostToDevice));
		}
		e->stageMs[6] = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - tFb).count();
	}
	if(stats) for(int k = 0; k < 8; k++) stats[k] = e->stats[k];
	return 0;
}

int bt2g_xengine_streams(bt2g_xengine *e, void **stream, void **stream_hi) {
	if(!e) return -1;
	if(stream) *stream = (void *)e->stream;
	if(stream_hi) *stream_hi = (void *)e->streamHi;
	return 0;
}

int bt2g_xengine_stage_ms(bt2g_xengine *e, float *ms, uint64_t *launches) {
	if(!e || !ms) return -1;
	for(int k = 0; k < 10; k++) ms[k] = e->stageMs[k];
	if(launches) *launches = e->launches;
	return 0;
}

int bt2g_xengine_results_dev(bt2g_xengine *e, bt2g_read_result **res, uint8_t **ops, uint32_t *maxOps, bt2g_pair_result **pairs) {
	if(!e) return -1;
	if(res) *res = e->d.res;
	if(ops) *ops = e->d.resOps;
	if(maxOps) *maxOps = e->maxOps;
	if(pairs) *pairs = e->d.pairs;
	return 0;
}

// host buffers in, host results out: res[n_reads], ops[n_reads * max_ops] (max_ops >= the engine's own stride is not required:
// rows are copied with the smaller of the two strides), pairs[n_reads / 2] when paired
int bt2g_xengine_align(bt2g_xengine *e, const bt2g_reads *reads, const char *names, uint32_t nameStride, bt2g_read_result *res, uint8_t *ops,
                       uint32_t maxOps, bt2g_pair_result *pairs, uint64_t *stats) {
	if(!e || !reads || !reads->qual || !res || !ops) return -1;
	bt2g_ctx *ctx = e->ctx;
	const uint64_t n = reads->n_reads;
	if(n > e->maxReads || reads->off[n] > e->maxBases) { ctx->err = "xengine: batch larger than the engine was created for"; return -1; }
	if(e->P.paired && !pairs) return -1;
	if(n == 0) return 0;
	for(uint64_t i = 0; i < n; i++)
		if(reads->off[i + 1] - reads->off[i] > (uint64_t)e->maxLen) { ctx->err = "xengine: a read is longer than the max_len the engine was created for"; return -1; }
	BT2G_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
	cudaStream_t st = e->stream;                      // engines of one context overlap their copies and waves
	const uint64_t nb = reads->off[n];
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(e->dSeq, reads->seq, nb, cudaMemcpyHostToDevice, st));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(e->dQual, reads->qual, nb, cudaMemcpyHostToDevice, st));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(e->dOff, reads->off, (n + 1) * 8, cudaMemcpyHostToDevice, st));
	char *dn = nullptr;
	if(names) {
		if((uint64_t)nameStride * n > (uint64_t)e->nameStrideCap * e->maxReads || !e->dNames) {
			if(xalloc(e, e->dNames, (uint64_t)nameStride * e->maxReads)) return -2;
			e->nameStrideCap = nameStride;
		}
		BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(e->dNames, names, (uint64_t)nameStride * n, cudaMemcpyHostToDevice, st));
		dn = e->dNames;
	}
	const int rc = bt2g_xengine_run_dev(e, e->dSeq, e->dQual, e->dOff, n, dn, nameStride, st, stats);
	if(rc) return rc;
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(res, e->d.res, n * sizeof(bt2g_read_result), cudaMemcpyDeviceToHost, st));
	if(maxOps == e->maxOps) BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(ops, e->d.resOps, n * (uint64_t)maxOps, cudaMemcpyDeviceToHost, st));
	else BT2G_CUDA_TRY(ctx, cudaMemcpy2DAsync(ops, maxOps, e->d.resOps, e->maxOps, maxOps < e->maxOps ? maxOps : e->maxOps, n, cudaMemcpyDeviceToHost, st));
	if(pairs && e->P.paired) BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(pairs, e->d.pairs, (n / 2) * sizeof(bt2g_pair_result), cudaMemcpyDeviceToHost, st));
	BT2G_CUDA_TRY(ctx, cudaStreamSynchronize(st));
	return 0;
}

} // extern "C"
