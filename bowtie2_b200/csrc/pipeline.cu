// pipeline.cu -- the batched hot path: one pass of  exactSweep -> multiseed search -> SA-offset
// resolution -> seed-extension DP (fill + backtrace)  over a batch of reads, entirely on the
// device (seven launches, no host round trip between stages).
//
// This is the data-parallel core the reference runs one read at a time inside
// multiseedSearchWorker (bt2_search.cpp:3094-4254; stages [A] :3514, [C] :3931-3955,
// SwDriver::extendSeeds aligner_sw_driver.cpp:921-1494).  Each stage is the same kernel the
// stand-alone entry points expose (parity-tested one by one against the oracle); what this
// file adds is the glue that the reference interleaves per read:
//   collect : which BW rows to resolve.  Exact end-to-end hits first (eeSaTups, :66-291);
//             otherwise seed ranges smallest-first (SATuple::operator<, aligner_cache.h:397-405),
//             every row of ranges up to `range_max` until `row_cap` rows (the reference instead
//             samples rows with its per-read RNG and stops early by policy -- see DESIGN.md
//             "speculative pipeline vs sequential policy").
//   frame   : refoff = textoff - rdoff, duplicate diagonals dropped (seenDiags1_, :1162-1170),
//             DynProgFramer::frameSeedExtensionRect (dp_framer.cpp:81-129).
//   pick    : best-scoring alignment per read (+ runner-up score).
#include "fm_device.cuh"
#include "dp_device.cuh"
#include "pe_device.cuh"
#include "mapq_device.cuh"
#include "launch.cuh"
#include <new>
#include <cstring>

struct PipeBufs {
	// inputs (device copies for the host-buffer entry point)
	uint8_t *seq, *qual; uint64_t *roff;
	// per-length policy tables
	int32_t *minscByLen, *nceilByLen, *nceilRawByLen, *ivalByLen, *rdgapsByLen, *rfgapsByLen;
	int32_t *interval, *offset;               // per read
	uint8_t *mine; uint64_t *ee;              // exact sweep
	uint64_t *ranges; int32_t *nseeds;        // seed search
	uint64_t *packed; uint32_t *nmask; unsigned long long *nextTask;   // 2-bit reads + task counter
	uint64_t *rows; uint32_t *hitlen, *meta;  // collect (dense: rows of read r at [rowBase[r], +rowCnt[r]))
	uint32_t *nRows, *rowBase, *rowCnt;
	uint64_t *tidx, *textoff, *tlen; uint8_t *rflags;   // resolve
	bt2g_dp_problem *probs; uint32_t *nProb; int32_t *readProb; int32_t *readNProb;
	uint8_t *codes; int32_t *lastH; uint64_t *rawKeys;
	bt2g_dp_summary *summ; bt2g_dp_cand *cands; bt2g_dp_aln *alns; uint8_t *ops;
	bt2g_read_result *res; uint8_t *resOps;
	unsigned long long *counters;             // [4]: sweep sides, seed sides, resolve sides, dp cells
	uint64_t *probTlen, *resTlen;             // reference length per DP problem / per read result
	// paired-end tail
	bt2g_dp_problem *mProbs; uint32_t *nMateProb; int32_t *mateOfRead;
	bt2g_dp_summary *mSumm; bt2g_dp_cand *mCands; bt2g_dp_aln *mAlns; uint8_t *mOps;
	bt2g_pair_result *pairs; unsigned long long *mateCells;
};

struct bt2g_pipeline {
	bt2g_ctx *ctx;
	bt2g_pipeline_params prm;
	bt2g_scoring sc;                          // scoring scheme at creation time
	uint64_t maxReads, maxBases;
	PipeBufs b;
	std::vector<void *> allocs;
	uint64_t numSlots, codeStride, maxProbs;
	int packed = 0;                           // DP kernel mode (dp_kernel_mode)
	uint64_t dpChunk = 0, mateChunk = 0;      // mode 3: problems per fill/tail chunk
	int maxCol, R, sms = 148;
	cudaEvent_t ev[9], pev[4];
	bool pairsOn = false; bt2g_pe_policy pe{}; int mateMaxCol = 0; uint64_t mateCodeStride = 0;
	bt2g_pair_result *hPairs = nullptr;
	bool evOk = false;
	// pinned staging for the host entry point
	uint8_t *hSeq = nullptr, *hQual = nullptr; uint64_t *hOff = nullptr;
	bt2g_read_result *hRes = nullptr; uint8_t *hOps = nullptr;
	uint64_t lastN = 0;
	// copy streams / events of the chunked host entry point
	cudaStream_t sIn = nullptr, sOut = nullptr;
	cudaEvent_t evIn[8], evDone[8];
	bool chunkOk = false;
};

#define PIPE_MAX_RAW 8192
#define META_STRAND(m) (((m) >> 31) & 1u)
#define META_EE(m)     (((m) >> 30) & 1u)
#define META_SEED(m)   (((m) >> 16) & 0x3fffu)

// per-read seed plan from the per-length tables
__global__ void k_plan(const uint64_t *roff, uint64_t n, const int32_t *ivalByLen, int maxLen, int32_t *interval, int32_t *offset) {
	uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if(i >= n) return;
	int len = (int)(roff[i + 1] - roff[i]);
	interval[i] = ivalByLen[len > maxLen ? maxLen : len];
	offset[i] = 0;
}

// collect: one thread per read; rows are appended to one dense list (a contiguous block per read)
__global__ void k_collect(uint64_t n, const uint64_t *roff, const uint64_t *ee, const uint64_t *ranges, const int32_t *nseeds,
                          int maxSeeds, int seedLen, int rowCap, int rangeMax,
                          uint64_t *rows, uint32_t *hitlen, uint32_t *meta, uint32_t *nRows, uint32_t *rowBase, uint32_t *rowCnt) {
	uint64_t rd = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if(rd >= n) return;
	const int len = (int)(roff[rd + 1] - roff[rd]);
	const uint64_t *e = ee + rd * 4;
	const int ns = nseeds[rd];
	const int sl = seedLen < len ? seedLen : len;
	const uint64_t *rg = ranges + rd * 2ull * maxSeeds * 4;
	uint64_t eeTot = (e[1] - e[0]) + (e[3] - e[2]);
	// pass 1: count
	int cnt = 0;
	if(eeTot > 0) cnt = eeTot < (uint64_t)rowCap ? (int)eeTot : rowCap;
	else {
		for(int strand = 0; strand < 2; strand++)
			for(int k = 0; k < ns; k++) {
				const uint64_t *q = rg + ((size_t)strand * maxSeeds + k) * 4;
				const uint64_t sz = q[1] - q[0];
				if(sz >= 1 && sz <= (uint64_t)rangeMax) cnt += (int)sz;
			}
		if(cnt > rowCap) cnt = rowCap;
	}
	const uint32_t base = cnt ? atomicAdd(nRows, (uint32_t)cnt) : 0;
	rowBase[rd] = base; rowCnt[rd] = (uint32_t)cnt;
	uint64_t *ro = rows + base;
	uint32_t *ho = hitlen + base, *mo = meta + base;
	// pass 2: write (exact end-to-end hits first, else seed ranges smallest first)
	int w = 0;
	if(eeTot > 0) {
		for(int strand = 0; strand < 2; strand++)
			for(uint64_t r = e[2 * strand]; r < e[2 * strand + 1] && w < cnt; r++) {
				ro[w] = r; ho[w] = (uint32_t)len; mo[w] = ((uint32_t)strand << 31) | (1u << 30); w++;
			}
	} else {
		for(int sz = 1; sz <= rangeMax && w < cnt; sz++)
			for(int strand = 0; strand < 2 && w < cnt; strand++)
				for(int k = 0; k < ns && w < cnt; k++) {
					const uint64_t *q = rg + ((size_t)strand * maxSeeds + k) * 4;
					if((int)(q[1] - q[0]) != sz) continue;
					for(uint64_t r = q[0]; r < q[1] && w < cnt; r++) {
						ro[w] = r; ho[w] = (uint32_t)sl; mo[w] = ((uint32_t)strand << 31) | ((uint32_t)k << 16); w++;
					}
				}
	}
}

// frame: one thread per read
__global__ void k_frame(uint64_t n, const uint64_t *roff, const int32_t *interval, const int32_t *offset,
                        const uint64_t *rows, const uint32_t *hitlen, const uint32_t *meta,
                        const uint64_t *tidx, const uint64_t *textoff, const uint64_t *tlen, const uint8_t *rflags,
                        const uint32_t *rowBase, const uint32_t *rowCnt,
                        int rowCap, int maxLen, int maxhalf, int matchBonus,
                        const int32_t *minscByLen, const int32_t *nceilRawByLen, const int32_t *rdgapsByLen, const int32_t *rfgapsByLen,
                        bt2g_dp_problem *probs, uint32_t *nProb, uint32_t maxProbs, int32_t *readProb, int32_t *readNProb, bt2g_read_result *res,
                        uint64_t *probTlen, uint64_t *resTlen) {
	uint64_t rd = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if(rd >= n) return;
	const int len = (int)(roff[rd + 1] - roff[rd]);
	const int li = len > maxLen ? maxLen : len;
	bt2g_read_result r;
	r.found = 0; r.score = 0; r.score2 = INT32_MIN; r.fw = 0; r.tidx = 0; r.refoff = 0; r.nops = 0; r.ndp = 0; r.trim_left = 0; r.trim_right = 0; r.mapq = 0; r.pad = 0;
	int np = 0;
	uint64_t seenT[32]; int64_t seenO[32]; uint8_t seenS[32]; int nseen = 0;
	const int minsc = minscByLen[li];
	const uint32_t rb = rowBase[rd], rcnt = rowCnt[rd];
	for(uint32_t i = 0; i < rcnt; i++) {
		uint64_t s = (uint64_t)rb + i;
		uint32_t m = meta[s];
		const bool isEE = META_EE(m) != 0;
		const uint8_t fl = rflags[s];
		if(fl & 2) continue;
		if(isEE && (fl & 1)) continue;                     // eeMode rejects straddlers (aligner_sw_driver.cpp:1141)
		const int strand = (int)META_STRAND(m);
		int rdoff = 0;
		if(!isEE) {
			int depth = (int)META_SEED(m) * interval[rd] + offset[rd];
			rdoff = strand == 0 ? depth : len - depth - (int)hitlen[s];
		}
		const int64_t refoff = (int64_t)textoff[s] - rdoff;
		bool dup = false;
		for(int k = 0; k < nseen; k++) if(seenT[k] == tidx[s] && seenO[k] == refoff && seenS[k] == strand) { dup = true; break; }
		if(dup) continue;
		if(nseen < 32) { seenT[nseen] = tidx[s]; seenO[nseen] = refoff; seenS[nseen] = (uint8_t)strand; nseen++; }
		if(isEE) {
			if(r.found == 0) { r.found = 2; r.score = len * matchBonus; r.fw = strand == 0; r.tidx = tidx[s]; r.refoff = refoff; resTlen[rd] = tlen[s]; }
			else if(r.score2 == INT32_MIN) r.score2 = len * matchBonus;
			continue;
		}
		// DynProgFramer::frameSeedExtensionRect (dp_framer.cpp:81-129), trimToRef
		int maxgap = rdgapsByLen[li] > rfgapsByLen[li] ? rdgapsByLen[li] : rfgapsByLen[li];
		if(maxgap < 0 || maxgap > maxhalf) maxgap = maxhalf;
		int64_t refl = refoff - 2 * maxgap, refr = refoff + (len - 1) + 2 * maxgap;
		const int64_t reflen = (int64_t)tlen[s];
		int64_t triml = 0, trimr = 0;
		if(refr >= reflen) trimr = refr - (reflen - 1);
		if(refl < 0) triml = -refl;
		if(refr - trimr < refl + triml) continue;
		uint32_t pi = atomicAdd(nProb, 1u);
		if(pi >= maxProbs) { atomicSub(nProb, 1u); r.found |= 0x100; break; }   // workspace full: flagged, never silent
		bt2g_dp_problem &p = probs[pi];
		p.read_idx = (uint32_t)rd; p.fw = strand == 0; p.tidx = tidx[s];
		p.refl = refl + triml; p.refr = refr - trimr; p.triml = (int32_t)triml;
		p.corel = maxgap; p.corer = 3 * maxgap; p.minsc = minsc; p.nceil = nceilRawByLen[li]; p.reserved = 0;
		readProb[rd * rowCap + np] = (int32_t)pi;
		probTlen[pi] = tlen[s];
		np++;
	}
	readNProb[rd] = np;
	r.ndp = np;
	res[rd] = r;
}

// pick: one thread per read
__global__ void k_pick(uint64_t n, int rowCap, int maxAlns, int maxOps, const int32_t *readProb, const int32_t *readNProb,
                       const bt2g_dp_problem *probs, const bt2g_dp_summary *summ, const bt2g_dp_aln *alns, const uint8_t *ops,
                       bt2g_read_result *res, uint8_t *resOps, unsigned long long *cellCnt, const uint64_t *roff,
                       const uint64_t *probTlen, uint64_t *resTlen, const int32_t *minscByLen, int maxLen, int matchBonus, int monotone) {
	uint64_t rd = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if(rd >= n) return;
	bt2g_read_result r = res[rd];
	const int np = readNProb[rd];
	int bestP = -1, bestA = 0;
	unsigned long long cells = 0;
	const int len = (int)(roff[rd + 1] - roff[rd]);
	for(int k = 0; k < np; k++) {
		const int pi = readProb[rd * rowCap + k];
		cells += (unsigned long long)len * (unsigned long long)(probs[pi].refr - probs[pi].refl + 1);
		const int na = summ[pi].naln < maxAlns ? summ[pi].naln : maxAlns;
		for(int a = 0; a < na; a++) {
			const bt2g_dp_aln &al = alns[(size_t)pi * maxAlns + a];
			if(r.found == 0 || al.score > r.score) {
				if(r.found) r.score2 = r.score2 > r.score ? r.score2 : r.score;
				r.found = 1; r.score = al.score; bestP = pi; bestA = a;
			} else if(al.score > r.score2) r.score2 = al.score;
		}
	}
	if(bestP >= 0 && r.found == 1) {
		const bt2g_dp_aln &al = alns[(size_t)bestP * maxAlns + bestA];
		r.fw = probs[bestP].fw; r.tidx = probs[bestP].tidx; r.refoff = probs[bestP].refl + al.col0;
		resTlen[rd] = probTlen[bestP];
		r.nops = al.nops < maxOps ? al.nops : maxOps;
		r.trim_left = al.trim_beg; r.trim_right = al.trim_end; r.pad = al.refns;
		const uint8_t *src = ops + ((size_t)bestP * maxAlns + bestA) * maxOps;
		uint8_t *dst = resOps + rd * (size_t)maxOps;
		for(int k = 0; k < r.nops; k++) dst[k] = src[k];
	}
	if((r.found & 0xff) != 0) {
		const int li = len > maxLen ? maxLen : len;
		r.mapq = mapq_v2(r.score, r.score2 != INT32_MIN, r.score2, minscByLen[li], (long long)len * matchBonus, monotone != 0);
	}
	res[rd] = r;
	if(cellCnt && cells) atomicAdd(cellCnt, cells);
}


// ---- paired-end tail ------------------------------------------------------------------------
// number of reference positions an alignment covers: ops are M/MM (read+ref), READGAP (ref only), REFGAP (read only)
__device__ __forceinline__ int pe_ref_extent(const bt2g_read_result &r, const uint8_t *ops, int len) {
	if(r.found == 2) return len;
	int e = 0;
	for(int k = 0; k < r.nops; k++) e += (ops[k] & 3) != BT2G_OP_REFGAP;
	return e;
}

// frame: one thread per read (the anchor); emits at most one mate-finding DP problem for the opposite mate
__global__ void k_frame_mates(uint64_t nReads, const uint64_t *roff, const bt2g_read_result *res, const uint8_t *resOps, int maxOps,
                              const uint64_t *resTlen, bt2g_pe_policy pp, int maxLen, int maxhalf, int mateMaxCol,
                              const int32_t *minscByLen, const int32_t *nceilRawByLen, const int32_t *rdgapsByLen, const int32_t *rfgapsByLen,
                              bt2g_dp_problem *mProbs, uint32_t *nMateProb, int32_t *mateOfRead) {
	const uint64_t rd = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if(rd >= nReads) return;
	mateOfRead[rd] = -1;
	const bt2g_read_result a = res[rd];
	if((a.found & 0xff) == 0) return;
	const uint64_t od = rd ^ 1ull;
	const bt2g_read_result o = res[od];
	const int alen = (int)(roff[rd + 1] - roff[rd]), olen = (int)(roff[od + 1] - roff[od]);
	const bool anchor1 = (rd & 1ull) == 0;
	if((o.found & 0xff) != 0 && o.tidx == a.tidx) {
		// the two independent alignments may already be a concordant pair
		const int ea = pe_ref_extent(a, resOps + rd * (size_t)maxOps, alen), eo = pe_ref_extent(o, resOps + od * (size_t)maxOps, olen);
		const int k = anchor1 ? pe_classify(pp, a.refoff, (uint64_t)ea, a.fw != 0, o.refoff, (uint64_t)eo, o.fw != 0)
		                      : pe_classify(pp, o.refoff, (uint64_t)eo, o.fw != 0, a.refoff, (uint64_t)ea, a.fw != 0);
		if(k != 5) return;
	}
	const int li = olen > maxLen ? maxLen : olen;
	bt2g_mate_anchor an;
	an.off = a.refoff; an.reflen = resTlen[rd];
	an.len1 = (uint32_t)(anchor1 ? alen : olen); an.len2 = (uint32_t)(anchor1 ? olen : alen);
	an.maxrdgap = rdgapsByLen[li]; an.maxrfgap = rfgapsByLen[li];
	an.maxalcols = olen + an.maxrdgap;
	an.maxns = nceilRawByLen[li]; an.maxhalf = maxhalf;
	an.is1 = anchor1; an.fw = a.fw != 0; an.pad[0] = an.pad[1] = 0;
	bt2g_mate_frame f;
	pe_frame_anchor(pp, an, f);
	if(f.status != 2) return;
	if(f.refr - f.refl + 1 > mateMaxCol) return;           // wider than the workspace: not attempted
	const uint32_t pi = atomicAdd(nMateProb, 1u);
	bt2g_dp_problem &q = mProbs[pi];
	q.read_idx = (uint32_t)od; q.fw = f.ofw; q.tidx = a.tidx;
	q.refl = f.refl; q.refr = f.refr; q.triml = (int32_t)f.triml;
	q.corel = (int32_t)f.corel; q.corer = (int32_t)f.corer;
	q.minsc = minscByLen[li]; q.nceil = nceilRawByLen[li]; q.reserved = 0;
	mateOfRead[rd] = (int32_t)pi;
}

// pick: one thread per pair
__global__ void k_pick_pairs(uint64_t nPairs, const uint64_t *roff, bt2g_read_result *res, uint8_t *resOps, int maxOps, int maxAlns,
                             bt2g_pe_policy pp, const int32_t *mateOfRead, const bt2g_dp_problem *mProbs, const bt2g_dp_summary *mSumm,
                             const bt2g_dp_aln *mAlns, const uint8_t *mOps, bt2g_pair_result *pairs, unsigned long long *mateCells,
                             const int32_t *minscByLen, int maxLen, int matchBonus, int monotone) {
	const uint64_t pr = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if(pr >= nPairs) return;
	const uint64_t r1 = 2 * pr, r2 = 2 * pr + 1;
	bt2g_read_result a1 = res[r1], a2 = res[r2];
	const int len1 = (int)(roff[r1 + 1] - roff[r1]), len2 = (int)(roff[r2 + 1] - roff[r2]);
	const bool f1 = (a1.found & 0xff) != 0, f2 = (a2.found & 0xff) != 0;
	bt2g_pair_result out;
	out.pair_type = (f1 && f2) ? 2 : ((f1 || f2) ? 3 : 0); out.kind = 5; out.source = 0; out.score_sum = 0; out.fraglen = 0;
	int bestSum = INT32_MIN, bestSrc = -1, bestKind = 5, bestAln = 0;
	// the runner-up concordant sum (for the pair's MAPQ, unique.h:205-222: a repeat with several equally good concordant
	// placements must not report 42): every other concordant (anchor, mate alignment) combination seen here, and each mate's
	// own runner-up alignment paired with the other mate's best
	int secSum = INT32_MIN;
	auto offer = [&](int sum) { if(sum > bestSum) { secSum = bestSum; bestSum = sum; return true; } if(sum > secSum) secSum = sum; return false; };
	const int e1 = f1 ? pe_ref_extent(a1, resOps + r1 * (size_t)maxOps, len1) : 0;
	const int e2 = f2 ? pe_ref_extent(a2, resOps + r2 * (size_t)maxOps, len2) : 0;
	if(f1 && f2 && a1.tidx == a2.tidx) {
		const int k = pe_classify(pp, a1.refoff, (uint64_t)e1, a1.fw != 0, a2.refoff, (uint64_t)e2, a2.fw != 0);
		if(k != 5) { offer(a1.score + a2.score); bestSrc = 0; bestKind = k; }
	}
	unsigned long long cells = 0;
	// anchor = mate 1 (source 1: mate 2 from the mate DP), anchor = mate 2 (source 2)
	for(int src = 1; src <= 2; src++) {
		const uint64_t ra = src == 1 ? r1 : r2;
		const bool fa = src == 1 ? f1 : f2;
		if(!fa) continue;
		const int pi = mateOfRead[ra];
		if(pi < 0) continue;
		const bt2g_dp_problem &q = mProbs[pi];
		cells += (unsigned long long)(src == 1 ? len2 : len1) * (unsigned long long)(q.refr - q.refl + 1);
		const int na = mSumm[pi].naln < maxAlns ? mSumm[pi].naln : maxAlns;
		const bt2g_read_result &an = src == 1 ? a1 : a2;
		const int ea = src == 1 ? e1 : e2;
		for(int k = 0; k < na; k++) {
			const bt2g_dp_aln &al = mAlns[(size_t)pi * maxAlns + k];
			const uint8_t *o = mOps + ((size_t)pi * maxAlns + k) * maxOps;
			int em = 0;
			const int no = al.nops < maxOps ? al.nops : maxOps;
			for(int x = 0; x < no; x++) em += (o[x] & 3) != BT2G_OP_REFGAP;
			const int64_t moff = q.refl + al.col0;
			const int kind = src == 1 ? pe_classify(pp, an.refoff, (uint64_t)ea, an.fw != 0, moff, (uint64_t)em, q.fw != 0)
			                          : pe_classify(pp, moff, (uint64_t)em, q.fw != 0, an.refoff, (uint64_t)ea, an.fw != 0);
			if(kind == 5) continue;
			const int sum = an.score + al.score;
			if(offer(sum)) { bestSrc = src; bestKind = kind; bestAln = k; }
		}
	}
	if(bestSrc > 0) {
		// replace the opposite mate's result by the mate-DP alignment
		const uint64_t ra = bestSrc == 1 ? r1 : r2, ro = bestSrc == 1 ? r2 : r1;
		const int pi = mateOfRead[ra];
		const bt2g_dp_problem &q = mProbs[pi];
		const bt2g_dp_aln &al = mAlns[(size_t)pi * maxAlns + bestAln];
		bt2g_read_result m = res[ro];
		if((m.found & 0xff) != 0 && m.score > m.score2) m.score2 = m.score;   // the displaced alignment becomes the runner-up
		m.found = (m.found & ~0xff) | 1; m.score = al.score; m.fw = q.fw; m.tidx = q.tidx; m.refoff = q.refl + al.col0;
		m.nops = al.nops < maxOps ? al.nops : maxOps; m.trim_left = al.trim_beg; m.trim_right = al.trim_end; m.pad = al.refns;
		const uint8_t *src = mOps + ((size_t)pi * maxAlns + bestAln) * maxOps;
		uint8_t *dst = resOps + ro * (size_t)maxOps;
		for(int k = 0; k < m.nops; k++) dst[k] = src[k];
		res[ro] = m;
		if(bestSrc == 1) a2 = m; else a1 = m;
	}
	if(bestSrc >= 0) {
		out.pair_type = 1; out.kind = bestKind; out.source = bestSrc; out.score_sum = bestSum;
		const int ee1 = pe_ref_extent(a1, resOps + r1 * (size_t)maxOps, len1), ee2 = pe_ref_extent(a2, resOps + r2 * (size_t)maxOps, len2);
		const int64_t lo = a1.refoff < a2.refoff ? a1.refoff : a2.refoff;
		const int64_t h1 = a1.refoff + ee1, h2 = a2.refoff + ee2;
		out.fraglen = (h1 > h2 ? h1 : h2) - lo;
		// MAPQ of a concordant pair: both mates from the pair's sums (unique.h:205-222)
		const int l1 = len1 > maxLen ? maxLen : len1, l2 = len2 > maxLen ? maxLen : len2;
		if(f1 && a1.score2 > INT32_MIN / 2 && (long long)a1.score2 + a2.score > secSum) secSum = a1.score2 + a2.score;
		if(f2 && a2.score2 > INT32_MIN / 2 && (long long)a1.score + a2.score2 > secSum) secSum = a1.score + a2.score2;
		if(secSum > bestSum) secSum = bestSum;
		const long long minPair = (long long)minscByLen[l1] + minscByLen[l2];
		const bool hasSec = secSum > INT32_MIN / 2 && secSum >= minPair;
		const int mq = mapq_v2(bestSum, hasSec, hasSec ? secSum : 0, minPair, (long long)(len1 + len2) * matchBonus, monotone != 0);
		res[r1].mapq = mq; res[r2].mapq = mq;
	}
	pairs[pr] = out;
	if(mateCells && cells) atomicAdd(mateCells, cells);
}

template <typename T> static int pipeAlloc(bt2g_pipeline *p, T *&ptr, uint64_t count) {
	void *v = nullptr;
	cudaError_t e = cudaMalloc(&v, (count ? count : 1) * sizeof(T));
	if(e != cudaSuccess) { p->ctx->err = std::string("pipeline cudaMalloc: ") + cudaGetErrorString(e); return -2; }
	p->allocs.push_back(v);
	ptr = (T *)v;
	return 0;
}

template <typename OFF>
static int runStages(bt2g_pipeline *p, const uint8_t *seq, const uint8_t *qual, const uint64_t *roff, uint64_t n, cudaStream_t st, bool count,
                     uint64_t resBase = 0) {
	bt2g_ctx *ctx = p->ctx;
	PipeBufs &b = p->b;
	const bt2g_pipeline_params &q = p->prm;
	DevIndex<OFF> ix = bt2g_dev_index<OFF>(ctx);
	unsigned long long *c = count ? b.counters : nullptr;
	const unsigned T = 128;
	auto grid = [&](uint64_t m) { return (unsigned)((m + T - 1) / T); };
	auto mark = [&](int i) { if(p->evOk) cudaEventRecord(p->ev[i], st); };
	if(count) BT2G_CUDA_TRY(ctx, cudaMemsetAsync(b.counters, 0, 4 * sizeof(unsigned long long), st));
	BT2G_CUDA_TRY(ctx, cudaMemsetAsync(b.nProb, 0, sizeof(uint32_t), st));
	BT2G_CUDA_TRY(ctx, cudaMemsetAsync(b.nRows, 0, sizeof(uint32_t), st));
	mark(0);
	k_plan<<<grid(n), T, 0, st>>>(roff, n, b.ivalByLen, q.max_len, b.interval, b.offset);
	mark(1);
	launch_pack_reads(seq, roff, n, q.max_len, b.packed, b.nmask, st);
	launch_exact_sweep2<OFF>(ix, roff, n, 0, 0, b.mine, b.ee, b.packed, b.nmask, b.nextTask, p->sms, st, c ? c + 0 : nullptr, 1 /* ee ranges only */);
	mark(2);
	launch_seed_search2<OFF>(ix, seq, roff, n, q.max_len, q.seed_len, q.max_seeds, 0, 0, b.interval, b.offset, b.ranges, b.nseeds,
	                         b.packed, b.nmask, b.nextTask, p->sms, st, c ? c + 1 : nullptr);
	mark(3);
	k_collect<<<grid(n), T, 0, st>>>(n, roff, b.ee, b.ranges, b.nseeds, q.max_seeds, q.seed_len, q.row_cap, q.range_max, b.rows, b.hitlen, b.meta,
	                                 b.nRows, b.rowBase, b.rowCnt);
	mark(4);
	launch_resolve2<OFF>(ix, b.rows, b.hitlen, 0, b.nRows, 0, nullptr, b.tidx, b.textoff, b.tlen, b.rflags, b.nextTask, p->sms, st, c ? c + 2 : nullptr);
	mark(5);
	k_frame<<<grid(n), T, 0, st>>>(n, roff, b.interval, b.offset, b.rows, b.hitlen, b.meta, b.tidx, b.textoff, b.tlen, b.rflags,
	                               b.rowBase, b.rowCnt, q.row_cap, q.max_len, q.maxhalf, p->sc.match_bonus,
	                               b.minscByLen, b.nceilRawByLen, b.rdgapsByLen, b.rfgapsByLen,
	                               b.probs, b.nProb, (uint32_t)p->maxProbs, b.readProb, b.readNProb, b.res + resBase, b.probTlen, b.resTlen + resBase);
	DpLaunch L;
	L.seq = seq; L.qual = qual; L.roff = roff; L.probs = b.probs; L.n = p->maxProbs; L.nDev = b.nProb;
	L.rawKeys = b.rawKeys; L.maxRaw = b.rawKeys ? PIPE_MAX_RAW : 0;
	L.numSlots = p->numSlots; L.codes = b.codes; L.lastH = b.lastH; L.codeStride = p->codeStride; L.maxCol = p->maxCol;
	L.maxCands = q.max_cands; L.maxAlns = q.max_alns; L.maxOps = q.max_ops; L.packed = p->packed; L.chunk = p->dpChunk;
	L.summ = b.summ; L.cands = b.cands; L.alns = b.alns; L.ops = b.ops;
	mark(6);
	const int drc = p->sc.local ? launch_dp_local<OFF>(ix, p->sc, L, q.max_len, st) : launch_dp_e2e<OFF>(ix, p->sc, L, q.max_len, st);
	if(drc) { ctx->err = "pipeline: DP launch rejected"; return -1; }
	mark(7);
	k_pick<<<grid(n), T, 0, st>>>(n, q.row_cap, q.max_alns, q.max_ops, b.readProb, b.readNProb, b.probs, b.summ, b.alns, b.ops,
	                              b.res + resBase, b.resOps + resBase * (uint64_t)q.max_ops, c ? c + 3 : nullptr, roff, b.probTlen, b.resTlen + resBase, b.minscByLen, q.max_len, p->sc.match_bonus, p->sc.match_bonus == 0);
	mark(8);
	BT2G_CUDA_TRY(ctx, cudaGetLastError());
	p->lastN = n;
	return 0;
}

template <typename OFF>
static int runPairTail(bt2g_pipeline *p, const uint8_t *seq, const uint8_t *qual, const uint64_t *roff, uint64_t nPairs, cudaStream_t st, bool count,
                       uint64_t resBase = 0) {
	bt2g_ctx *ctx = p->ctx;
	PipeBufs &b = p->b;
	const bt2g_pipeline_params &q = p->prm;
	DevIndex<OFF> ix = bt2g_dev_index<OFF>(ctx);
	const uint64_t n = 2 * nPairs;
	const unsigned T = 128;
	bt2g_read_result *res = b.res + resBase; uint8_t *resOps = b.resOps + resBase * (uint64_t)q.max_ops;
	const uint64_t *resTlen = b.resTlen + resBase; bt2g_pair_result *pairs = b.pairs + resBase / 2;
	BT2G_CUDA_TRY(ctx, cudaMemsetAsync(b.nMateProb, 0, sizeof(uint32_t), st));
	BT2G_CUDA_TRY(ctx, cudaMemsetAsync(b.mateCells, 0, sizeof(unsigned long long), st));
	cudaEventRecord(p->pev[0], st);
	k_frame_mates<<<(unsigned)((n + T - 1) / T), T, 0, st>>>(n, roff, res, resOps, q.max_ops, resTlen, p->pe, q.max_len, q.maxhalf, p->mateMaxCol,
	                                                         b.minscByLen, b.nceilRawByLen, b.rdgapsByLen, b.rfgapsByLen, b.mProbs, b.nMateProb, b.mateOfRead);
	cudaEventRecord(p->pev[1], st);
	DpLaunch L;
	L.seq = seq; L.qual = qual; L.roff = roff; L.probs = b.mProbs; L.n = p->maxReads; L.nDev = b.nMateProb;
	L.rawKeys = nullptr; L.maxRaw = 0;
	L.numSlots = p->numSlots; L.codes = b.codes; L.lastH = nullptr; L.codeStride = p->mateCodeStride; L.maxCol = p->mateMaxCol;
	L.maxCands = q.max_cands; L.maxAlns = q.max_alns; L.maxOps = q.max_ops; L.packed = p->packed; L.chunk = p->mateChunk;
	L.summ = b.mSumm; L.cands = b.mCands; L.alns = b.mAlns; L.ops = b.mOps;
	if(launch_dp_e2e<OFF>(ix, p->sc, L, q.max_len, st)) { ctx->err = "pipeline: mate DP launch rejected"; return -1; }
	cudaEventRecord(p->pev[2], st);
	k_pick_pairs<<<(unsigned)((nPairs + T - 1) / T), T, 0, st>>>(nPairs, roff, res, resOps, q.max_ops, q.max_alns, p->pe, b.mateOfRead, b.mProbs,
	                                                             b.mSumm, b.mAlns, b.mOps, pairs, count ? b.mateCells : nullptr, b.minscByLen, q.max_len, p->sc.match_bonus, p->sc.match_bonus == 0);
	cudaEventRecord(p->pev[3], st);
	BT2G_CUDA_TRY(ctx, cudaGetLastError());
	return 0;
}

extern "C" {

int bt2g_pipeline_create(bt2g_ctx *ctx, const bt2g_pipeline_params *prm, uint64_t maxReads, uint64_t maxBases, bt2g_pipeline **out) {
	if(!ctx || !prm || !out) return -1;
	if(!ctx->loaded) { ctx->err = "no index loaded"; return -1; }
	if(ctx->scoring.gapbar < 1) bt2g_scoring_default(&ctx->scoring, 0);
	if(prm->seed_len > 32) { ctx->err = "pipeline: seed length must be <= 32"; return -1; }
	if(prm->max_len < 1 || prm->max_len > 512 || prm->row_cap < 1 || prm->row_cap > 32 || prm->max_seeds < 1 || prm->max_seeds > 16383) {
		ctx->err = "pipeline: bad parameters"; return -1;
	}
	cudaSetDevice(ctx->device);
	bt2g_pipeline *p = new(std::nothrow) bt2g_pipeline();
	if(!p) return -4;
	p->ctx = ctx; p->prm = *prm; p->sc = ctx->scoring; p->maxReads = maxReads; p->maxBases = maxBases;
	PipeBufs &b = p->b;
	memset(&b, 0, sizeof(b));
	const uint64_t n = maxReads, cap = prm->row_cap, nrowMax = n * cap;
	const uint64_t nprobMax = (prm->max_probs > 0 && (uint64_t)prm->max_probs < nrowMax) ? (uint64_t)prm->max_probs : nrowMax;
	p->maxProbs = nprobMax;
	int rc = 0;
	const int L1 = prm->max_len + 1;
	rc |= pipeAlloc(p, b.seq, maxBases); rc |= pipeAlloc(p, b.qual, maxBases); rc |= pipeAlloc(p, b.roff, n + 1);
	rc |= pipeAlloc(p, b.minscByLen, L1); rc |= pipeAlloc(p, b.nceilByLen, L1); rc |= pipeAlloc(p, b.nceilRawByLen, L1);
	rc |= pipeAlloc(p, b.ivalByLen, L1); rc |= pipeAlloc(p, b.rdgapsByLen, L1); rc |= pipeAlloc(p, b.rfgapsByLen, L1);
	rc |= pipeAlloc(p, b.interval, n); rc |= pipeAlloc(p, b.offset, n);
	rc |= pipeAlloc(p, b.mine, n * 2); rc |= pipeAlloc(p, b.ee, n * 4);
	rc |= pipeAlloc(p, b.ranges, n * 2ull * prm->max_seeds * 4); rc |= pipeAlloc(p, b.nseeds, n);
	rc |= pipeAlloc(p, b.packed, (maxBases >> 5) + n + 2); rc |= pipeAlloc(p, b.nmask, (maxBases >> 5) + n + 2); rc |= pipeAlloc(p, b.nextTask, 1);
	rc |= pipeAlloc(p, b.nRows, 1); rc |= pipeAlloc(p, b.rowBase, n); rc |= pipeAlloc(p, b.rowCnt, n);
	rc |= pipeAlloc(p, b.rows, nrowMax); rc |= pipeAlloc(p, b.hitlen, nrowMax); rc |= pipeAlloc(p, b.meta, nrowMax);
	rc |= pipeAlloc(p, b.tidx, nrowMax); rc |= pipeAlloc(p, b.textoff, nrowMax); rc |= pipeAlloc(p, b.tlen, nrowMax); rc |= pipeAlloc(p, b.rflags, nrowMax);
	rc |= pipeAlloc(p, b.probs, nprobMax); rc |= pipeAlloc(p, b.nProb, 1); rc |= pipeAlloc(p, b.readProb, nrowMax); rc |= pipeAlloc(p, b.readNProb, n);
	p->maxCol = prm->max_len + 4 * prm->maxhalf + 4;
	int sms = 148; cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
	p->sms = sms;
	p->numSlots = (uint64_t)sms * 24;
	{
		int64_t mn = 0;
		for(int l = 1; l <= prm->max_len; l++) if(prm->minsc_by_len[l] < mn) mn = prm->minsc_by_len[l];
		p->packed = p->sc.local ? 0 : dp_kernel_mode(p->sc, mn, prm->max_len, ctx->dpModeCap);
	}
	p->R = dp_rows_per_lane(prm->max_len, p->packed);
	p->codeStride = dp_code_stride(p->maxCol, prm->max_len, p->packed);
	if(p->packed == 3) {
		p->dpChunk = dp_chunk_problems(p->codeStride, nprobMax);
		rc |= pipeAlloc(p, b.codes, p->dpChunk * p->codeStride);
	} else {
		rc |= pipeAlloc(p, b.codes, p->numSlots * p->codeStride * (p->packed ? 2 : 1));
	} rc |= pipeAlloc(p, b.lastH, p->numSlots * (uint64_t)p->maxCol);
	// local mode gathers candidate cells during the fill (k_dp_local): a raw key list per warp slot
	if(ctx->scoring.local) rc |= pipeAlloc(p, b.rawKeys, p->numSlots * (uint64_t)PIPE_MAX_RAW);
	rc |= pipeAlloc(p, b.summ, nprobMax); rc |= pipeAlloc(p, b.cands, nprobMax * prm->max_cands);
	rc |= pipeAlloc(p, b.alns, nprobMax * prm->max_alns); rc |= pipeAlloc(p, b.ops, nprobMax * prm->max_alns * (uint64_t)prm->max_ops);
	rc |= pipeAlloc(p, b.res, n); rc |= pipeAlloc(p, b.resOps, n * (uint64_t)prm->max_ops);
	rc |= pipeAlloc(p, b.counters, 4);
	rc |= pipeAlloc(p, b.probTlen, nprobMax); rc |= pipeAlloc(p, b.resTlen, n);
	if(rc) { bt2g_pipeline_destroy(p); return -2; }
	cudaError_t e = cudaSuccess;
	auto up = [&](int32_t *dst, const int32_t *src) { if(e == cudaSuccess) e = cudaMemcpy(dst, src, L1 * sizeof(int32_t), cudaMemcpyHostToDevice); };
	up(b.minscByLen, prm->minsc_by_len); up(b.nceilByLen, prm->nceil_by_len); up(b.nceilRawByLen, prm->nceil_raw_by_len);
	up(b.ivalByLen, prm->interval_by_len); up(b.rdgapsByLen, prm->rdgaps_by_len); up(b.rfgapsByLen, prm->rfgaps_by_len);
	if(e == cudaSuccess) e = cudaMemset(b.alns, 0, nprobMax * prm->max_alns * sizeof(bt2g_dp_aln));
	if(e == cudaSuccess) e = cudaMemset(b.cands, 0, nprobMax * prm->max_cands * sizeof(bt2g_dp_cand));
	// pinned staging
	if(e == cudaSuccess) e = cudaHostAlloc((void **)&p->hSeq, maxBases, cudaHostAllocDefault);
	if(e == cudaSuccess) e = cudaHostAlloc((void **)&p->hQual, maxBases, cudaHostAllocDefault);
	if(e == cudaSuccess) e = cudaHostAlloc((void **)&p->hOff, (n + 1) * 8, cudaHostAllocDefault);
	if(e == cudaSuccess) e = cudaHostAlloc((void **)&p->hRes, n * sizeof(bt2g_read_result), cudaHostAllocDefault);
	if(e == cudaSuccess) e = cudaHostAlloc((void **)&p->hOps, n * (uint64_t)prm->max_ops, cudaHostAllocDefault);
	if(e != cudaSuccess) { ctx->err = std::string("pipeline setup: ") + cudaGetErrorString(e); bt2g_pipeline_destroy(p); return -2; }
	p->evOk = true;
	for(int i = 0; i < 9; i++) if(cudaEventCreate(&p->ev[i]) != cudaSuccess) p->evOk = false;
	p->chunkOk = cudaStreamCreateWithFlags(&p->sIn, cudaStreamNonBlocking) == cudaSuccess &&
	             cudaStreamCreateWithFlags(&p->sOut, cudaStreamNonBlocking) == cudaSuccess;
	for(int i = 0; i < 8 && p->chunkOk; i++)
		p->chunkOk = cudaEventCreateWithFlags(&p->evIn[i], cudaEventDisableTiming) == cudaSuccess &&
		             cudaEventCreateWithFlags(&p->evDone[i], cudaEventDisableTiming) == cudaSuccess;
	// the params struct keeps host pointers that may die; null them
	p->prm.minsc_by_len = p->prm.nceil_by_len = p->prm.nceil_raw_by_len = p->prm.interval_by_len = p->prm.rdgaps_by_len = p->prm.rfgaps_by_len = nullptr;
	*out = p;
	return 0;
}

void bt2g_pipeline_destroy(bt2g_pipeline *p) {
	if(!p) return;
	cudaSetDevice(p->ctx->device);
	for(void *v : p->allocs) cudaFree(v);
	if(p->evOk) for(int i = 0; i < 9; i++) cudaEventDestroy(p->ev[i]);
	if(p->chunkOk) { for(int i = 0; i < 8; i++) { cudaEventDestroy(p->evIn[i]); cudaEventDestroy(p->evDone[i]); } }
	if(p->sIn) cudaStreamDestroy(p->sIn);
	if(p->sOut) cudaStreamDestroy(p->sOut);
	if(p->hSeq) cudaFreeHost(p->hSeq);
	if(p->hQual) cudaFreeHost(p->hQual);
	if(p->hOff) cudaFreeHost(p->hOff);
	if(p->hRes) cudaFreeHost(p->hRes);
	if(p->hOps) cudaFreeHost(p->hOps);
	if(p->hPairs) cudaFreeHost(p->hPairs);
	if(p->pairsOn) for(int i = 0; i < 4; i++) cudaEventDestroy(p->pev[i]);
	delete p;
}

int bt2g_pipeline_run_dev(bt2g_pipeline *p, const uint8_t *dSeq, const uint8_t *dQual, const uint64_t *dOff,
                          uint64_t nReads, void *stream, int count) {
	if(!p || !dSeq || !dQual || !dOff) return -1;
	if(nReads > p->maxReads) { p->ctx->err = "pipeline: batch larger than max_reads"; return -1; }
	if(nReads == 0) return 0;
	BT2G_CUDA_TRY(p->ctx, cudaSetDevice(p->ctx->device));
	cudaStream_t st = stream ? (cudaStream_t)stream : p->ctx->stream;
	if(p->ctx->info.off_size == 4) return runStages<uint32_t>(p, dSeq, dQual, dOff, nReads, st, count != 0);
	return runStages<uint64_t>(p, dSeq, dQual, dOff, nReads, st, count != 0);
}

int bt2g_pipeline_run_host(bt2g_pipeline *p, const bt2g_reads *reads, bt2g_read_result *res, uint8_t *ops) {
	if(!p || !reads || !reads->qual || !res) return -1;
	bt2g_ctx *ctx = p->ctx;
	const uint64_t n = reads->n_reads;
	if(n > p->maxReads || reads->off[n] > p->maxBases) { ctx->err = "pipeline: batch larger than the pipeline was created for"; return -1; }
	if(n == 0) return 0;
	BT2G_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
	cudaStream_t st = ctx->stream;
	const uint64_t nb = reads->off[n];
	const uint64_t maxOps = (uint64_t)p->prm.max_ops;
	// Large batches go through in chunks: the upload of chunk c+1 and the download of chunk c-1 run on
	// their own streams (both copy engines) while chunk c computes.  Caller buffers may be pageable:
	// the copies are then staged by the driver and overlap less.
	uint64_t chunkMin = 1u << 18;
	if(const char *e = getenv("BT2G_HOST_CHUNK_MIN")) chunkMin = strtoull(e, nullptr, 10);
	const int nChunks = (p->chunkOk && n >= chunkMin && n >= 4) ? 4 : 1;
	if(nChunks == 1) {
		BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(p->b.seq, reads->seq, nb, cudaMemcpyHostToDevice, st));
		BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(p->b.qual, reads->qual, nb, cudaMemcpyHostToDevice, st));
		BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(p->b.roff, reads->off, (n + 1) * 8, cudaMemcpyHostToDevice, st));
		int rc = bt2g_pipeline_run_dev(p, p->b.seq, p->b.qual, p->b.roff, n, st, 0);
		if(rc) return rc;
		BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(res, p->b.res, n * sizeof(bt2g_read_result), cudaMemcpyDeviceToHost, st));
		if(ops) BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(ops, p->b.resOps, n * maxOps, cudaMemcpyDeviceToHost, st));
		BT2G_CUDA_TRY(ctx, cudaStreamSynchronize(st));
		return 0;
	}
	BT2G_CUDA_TRY(ctx, cudaStreamSynchronize(st));                 // earlier work on the compute stream owns the buffers
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(p->b.roff, reads->off, (n + 1) * 8, cudaMemcpyHostToDevice, p->sIn));
	const uint64_t per = (n + nChunks - 1) / nChunks;
	for(int c = 0; c < nChunks; c++) {
		const uint64_t s0 = c * per, s1 = (s0 + per < n) ? s0 + per : n;
		const uint64_t b0 = reads->off[s0], b1 = reads->off[s1];
		BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(p->b.seq + b0, reads->seq + b0, b1 - b0, cudaMemcpyHostToDevice, p->sIn));
		BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(p->b.qual + b0, reads->qual + b0, b1 - b0, cudaMemcpyHostToDevice, p->sIn));
		BT2G_CUDA_TRY(ctx, cudaEventRecord(p->evIn[c], p->sIn));
	}
	for(int c = 0; c < nChunks; c++) {
		const uint64_t s0 = c * per, s1 = (s0 + per < n) ? s0 + per : n;
		BT2G_CUDA_TRY(ctx, cudaStreamWaitEvent(st, p->evIn[c], 0));
		int rc;
		if(ctx->info.off_size == 4) rc = runStages<uint32_t>(p, p->b.seq, p->b.qual, p->b.roff + s0, s1 - s0, st, false, s0);
		else rc = runStages<uint64_t>(p, p->b.seq, p->b.qual, p->b.roff + s0, s1 - s0, st, false, s0);
		if(rc) return rc;
		BT2G_CUDA_TRY(ctx, cudaEventRecord(p->evDone[c], st));
		BT2G_CUDA_TRY(ctx, cudaStreamWaitEvent(p->sOut, p->evDone[c], 0));
		BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(res + s0, p->b.res + s0, (s1 - s0) * sizeof(bt2g_read_result), cudaMemcpyDeviceToHost, p->sOut));
		if(ops) BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(ops + s0 * maxOps, p->b.resOps + s0 * maxOps, (s1 - s0) * maxOps, cudaMemcpyDeviceToHost, p->sOut));
	}
	BT2G_CUDA_TRY(ctx, cudaStreamSynchronize(p->sOut));
	BT2G_CUDA_TRY(ctx, cudaStreamSynchronize(st));
	p->lastN = n;
	return 0;
}

int bt2g_pipeline_enable_pairs(bt2g_pipeline *p, const bt2g_pe_policy *pol) {
	if(!p || !pol) return -1;
	bt2g_ctx *ctx = p->ctx;
	if(pol->pol < 1 || pol->pol > 4) { ctx->err = "pipeline: bad paired-end policy"; return -1; }
	if(p->sc.local) { ctx->err = "pipeline: paired-end pass is end-to-end only in this build"; return -1; }
	if(p->pairsOn) { p->pe = *pol; return 0; }
	BT2G_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
	PipeBufs &b = p->b;
	const bt2g_pipeline_params &q = p->prm;
	const uint64_t n = p->maxReads;
	// widest mate rectangle: (maxfrag [expanded to the longer mate]) + rdlen - 1 + 2 * maxgap columns
	uint64_t maxfrag = pol->maxfrag > (uint64_t)q.max_len ? pol->maxfrag : (uint64_t)q.max_len;
	const int maxgap = q.maxhalf > 32 ? q.maxhalf : 32;
	p->mateMaxCol = (int)(maxfrag + q.max_len + 2 * maxgap + 8);
	if(p->mateMaxCol > 8192) { ctx->err = "pipeline: -X too large for the mate-finding workspace"; return -1; }
	p->mateCodeStride = dp_code_stride(p->mateMaxCol, q.max_len, p->packed);
	int rc = 0;
	uint8_t *codes2 = nullptr;
	if(p->packed == 3) {
		p->mateChunk = dp_chunk_problems(p->mateCodeStride, n);
		const uint64_t need = p->mateChunk * p->mateCodeStride, have = p->dpChunk * p->codeStride;
		rc |= pipeAlloc(p, codes2, need > have ? need : have);
	} else {
		rc |= pipeAlloc(p, codes2, p->numSlots * p->mateCodeStride * (p->packed ? 2 : 1));
	}
	rc |= pipeAlloc(p, b.mProbs, n); rc |= pipeAlloc(p, b.nMateProb, 1); rc |= pipeAlloc(p, b.mateOfRead, n);
	rc |= pipeAlloc(p, b.mSumm, n); rc |= pipeAlloc(p, b.mCands, n * q.max_cands);
	rc |= pipeAlloc(p, b.mAlns, n * q.max_alns); rc |= pipeAlloc(p, b.mOps, n * q.max_alns * (uint64_t)q.max_ops);
	rc |= pipeAlloc(p, b.pairs, n / 2 + 1); rc |= pipeAlloc(p, b.mateCells, 1);
	if(rc) return -2;
	b.codes = codes2;        // the wider workspace serves both DP passes
	if(p->packed != 3) p->codeStride = p->mateCodeStride;
	cudaError_t e = cudaMemset(b.mAlns, 0, n * q.max_alns * sizeof(bt2g_dp_aln));
	if(e == cudaSuccess) e = cudaMemset(b.mCands, 0, n * q.max_cands * sizeof(bt2g_dp_cand));
	if(e == cudaSuccess) e = cudaHostAlloc((void **)&p->hPairs, (n / 2 + 1) * sizeof(bt2g_pair_result), cudaHostAllocDefault);
	for(int i = 0; i < 4 && e == cudaSuccess; i++) e = cudaEventCreate(&p->pev[i]);
	if(e != cudaSuccess) { ctx->err = std::string("pipeline pairs setup: ") + cudaGetErrorString(e); return -2; }
	p->pe = *pol; p->pairsOn = true;
	return 0;
}

int bt2g_pipeline_run_paired_dev(bt2g_pipeline *p, const uint8_t *dSeq, const uint8_t *dQual, const uint64_t *dOff,
                                 uint64_t nPairs, void *stream, int count) {
	if(!p || !dSeq || !dQual || !dOff) return -1;
	if(!p->pairsOn) { p->ctx->err = "pipeline: call bt2g_pipeline_enable_pairs first"; return -1; }
	if(2 * nPairs > p->maxReads) { p->ctx->err = "pipeline: batch larger than max_reads"; return -1; }
	if(nPairs == 0) return 0;
	int rc = bt2g_pipeline_run_dev(p, dSeq, dQual, dOff, 2 * nPairs, stream, count);
	if(rc) return rc;
	cudaStream_t st = stream ? (cudaStream_t)stream : p->ctx->stream;
	if(p->ctx->info.off_size == 4) return runPairTail<uint32_t>(p, dSeq, dQual, dOff, nPairs, st, count != 0);
	return runPairTail<uint64_t>(p, dSeq, dQual, dOff, nPairs, st, count != 0);
}

int bt2g_pipeline_run_paired_host(bt2g_pipeline *p, const bt2g_reads *reads, bt2g_read_result *res, uint8_t *ops, bt2g_pair_result *pairs) {
	if(!p || !reads || !reads->qual || !res || !pairs) return -1;
	bt2g_ctx *ctx = p->ctx;
	if(!p->pairsOn) { ctx->err = "pipeline: call bt2g_pipeline_enable_pairs first"; return -1; }
	const uint64_t n = reads->n_reads;
	if(n & 1ull) { ctx->err = "pipeline: paired input needs an even number of reads (mate 1, mate 2 interleaved)"; return -1; }
	if(n > p->maxReads || reads->off[n] > p->maxBases) { ctx->err = "pipeline: batch larger than the pipeline was created for"; return -1; }
	if(n == 0) return 0;
	BT2G_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
	cudaStream_t st = ctx->stream;
	const uint64_t maxOps = (uint64_t)p->prm.max_ops;
	uint64_t chunkMin = 1u << 18;
	if(const char *e = getenv("BT2G_HOST_CHUNK_MIN")) chunkMin = strtoull(e, nullptr, 10);
	const int nChunks = (p->chunkOk && n >= chunkMin && n >= 8) ? 4 : 1;
	// same overlap scheme as bt2g_pipeline_run_host; chunks hold whole pairs
	BT2G_CUDA_TRY(ctx, cudaStreamSynchronize(st));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(p->b.roff, reads->off, (n + 1) * 8, cudaMemcpyHostToDevice, p->sIn));
	const uint64_t per = (((n / 2) + nChunks - 1) / nChunks) * 2;
	for(int c = 0; c < nChunks; c++) {
		const uint64_t s0 = (uint64_t)c * per < n ? (uint64_t)c * per : n, s1 = (s0 + per < n) ? s0 + per : n;
		const uint64_t b0 = reads->off[s0], b1 = reads->off[s1];
		if(b1 > b0) {
			BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(p->b.seq + b0, reads->seq + b0, b1 - b0, cudaMemcpyHostToDevice, p->sIn));
			BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(p->b.qual + b0, reads->qual + b0, b1 - b0, cudaMemcpyHostToDevice, p->sIn));
		}
		BT2G_CUDA_TRY(ctx, cudaEventRecord(p->evIn[c], p->sIn));
	}
	for(int c = 0; c < nChunks; c++) {
		const uint64_t s0 = (uint64_t)c * per < n ? (uint64_t)c * per : n, s1 = (s0 + per < n) ? s0 + per : n;
		BT2G_CUDA_TRY(ctx, cudaStreamWaitEvent(st, p->evIn[c], 0));
		if(s1 == s0) continue;
		int rc;
		if(ctx->info.off_size == 4) {
			rc = runStages<uint32_t>(p, p->b.seq, p->b.qual, p->b.roff + s0, s1 - s0, st, false, s0);
			if(!rc) rc = runPairTail<uint32_t>(p, p->b.seq, p->b.qual, p->b.roff + s0, (s1 - s0) / 2, st, false, s0);
		} else {
			rc = runStages<uint64_t>(p, p->b.seq, p->b.qual, p->b.roff + s0, s1 - s0, st, false, s0);
			if(!rc) rc = runPairTail<uint64_t>(p, p->b.seq, p->b.qual, p->b.roff + s0, (s1 - s0) / 2, st, false, s0);
		}
		if(rc) return rc;
		BT2G_CUDA_TRY(ctx, cudaEventRecord(p->evDone[c], st));
		BT2G_CUDA_TRY(ctx, cudaStreamWaitEvent(p->sOut, p->evDone[c], 0));
		BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(res + s0, p->b.res + s0, (s1 - s0) * sizeof(bt2g_read_result), cudaMemcpyDeviceToHost, p->sOut));
		if(ops) BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(ops + s0 * maxOps, p->b.resOps + s0 * maxOps, (s1 - s0) * maxOps, cudaMemcpyDeviceToHost, p->sOut));
		BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(pairs + s0 / 2, p->b.pairs + s0 / 2, ((s1 - s0) / 2) * sizeof(bt2g_pair_result), cudaMemcpyDeviceToHost, p->sOut));
	}
	BT2G_CUDA_TRY(ctx, cudaStreamSynchronize(p->sOut));
	BT2G_CUDA_TRY(ctx, cudaStreamSynchronize(st));
	p->lastN = n;
	return 0;
}

int bt2g_pipeline_pairs_dev(bt2g_pipeline *p, bt2g_pair_result **pairs) {
	if(!p || !pairs || !p->pairsOn) return -1;
	*pairs = p->b.pairs;
	return 0;
}

int bt2g_pipeline_pair_counters(bt2g_pipeline *p, uint64_t *out2) {
	if(!p || !out2 || !p->pairsOn) return -1;
	bt2g_ctx *ctx = p->ctx;
	BT2G_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
	BT2G_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
	uint32_t np = 0; unsigned long long cells = 0;
	BT2G_CUDA_TRY(ctx, cudaMemcpy(&np, p->b.nMateProb, sizeof(np), cudaMemcpyDeviceToHost));
	BT2G_CUDA_TRY(ctx, cudaMemcpy(&cells, p->b.mateCells, sizeof(cells), cudaMemcpyDeviceToHost));
	out2[0] = np; out2[1] = cells;
	return 0;
}

int bt2g_pipeline_pair_stage_ms(bt2g_pipeline *p, float *out3) {
	if(!p || !out3 || !p->pairsOn) return -1;
	bt2g_ctx *ctx = p->ctx;
	BT2G_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
	BT2G_CUDA_TRY(ctx, cudaEventSynchronize(p->pev[3]));
	for(int i = 0; i < 3; i++) BT2G_CUDA_TRY(ctx, cudaEventElapsedTime(&out3[i], p->pev[i], p->pev[i + 1]));
	return 0;
}

// kernels launched by one bt2g_pipeline_run_dev (after bt2g_pipeline_enable_pairs: run_paired_dev) call (k_plan, k_pack_reads, k_exact_sweep2, k_seed_search3,
// k_collect, k_resolve2, k_frame, the DP kernel(s), k_pick); the split DP mode launches a fill and a tail
// kernel per workspace chunk
int bt2g_pipeline_kernel_launches(bt2g_pipeline *p) {
	if(!p) return -1;
	int dp = 1;
	if(p->packed == 3 && p->dpChunk) dp = 2 * (int)((p->maxProbs + p->dpChunk - 1) / p->dpChunk);
	int pe = 0;
	if(p->pairsOn) {
		// k_frame_mates, the mate DP kernel(s), k_pick_pairs
		int mdp = 1;
		if(p->packed == 3 && p->mateChunk) mdp = 2 * (int)((p->maxReads + p->mateChunk - 1) / p->mateChunk);
		pe = 2 + mdp;
	}
	return 8 + dp + pe;
}

int bt2g_pipeline_results_dev(bt2g_pipeline *p, bt2g_read_result **res, uint8_t **ops) {
	if(!p) return -1;
	if(res) *res = p->b.res;
	if(ops) *ops = p->b.resOps;
	return 0;
}

// device time of each stage of the LAST run, measured with CUDA events on the launching stream:
// [0] plan, [1] exact sweep, [2] seed search, [3] collect, [4] resolve, [5] frame, [6] DP, [7] pick
int bt2g_pipeline_stage_ms(bt2g_pipeline *p, float *out8) {
	if(!p || !out8 || !p->evOk) return -1;
	bt2g_ctx *ctx = p->ctx;
	BT2G_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
	BT2G_CUDA_TRY(ctx, cudaEventSynchronize(p->ev[8]));
	for(int i = 0; i < 8; i++) BT2G_CUDA_TRY(ctx, cudaEventElapsedTime(&out8[i], p->ev[i], p->ev[i + 1]));
	return 0;
}

// counters of the last run made with count=1: [0] exact-sweep side fetches, [1] seed-search side
// fetches, [2] resolve side fetches, [3] DP cells, [4] DP problems, [5] reads
int bt2g_pipeline_counters(bt2g_pipeline *p, uint64_t *out6) {
	if(!p || !out6) return -1;
	bt2g_ctx *ctx = p->ctx;
	BT2G_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
	BT2G_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
	unsigned long long c[4]; uint32_t np = 0;
	BT2G_CUDA_TRY(ctx, cudaMemcpy(c, p->b.counters, sizeof(c), cudaMemcpyDeviceToHost));
	BT2G_CUDA_TRY(ctx, cudaMemcpy(&np, p->b.nProb, sizeof(np), cudaMemcpyDeviceToHost));
	for(int i = 0; i < 4; i++) out6[i] = c[i];
	out6[4] = np; out6[5] = p->lastN;
	return 0;
}

} // extern "C"
