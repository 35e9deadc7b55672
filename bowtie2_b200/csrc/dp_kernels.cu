// dp_kernels.cu -- K3: seed-extension dynamic programming (fill + candidate gather + backtrace)
// for sm_100a.
//
// The reference fills the whole rdlen x (refr-refl+1) rectangle with a striped (Farrar) SSE
// kernel that stores E, F and H for every cell and then repairs the vertical-gap dependency
// in a "lazy F" fix-up loop (aligner_swsse_ee_u8.cpp:775-1146; the fix-up loop dominates its
// run time, SURVEY.md section 3.5).  This kernel is a different design:
//   * persistent warps, one DP problem at a time per warp; lane k owns R consecutive read rows;
//     at step t lane k computes column t-k, so the 32 lanes sweep an anti-diagonal wavefront and
//     the vertical (F) and diagonal dependencies cross lanes through one __shfl_up per step --
//     no fix-up loop;
//   * exact 32-bit arithmetic with DPX max/add-max (no saturating 8/16-bit lanes, so the
//     reference's u8 -> i16 fallback (aligner_sw.cpp:518,569-605) has no equivalent here;
//     the two paths produce identical scores by the reference's own debug asserts :622-677);
//   * instead of spilling E/F/H (6 bytes/cell) the fill emits ONE byte per cell: the move the
//     reference's backtrace would take from the H, E and F states of that cell under its fixed
//     preference order diag > ref-gap open > ref-gap extend > read-gap open > read-gap extend
//     (aligner_swsse_ee_u8.cpp:1509-1520, E: :1376-1380, F: :1434-1438).  Bytes are laid out
//     wavefront-major ([step][lane][R]) so every step's store is one coalesced line per warp,
//     in a per-warp-slot workspace that is reused problem after problem and stays in L2;
//   * the backtrace replays SwAligner::nextAlignment (aligner_sw.cpp:737-1146) for ALL
//     candidates in their sorted order, marking visited cells in bit 7 of the move byte.  In
//     the reference a backtrace that reaches an already reported-through cell unwinds its whole
//     branch stack (every stacked cell is itself already marked, :1336-1340,:1561-1585) and
//     fails, so the remaining-option masks never matter and the walk is a pure function of the
//     move bytes + visited bits.  The walk is warp-cooperative: the 32 lanes prefetch the next
//     32 cells of the current diagonal in one load, every lane then steps through them in
//     lock-step (uniform control flow), so the latency chain is one L2 round trip per diagonal
//     run instead of one per cell.
#include "fm_device.cuh"
#include "dp_device.cuh"
#include "launch.cuh"

#define DP_NEG (-(1 << 28))
#define DP_BIG (1 << 20)

// per-warp shared memory: maxCol ints (last-row scores), maxCol u16 (candidate columns), the reference window
__host__ __device__ __forceinline__ size_t dp_smem_per_warp(int maxCol) { return ((size_t)maxCol * 7 + 16 + 15) & ~(size_t)15; }

__device__ __forceinline__ int dp_max(int a, int b) { return a > b ? a : b; }

// ---- SwAligner::nextAlignment over every candidate (aligner_sw.cpp:737-1146), shared by the
// end-to-end and local kernels.  Warp-cooperative (see the header comment).
template <int R>
__device__ __forceinline__ void dp_backtrace_all(const DpLaunch &L, const bt2g_scoring &sc, const bt2g_dp_problem &p, uint64_t w,
                                                 const uint8_t *rs, const uint8_t *rq, int rdlen, const uint8_t *refw,
                                                 uint8_t *codes, bt2g_dp_cand *cands, int ncand, bt2g_dp_summary *summ,
                                                 int lane, bool local) {
	const int rdgapo = sc.rdgap_const + sc.rdgap_linear, rdgape = sc.rdgap_linear;
	const int rfgapo = sc.rfgap_const + sc.rfgap_linear, rfgape = sc.rfgap_linear;
	int SQ = rdlen >> 4; if(SQ == 0) SQ = 1;                 // aligner_sw.cpp:754-755
	bt2g_dp_aln *alns = L.alns + w * (uint64_t)L.maxAlns;
	uint8_t *ops = L.ops + w * (uint64_t)L.maxAlns * L.maxOps;
	int naln = 0, flags = 0;
	auto cell = [&](int rr, int cc) -> uint8_t * { int k = rr / R; return codes + ((size_t)(cc + k) * 32 + k) * R + (rr - k * R); };
	for(int ci = 0; ci < ncand; ci++) {
		int row = cands[ci].row, col = cands[ci].col;      // same address in every lane: one broadcast load
		const int startRow = row;
		if(local) {
			// start cell already reported through (aligner_sw.cpp:771-789) is checked before domination
			const bool vis = (*cell(row, col) & 0x80) != 0;
			if(vis) { if(lane == 0) cands[ci].fate = BT2G_CAND_FILT_START; continue; }
			// domination by an already attempted candidate (:946-971): within SQ rows and columns
			bool dom = false;
			for(int k = lane; k < ci; k += 32) {
				const int f = cands[k].fate;
				if(f == BT2G_CAND_FAILED || f == BT2G_CAND_SUCCEEDED) {
					int dr = cands[k].row - row, dc = cands[k].col - col;
					dr = dr < 0 ? -dr : dr; dc = dc < 0 ? -dc : dc;
					if(dr <= SQ && dc <= SQ) dom = true;
				}
			}
			if(__any_sync(0xffffffffu, dom)) { if(lane == 0) cands[ci].fate = BT2G_CAND_FILT_DOMINATED; __syncwarp(); continue; }
		}
		// backtraceNucleotidesEnd2EndSseU8 (aligner_swsse_ee_u8.cpp:1283-1877).  Lane k holds cell k of the
		// current diagonal (row-k, col-k).  In the H state the walk follows the diagonal as long as the
		// cells say "diagonal move" and are not yet reported through, so the length of that run is one
		// ballot, and the run's cells are processed by their own lanes in parallel (edit op, N count,
		// reported-through mark); only the cell that ends a run (gap move, row 0, visited cell, soft trim)
		// is handled by uniform scalar code.  The alignment score is the candidate cell's score: the
		// walk follows exact equalities of the recurrences (the reference asserts the same, :1842-1846).
		uint8_t *o = ops + (size_t)naln * L.maxOps;
		const bool room = naln < L.maxAlns;
		int nops = 0, ns = 0, gaps = 0, ct = 0;              // ct: 0 H, 1 E, 2 F
		bool fail = false, core = false, done = false, first = true, filtStart = false;
		const int origCol = col;
		int trimBeg = 0;
		auto rdchar = [&](int rr) -> int { const int pos = p.fw ? rr : rdlen - 1 - rr; int c = rs[pos]; return p.fw ? c : (c > 3 ? 4 : 3 - c); };
		while(!done && !fail) {
			const int rk = row - lane, ck = col - lane;
			uint8_t *cp = (rk >= 0 && ck >= 0) ? cell(rk, ck) : nullptr;
			const uint8_t mine = cp ? *cp : 0xff;
			int stop = 0;                                     // lane holding the cell that ends this round
			if(ct == 0) {
				const bool cont = !(mine & 0x80) && ((mine & 7) == 1) && rk > 0;
				const uint32_t m = __ballot_sync(0xffffffffu, cont);
				const int run = (m == 0xffffffffu) ? 32 : __ffs(~m) - 1;
				if(run > 0) {
					first = false;
					const int diagi = col - row + p.triml;
					if(diagi >= p.corel && diagi <= p.corer) core = true;
					bool isN = false;
					if(lane < run) {
						const int c = rdchar(rk), refc = refw[ck];
						isN = c > 3 || refc > 3;
						const uint8_t op = (uint8_t)(((!isN && c == refc) ? BT2G_OP_MATCH : BT2G_OP_MM) | (refc << 2));
						if(room && nops + lane < L.maxOps) o[nops + lane] = op;
						*cp = mine | 0x80;                        // setReportedThrough (:1555)
					}
					ns += __popc(__ballot_sync(0xffffffffu, isN));
					nops += run; row -= run; col -= run;
				}
				if(run == 32) { __syncwarp(); continue; }
				stop = run;
			}
			// the cell at (row, col), held by lane `stop`
			const uint8_t code = (uint8_t)__shfl_sync(0xffffffffu, (int)mine, stop);
			if(code & 0x80) {
				// start cell already reported through -> BT_CAND_FATE_FILT_START (:771-789);
				// anywhere else the backtrace fails
				if(first) filtStart = true;
				fail = true; break;
			}
			first = false;
			if(lane == stop) *cp = mine | 0x80;
			{
				const int diagi = col - row + p.triml;
				if(diagi >= p.corel && diagi <= p.corer) core = true;
			}
			if(row == 0) { done = true; break; }
			int mv;   // 2 refopen, 3 rfext, 4 rdopen, 5 rdext (a diagonal move never ends a run above row 0)
			if(ct == 0) { mv = code & 7; if(mv == 0) { trimBeg = row; done = true; break; } }
			else if(ct == 1) { int e = (code >> 3) & 3; if(e == 0) { fail = true; break; } mv = e == 1 ? 4 : 5; }
			else { int f = (code >> 5) & 3; if(f == 0) { fail = true; break; } mv = f == 1 ? 2 : 3; }
			uint8_t op;
			gaps++;
			if(mv == 2 || mv == 3) {
				op = BT2G_OP_REFGAP;
				row--; ct = (mv == 2) ? 0 : 2;
			} else {
				op = (uint8_t)(BT2G_OP_READGAP | (refw[col] << 2));
				col--; ct = (mv == 4) ? 0 : 1;
			}
			if(room && lane == 0 && nops < L.maxOps) o[nops] = op;
			nops++;
			__syncwarp();
		}
		if(filtStart) { if(lane == 0) cands[ci].fate = BT2G_CAND_FILT_START; continue; }
		if(!fail) {
			// the alignment's first cell (row, col) (:1797-1813)
			const int c = rdchar(row), refc = refw[col];
			const bool isN = c > 3 || refc > 3;
			ns += isN;
			const uint8_t op = (uint8_t)(((!isN && c == refc) ? BT2G_OP_MATCH : BT2G_OP_MM) | (refc << 2));
			if(!core) fail = true;                   // core-diagonal rejection (:1764-1795)
			else if(ns > p.nceil) fail = true;       // N ceiling (:1813-1818)
			else {
				if(room && lane == 0 && nops < L.maxOps) o[nops] = op;
				nops++;
			}
		}
		const bool opOverflow = nops > L.maxOps;
		if(fail) { if(lane == 0) cands[ci].fate = BT2G_CAND_FAILED; continue; }
		if(lane == 0) cands[ci].fate = BT2G_CAND_SUCCEEDED;
		if(room) {
			int refns = 0;
			for(int k = col + lane; k <= origCol; k += 32) refns += refw[k] > 3;
			refns = __reduce_add_sync(0xffffffffu, refns);
			if(lane == 0) {
				bt2g_dp_aln &a = alns[naln];
				a.cand_idx = ci; a.score = cands[ci].score; a.ns = ns; a.gaps = gaps; a.col0 = col; a.row0 = row;
				a.trim_beg = trimBeg; a.trim_end = rdlen - 1 - startRow; a.nops = nops;
				a.refns = refns;
			}
			if(opOverflow) flags |= BT2G_DP_FLAG_OPS_OVERFLOW;
		} else {
			flags |= BT2G_DP_FLAG_ALN_OVERFLOW;
		}
		naln++;
	}
	if(lane == 0) { summ->naln = naln; summ->flags |= flags; }
}

template <int R>
__device__ __forceinline__ void dp_backtrace_h(const DpLaunch &L, const bt2g_scoring &sc, const bt2g_dp_problem &p, uint64_t w,
                                               const uint8_t *rs, const uint8_t *rq, int rdlen, const uint8_t *refw,
                                               uint8_t *hb, bt2g_dp_cand *cands, int ncand, bt2g_dp_summary *summ, int lane,
                                               const uint8_t *prof);

// ---- end-to-end tail: best of the last row, candidate list (gatherCellsNucleotidesEnd2End), backtraces.
// HB: the workspace holds H bytes (k_dp_fill_h) instead of move codes.
template <int R, bool HB = false>
__device__ __forceinline__ void dp_e2e_tail(const DpLaunch &L, const bt2g_scoring &sc, const bt2g_dp_problem &p, uint64_t w,
                                            const uint8_t *rs, const uint8_t *rq, int rdlen, int ncol, int32_t *lastH,
                                            uint16_t *candCol, const uint8_t *refw, uint8_t *codes, bt2g_dp_summary *summ, int lane,
                                            const uint8_t *prof = nullptr) {
	__syncwarp();
	// best = max of the last row (aligner_swsse_ee_u8.cpp:1095-1100)
	int best = DP_NEG;
	for(int k = lane; k < ncol; k += 32) best = dp_max(best, lastH[k]);
#pragma unroll
	for(int o = 16; o > 0; o >>= 1) best = dp_max(best, __shfl_xor_sync(0xffffffffu, best, o));

	// ---- SwAligner::align tail (aligner_sw.cpp:679-729) + gatherCellsNucleotidesEnd2End (:1176-1208)
	if(lane == 0) { summ->best = best; summ->flags = 0; summ->naln = 0; summ->ncand = 0; summ->found = 0; }
	if(best < p.minsc) return;
	bt2g_dp_cand *cands = L.cands + w * (uint64_t)L.maxCands;
	// compact the last-row cells with score >= minsc (in place: slot k <= column j), then rank them
	// under DpBtCandidate::operator< (score desc, row equal, col desc; aligner_sw_nuc.h:149-157)
	int totalCand = 0;
	for(int j0 = 0; j0 < ncol; j0 += 32) {
		const int j = j0 + lane;
		const int s = j < ncol ? lastH[j] : DP_NEG;
		const bool isC = j < ncol && s >= p.minsc;
		const uint32_t m = __ballot_sync(0xffffffffu, isC);
		if(isC) {
			const int k = totalCand + __popc(m & ((1u << lane) - 1u));
			lastH[k] = s; candCol[k] = (uint16_t)j;
		}
		totalCand += __popc(m);
		__syncwarp();
	}
	for(int a0 = 0; a0 < totalCand; a0 += 32) {
		const int a = a0 + lane;
		if(a < totalCand) {
			const int s = lastH[a];
			int rank = 0;
			for(int k = 0; k < totalCand; k++) {
				const int sk = lastH[k];
				rank += (sk > s) || (sk == s && k > a);
			}
			if(rank < L.maxCands) { cands[rank].score = s; cands[rank].col = candCol[a]; cands[rank].row = rdlen - 1; cands[rank].fate = 0; }
		}
	}
	const int ncand = totalCand < L.maxCands ? totalCand : L.maxCands;
	if(lane == 0) {
		summ->ncand = totalCand; summ->found = totalCand > 0;
		if(totalCand > L.maxCands) summ->flags |= BT2G_DP_FLAG_CAND_OVERFLOW;
	}
	__syncwarp();

	if(HB) dp_backtrace_h<R>(L, sc, p, w, rs, rq, rdlen, refw, codes, cands, ncand, summ, lane, prof);
	else dp_backtrace_all<R>(L, sc, p, w, rs, rq, rdlen, refw, codes, cands, ncand, summ, lane, false);
}

// R = rows per lane (rdlen <= 32*R)
template <typename OFF, int R>
__global__ void __launch_bounds__(128) k_dp_e2e(DevIndex<OFF> ix, bt2g_scoring sc, DpLaunch L) {
	extern __shared__ uint8_t smem[];
	const int warpInBlock = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const uint64_t slot = blockIdx.x * (uint64_t)(blockDim.x >> 5) + warpInBlock;
	const uint64_t nSlots = (uint64_t)gridDim.x * (blockDim.x >> 5);
	const uint64_t nProb = L.nDev ? (uint64_t)*L.nDev : L.n;
	// per-warp shared memory: last-row scores (ints) then the reference window (bytes)
	const size_t perWarp = dp_smem_per_warp(L.maxCol);
	int32_t *lastH = reinterpret_cast<int32_t *>(smem + (size_t)warpInBlock * perWarp);
	uint16_t *candCol = reinterpret_cast<uint16_t *>(lastH + L.maxCol);
	uint8_t *refw = reinterpret_cast<uint8_t *>(candCol + L.maxCol);
	// persistent warps: the move-byte workspace belongs to the warp SLOT, not to the problem, so
	// it is (#SMs x resident warps) x codeStride bytes and stays L2-resident across problems
	uint8_t *codes = L.codes + slot * L.codeStride;
	const int rdgapo = sc.rdgap_const + sc.rdgap_linear, rdgape = sc.rdgap_linear;
	const int rfgapo = sc.rfgap_const + sc.rfgap_linear, rfgape = sc.rfgap_linear;

	for(uint64_t w = slot; w < nProb; w += nSlots) {
		const bt2g_dp_problem p = L.probs[w];
		const uint8_t *rs = L.seq + L.roff[p.read_idx];
		const uint8_t *rq = L.qual + L.roff[p.read_idx];
		const int rdlen = (int)(L.roff[p.read_idx + 1] - L.roff[p.read_idx]);
		const int ncol = (int)(p.refr - p.refl + 1);
		bt2g_dp_summary *summ = L.summ + w;
		__syncwarp();
		if(ncol <= 0 || ncol > L.maxCol || rdlen > 32 * R || rdlen <= 0) {
			if(lane == 0) { summ->found = 0; summ->best = DP_NEG; summ->ncand = 0; summ->naln = 0; summ->flags = BT2G_DP_FLAG_BADSHAPE; }
			continue;
		}
		// reference window (SwAligner::initRef, aligner_sw.cpp:155-271): codes 0..3, 4 = N / off-end
		for(int k = lane; k < ncol; k += 32) refw[k] = (uint8_t)ref_base<OFF>(ix, p.tidx, p.refl + k);
		__syncwarp();

		// per-row constants (buildQueryProfileEnd2EndSseU8, aligner_swsse_ee_u8.cpp:75-142).  Penalties are
		// kept negated; the gap barrier (:944-945,:966-969,:983-985) is folded into per-row gap-open/extend
		// costs: in a barrier row they are DP_BIG, which puts E and F far below any minimum score.
		int rc[R], mmpN[R], npnN[R], rfo[R], rfe[R], rdo[R];
#pragma unroll
		for(int r = 0; r < R; r++) {
			int i = lane * R + r;
			bool bar = true;
			if(i < rdlen) {
				int pos = p.fw ? i : rdlen - 1 - i;
				int c = rs[pos];
				rc[r] = p.fw ? c : (c > 3 ? 4 : 3 - c);
				int q = (int)rq[pos] - 33;
				q = q < 0 ? 0 : (q > 63 ? 63 : q);
				npnN[r] = -sc.npen[q];
				// a read N never "equals" a reference base and is charged the N penalty (Scoring::score, scoring.h:241-251)
				mmpN[r] = rc[r] > 3 ? npnN[r] : -sc.mmpen[q];
				if(rc[r] > 3) rc[r] = 5;
				bar = (i < sc.gapbar) || (rdlen - 1 - i < sc.gapbar);
			} else { rc[r] = 5; mmpN[r] = 0; npnN[r] = 0; }
			rfo[r] = bar ? DP_BIG : rfgapo; rfe[r] = bar ? DP_BIG : rfgape; rdo[r] = bar ? DP_BIG : rdgapo;
		}
		const int lastLane = (rdlen - 1) / R, lastR = (rdlen - 1) % R;
		const int bonus = sc.match_bonus;

		// Branch-free move codes.  With E = max(E'-rdgape, H'-rdgapo) and F = max(F^-rfgape, H^-rfgapo),
		// "which term is the max (open wins ties)" IS the E/F move, and the H move is
		//   diag if H == Hd, else the F move if H == F, else the E move
		// -- the same choice the reference makes from its five equality tests in preference order
		// (aligner_swsse_ee_u8.cpp:1468-1520): H==F with F==open implies H==H^-rfgapo (bit 0), H==F with
		// F==extend only implies bit 2, and likewise for E (bits 1, 3).  Cells below the minimum score
		// (all of E and F in barrier rows included) may get arbitrary codes; no backtrace visits them
		// (scores are monotone along a path).  Byte = hsel | (esel << 3) | (fsel << 5) with esel, fsel in
		// {1 open, 2 extend}; the state kept per row is ev = 3 + esel so that ev is also the H code of an
		// E move, and fv = 1 + fsel is the H code of an F move; the constant (3 << 3) + (1 << 5) comes off
		// once per packed word.
		int Hleft[R], Earr[R], ev[R];
#pragma unroll
		for(int r = 0; r < R; r++) { Hleft[r] = DP_NEG; Earr[r] = DP_NEG; ev[r] = 4; }
		int botH = DP_NEG, botF = DP_NEG, prevInH = DP_NEG;
		const int nsteps = ncol + lastLane;   // lanes beyond lastLane hold no rows
		uint8_t *dst = codes + (size_t)lane * R;
		for(int t = 0; t < nsteps; t++, dst += 32 * R) {
			int inH = __shfl_up_sync(0xffffffffu, botH, 1);
			int inF = __shfl_up_sync(0xffffffffu, botF, 1);
			if(lane == 0) { inH = DP_NEG; inF = DP_NEG; }
			const int j = t - lane;
			if(j >= 0 && j < ncol && lane <= lastLane) {
				const int refc = refw[j];
				const bool refN = refc > 3;
				// H[i0-1][j-1]: row -1 is the free start row of end-to-end mode (vhilsw, :853,923-927)
				int diag = (lane == 0) ? 0 : prevInH;
				int upH = inH, upF = inF;
				uint32_t packed[(R + 3) / 4];
#pragma unroll
				for(int q4 = 0; q4 < (R + 3) / 4; q4++) packed[q4] = 0u - 0x38383838u;
#pragma unroll
				for(int r = 0; r < R; r++) {
					// F[i][j] = max(F[i-1][j]-rfgape, H[i-1][j]-rfgapo)
					const int fo = upH - rfo[r], fe = upF - rfe[r];
					const bool fopen = fo >= fe;
					const int F = fopen ? fo : fe;
					const int fv = fopen ? 2 : 3;
					const int pen = refN ? npnN[r] : mmpN[r];
					const int Hd = diag + ((rc[r] == refc) ? bonus : pen);
					const int E = Earr[r];
					const int H = __vimax3_s32(Hd, E, F);
					const int x = (H != F) ? ev[r] : fv;
					const int hsel = (H != Hd) ? x : 1;
					packed[r >> 2] += (uint32_t)(hsel + ev[r] * 8 + fv * 32) << ((r & 3) * 8);
					// E[i][j+1] = max(E[i][j]-rdgape, H[i][j]-rdgapo)
					const int eo = H - rdo[r], ee = E - rdgape;
					const bool eopen = eo >= ee;
					Earr[r] = eopen ? eo : ee;
					ev[r] = eopen ? 4 : 5;
					diag = Hleft[r]; Hleft[r] = H;
					upH = H; upF = F;
				}
				if(lane == lastLane) {
					int hl = Hleft[0];
#pragma unroll
					for(int r = 1; r < R; r++) hl = (lastR == r) ? Hleft[r] : hl;
					lastH[j] = hl;
				}
				botH = upH; botF = upF;
				prevInH = inH;
				if(R == 4) *reinterpret_cast<uint32_t *>(dst) = packed[0];
				else if(R == 8) *reinterpret_cast<uint2 *>(dst) = make_uint2(packed[0], packed[1]);
				else {
#pragma unroll
					for(int q4 = 0; q4 < (R + 3) / 4; q4++) reinterpret_cast<uint32_t *>(dst)[q4] = packed[q4];
				}
			} else if(j >= ncol) {
				botH = DP_NEG; botF = DP_NEG;
			}
		}
		dp_e2e_tail<R>(L, sc, p, w, rs, rq, rdlen, ncol, lastH, candCol, refw, codes, summ, lane);
	} // persistent loop over problems
}

// ----------------------------------------------------------------------------------------
// Two problems per warp, packed as signed 16-bit pairs (DPX s16x2): the low half of every value
// belongs to problem A, the high half to problem B; lane k holds rows kR..kR+R-1 of both.
// Same recurrences and the same move bytes as k_dp_e2e, with
//   * add+max fused (VIADDMNMX.S16x2), every sum clamped at DPX_FLOOR so nothing wraps
//     (|gap cost| <= DPX_BIG, so a + b >= DPX_FLOOR - DPX_BIG > -32768);
//   * "which operand won" taken from XOR + unsigned min instead of predicates: (F != fo) is 1 exactly
//     when the extension beat the open (open wins ties), (H != Hd) / (H != F) select the H move;
//     0/1 halves times 0xffff give half-word masks for LOP3 selects;
//   * small non-negative code arithmetic done with plain 32-bit adds (no half can borrow).
// The host only selects this kernel when every score fits (|minsc|, perfect score <= DPX_LIMIT).
#define DPX_FLOOR (-16384)
#define DPX_BIG   16000
#define DPX_LIMIT 8000

__device__ __forceinline__ uint32_t dpx_pack(int lo, int hi) { return ((uint32_t)lo & 0xffffu) | ((uint32_t)hi << 16); }
__device__ __forceinline__ uint32_t dpx_both(int v) { return dpx_pack(v, v); }
__device__ __forceinline__ uint32_t dpx_ne01(uint32_t a, uint32_t b) { return __vminu2(a ^ b, 0x00010001u); }   // per half: a != b
__device__ __forceinline__ uint32_t dpx_sel(uint32_t mask, uint32_t a, uint32_t b) { return (a & mask) | (b & ~mask); }

template <typename OFF, int R>
__global__ void __launch_bounds__(128) k_dp_e2e_x2(DevIndex<OFF> ix, bt2g_scoring sc, DpLaunch L) {
	extern __shared__ uint8_t smem[];
	const int warpInBlock = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const uint64_t slot = blockIdx.x * (uint64_t)(blockDim.x >> 5) + warpInBlock;
	const uint64_t nSlots = (uint64_t)gridDim.x * (blockDim.x >> 5);
	const uint64_t nProb = L.nDev ? (uint64_t)*L.nDev : L.n;
	const uint64_t nPairs = (nProb + 1) >> 1;
	const size_t perProb = dp_smem_per_warp(L.maxCol);
	uint8_t *sm0 = smem + (size_t)warpInBlock * 2 * perProb;
	int32_t *lastH[2]; uint16_t *candCol[2]; uint8_t *refw[2]; uint8_t *codes[2];
#pragma unroll
	for(int x = 0; x < 2; x++) {
		lastH[x] = reinterpret_cast<int32_t *>(sm0 + x * perProb);
		candCol[x] = reinterpret_cast<uint16_t *>(lastH[x] + L.maxCol);
		refw[x] = reinterpret_cast<uint8_t *>(candCol[x] + L.maxCol);
		codes[x] = L.codes + (slot * 2 + x) * L.codeStride;
	}
	const int rdgapo = sc.rdgap_const + sc.rdgap_linear, rdgape = sc.rdgap_linear;
	const int rfgapo = sc.rfgap_const + sc.rfgap_linear, rfgape = sc.rfgap_linear;
	const uint32_t FLOORP = dpx_both(DPX_FLOOR), ONEP = 0x00010001u;
	const uint32_t bonusP = dpx_both(sc.match_bonus), nrdeP = dpx_both(-rdgape);

	for(uint64_t pw = slot; pw < nPairs; pw += nSlots) {
		uint64_t w[2] = {2 * pw, 2 * pw + 1};
		bool live[2] = {true, w[1] < nProb};
		if(!live[1]) w[1] = w[0];
		bt2g_dp_problem p[2] = {L.probs[w[0]], L.probs[w[1]]};
		const uint8_t *rs[2], *rq[2]; int rdlen[2], ncol[2];
		__syncwarp();
#pragma unroll
		for(int x = 0; x < 2; x++) {
			rs[x] = L.seq + L.roff[p[x].read_idx]; rq[x] = L.qual + L.roff[p[x].read_idx];
			rdlen[x] = (int)(L.roff[p[x].read_idx + 1] - L.roff[p[x].read_idx]);
			ncol[x] = (int)(p[x].refr - p[x].refl + 1);
			if(ncol[x] <= 0 || ncol[x] > L.maxCol || rdlen[x] > 32 * R || rdlen[x] <= 0) {
				if(live[x] && lane == 0) {
					bt2g_dp_summary *sm = L.summ + w[x];
					sm->found = 0; sm->best = DP_NEG; sm->ncand = 0; sm->naln = 0; sm->flags = BT2G_DP_FLAG_BADSHAPE;
				}
				live[x] = false;
			}
		}
		if(!live[0] && !live[1]) continue;
		// a dead half mirrors the live one (its results are discarded)
		if(!live[0]) { p[0] = p[1]; rs[0] = rs[1]; rq[0] = rq[1]; rdlen[0] = rdlen[1]; ncol[0] = ncol[1]; w[0] = w[1]; }
		if(!live[1]) { p[1] = p[0]; rs[1] = rs[0]; rq[1] = rq[0]; rdlen[1] = rdlen[0]; ncol[1] = ncol[0]; w[1] = w[0]; }
		// reference windows (SwAligner::initRef, aligner_sw.cpp:155-271): codes 0..3, 4 = N / off-end
#pragma unroll
		for(int x = 0; x < 2; x++)
			for(int k = lane; k < ncol[x]; k += 32) refw[x][k] = (uint8_t)ref_base<OFF>(ix, p[x].tidx, p[x].refl + k);
		const int ncolMax = ncol[0] > ncol[1] ? ncol[0] : ncol[1], ncolMin = ncol[0] < ncol[1] ? ncol[0] : ncol[1];
		// pad the shorter window so that the packed loop may read it (values are never used)
		for(int x = 0; x < 2; x++) for(int k = ncol[x] + lane; k < ncolMax; k += 32) refw[x][k] = 4;
		(void)ncolMin;
		__syncwarp();

		// per-row constants of both problems (buildQueryProfileEnd2EndSseU8, aligner_swsse_ee_u8.cpp:75-142)
		uint32_t rcP[R], mmpP[R], npnP[R], nrfoP[R], nrfeP[R], nrdoP[R];
#pragma unroll
		for(int r = 0; r < R; r++) {
			int v[2][6];
#pragma unroll
			for(int x = 0; x < 2; x++) {
				const int i = lane * R + r;
				bool bar = true;
				int c = 5, mm = 0, np = 0;
				if(i < rdlen[x]) {
					const int pos = p[x].fw ? i : rdlen[x] - 1 - i;
					c = rs[x][pos];
					c = p[x].fw ? c : (c > 3 ? 4 : 3 - c);
					int q = (int)rq[x][pos] - 33;
					q = q < 0 ? 0 : (q > 63 ? 63 : q);
					np = -(int)sc.npen[q];
					mm = c > 3 ? np : -(int)sc.mmpen[q];
					if(c > 3) c = 5;
					bar = (i < sc.gapbar) || (rdlen[x] - 1 - i < sc.gapbar);
				}
				v[x][0] = c; v[x][1] = mm; v[x][2] = np;
				v[x][3] = bar ? -DPX_BIG : -rfgapo; v[x][4] = bar ? -DPX_BIG : -rfgape; v[x][5] = bar ? -DPX_BIG : -rdgapo;
			}
			rcP[r] = dpx_pack(v[0][0], v[1][0]); mmpP[r] = dpx_pack(v[0][1], v[1][1]); npnP[r] = dpx_pack(v[0][2], v[1][2]);
			nrfoP[r] = dpx_pack(v[0][3], v[1][3]); nrfeP[r] = dpx_pack(v[0][4], v[1][4]); nrdoP[r] = dpx_pack(v[0][5], v[1][5]);
		}
		int lastLane[2], lastR[2];
#pragma unroll
		for(int x = 0; x < 2; x++) { lastLane[x] = (rdlen[x] - 1) / R; lastR[x] = (rdlen[x] - 1) % R; }
		const int lastLaneMax = lastLane[0] > lastLane[1] ? lastLane[0] : lastLane[1];

		uint32_t Hleft[R], Earr[R], ev[R];
#pragma unroll
		for(int r = 0; r < R; r++) { Hleft[r] = FLOORP; Earr[r] = FLOORP; ev[r] = 0x00040004u; }
		uint32_t botH = FLOORP, botF = FLOORP, prevInH = FLOORP;
		const int nsteps = ncolMax + lastLaneMax;
		uint8_t *dstA = codes[0] + (size_t)lane * R, *dstB = codes[1] + (size_t)lane * R;
		for(int t = 0; t < nsteps; t++, dstA += 32 * R, dstB += 32 * R) {
			uint32_t inH = __shfl_up_sync(0xffffffffu, botH, 1);
			uint32_t inF = __shfl_up_sync(0xffffffffu, botF, 1);
			if(lane == 0) { inH = FLOORP; inF = FLOORP; }
			const int j = t - lane;
			if(j >= 0 && j < ncolMax && lane <= lastLaneMax) {
				const uint32_t refcP = (uint32_t)refw[0][j] | ((uint32_t)refw[1][j] << 16);
				const uint32_t refNm = ((refcP >> 2) & ONEP) * 0xffffu;      // half mask: reference N
				// H[i0-1][j-1]: row -1 is the free start row of end-to-end mode (vhilsw, :853,923-927)
				uint32_t diag = (lane == 0) ? 0u : prevInH;
				uint32_t upH = inH, upF = inF;
				uint32_t cw[R];
#pragma unroll
				for(int r = 0; r < R; r++) {
					// F[i][j] = max(F[i-1][j]-rfgape, H[i-1][j]-rfgapo)
					const uint32_t fo = __viaddmax_s16x2(upH, nrfoP[r], FLOORP);
					const uint32_t F = __viaddmax_s16x2(upF, nrfeP[r], fo);
					const uint32_t fv = 0x00020002u + dpx_ne01(F, fo);
					const uint32_t pen = dpx_sel(refNm, npnP[r], mmpP[r]);
					const uint32_t mmask = dpx_ne01(rcP[r], refcP) * 0xffffu;
					const uint32_t Hd = __viaddmax_s16x2(diag, dpx_sel(mmask, pen, bonusP), FLOORP);
					const uint32_t E = Earr[r];
					const uint32_t H = __vimax3_s16x2(Hd, E, F);
					const uint32_t m0 = dpx_ne01(H, Hd) * 0xffffu, m1 = dpx_ne01(H, F) * 0xffffu;
					const uint32_t hsel = dpx_sel(m0, dpx_sel(m1, ev[r], fv), ONEP);
					cw[r] = hsel + ev[r] * 8u + fv * 32u;
					// E[i][j+1] = max(E[i][j]-rdgape, H[i][j]-rdgapo)
					const uint32_t eo = __viaddmax_s16x2(H, nrdoP[r], FLOORP);
					const uint32_t En = __viaddmax_s16x2(E, nrdeP, eo);
					ev[r] = 0x00040004u + dpx_ne01(En, eo);
					Earr[r] = En;
					diag = Hleft[r]; Hleft[r] = H;
					upH = H; upF = F;
				}
#pragma unroll
				for(int x = 0; x < 2; x++) {
					if(lane == lastLane[x] && j < ncol[x]) {
						uint32_t hl = Hleft[0];
#pragma unroll
						for(int r = 1; r < R; r++) hl = (lastR[x] == r) ? Hleft[r] : hl;
						lastH[x][j] = x == 0 ? (int)(int16_t)(hl & 0xffffu) : (int)(int16_t)(hl >> 16);
					}
				}
				botH = upH; botF = upF;
				prevInH = inH;
				// move bytes: byte 0 of every code word is problem A's, byte 2 problem B's
#pragma unroll
				for(int q4 = 0; q4 < R / 4; q4++) {
					const uint32_t t01 = __byte_perm(cw[4 * q4], cw[4 * q4 + 1], 0x6240), t23 = __byte_perm(cw[4 * q4 + 2], cw[4 * q4 + 3], 0x6240);
					reinterpret_cast<uint32_t *>(dstA)[q4] = __byte_perm(t01, t23, 0x5410) - 0x38383838u;
					reinterpret_cast<uint32_t *>(dstB)[q4] = __byte_perm(t01, t23, 0x7632) - 0x38383838u;
				}
			} else if(j >= ncolMax) {
				botH = FLOORP; botF = FLOORP;
			}
		}
#pragma unroll
		for(int x = 0; x < 2; x++) {
			if(!live[x]) continue;
			dp_e2e_tail<R>(L, sc, p[x], w[x], rs[x], rq[x], rdlen[x], ncol[x], lastH[x], candCol[x], refw[x], codes[x], L.summ + w[x], lane);
		}
	} // persistent loop over problem pairs
}

// ----------------------------------------------------------------------------------------
// H-byte kernels (two problems per warp, s16x2; see the description below).
// H-byte kernels take any R (rows per lane) and store RP = R rounded up to 4 bytes per lane and step
#define DP_RP(R) ((((R) + 3) / 4) * 4)
#define DP_QPROF_BYTES(R) ((size_t)(5 * (R) * 32 * 4))                      // fill kernel: query profile of one problem (32-bit entries)
#define DP_PROF_BYTES(R) ((size_t)(3 * 32 * (R) + 15) & ~(size_t)15)      // per-row profile of the tail kernel: 3 bytes x 32 R rows
// Workspace layout of one problem with S = maxCol + 32 step slots: R / 4 word planes [S][32] x 4 B holding rows
// 4g..4g+3 of each lane, then one byte plane [S][32] per remaining row, so that every store of a warp is one
// contiguous, fully written run of sectors and nothing but real cells reaches HBM (S * 32 * R bytes in all).
template <int R>
__device__ __forceinline__ size_t hb_index(int S, int rr, int cc) {
	const int k = rr / R, r = rr - k * R, st = cc + k;
	constexpr int G4 = R / 4;
	if(r < 4 * G4) return (size_t)(r >> 2) * ((size_t)S * 128) + ((size_t)st * 32 + k) * 4 + (r & 3);
	return (size_t)G4 * ((size_t)S * 128) + (size_t)(r - 4 * G4) * ((size_t)S * 32) + (size_t)st * 32 + k;
}

// ----------------------------------------------------------------------------------------
// The H-byte kernel runs as two launches per chunk: k_dp_fill_h writes the H bytes of a CHUNK of problems to a problem-indexed
// workspace (pure DPX compute, high occupancy), k_dp_tail_h then runs candidates + backtraces with one warp per
// problem (latency-bound on workspace reads, hidden by far more resident warps than one kernel doing both could hold).
template <typename OFF, int R, bool OFFDOM>
__global__ void __launch_bounds__(128, R <= 5 ? 8 : (R <= 6 ? 6 : 4)) k_dp_fill_h(DevIndex<OFF> ix, bt2g_scoring sc, DpLaunch L, uint64_t chunkStart, uint64_t chunkMax) {
	extern __shared__ uint8_t smem[];
	const int warpInBlock = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const uint64_t slot = blockIdx.x * (uint64_t)(blockDim.x >> 5) + warpInBlock;
	const uint64_t nSlots = (uint64_t)gridDim.x * (blockDim.x >> 5);
	const uint64_t nAll = L.nDev ? (uint64_t)*L.nDev : L.n;
	if(chunkStart >= nAll) return;
	const uint64_t nProb = (nAll - chunkStart < chunkMax) ? nAll - chunkStart : chunkMax;   // problems of this chunk
	const uint64_t nPairs = (nProb + 1) >> 1;
	// per warp: two reference windows, then the two query profiles [refc 0..4][row-in-lane][lane] as 16-bit scores
	// (buildQueryProfileEnd2EndSseU8, aligner_swsse_ee_u8.cpp:75-142): the substitution score of a cell is then two
	// shared-memory loads and one IMAD instead of five ALU-pipe instructions -- the ALU pipe is what bounds this kernel
	const size_t perProb = ((size_t)L.maxCol + 15) & ~(size_t)15;
	uint8_t *sm0 = smem + (size_t)warpInBlock * (2 * perProb + DP_QPROF_BYTES(R));
	uint8_t *refw[2] = {sm0, sm0 + perProb}; uint8_t *hb[2];
	// one 32-bit word per entry, [refc][row-in-lane][lane]: lane k always hits bank k whatever its reference character, so the
	// look-ups are conflict-free (16-bit entries put two lanes in one word: 45 % extra wavefronts in the ncu capture).  A word holds
	// problem A's score in its low half and problem B's in its high half; the packed pair of a cell is a bit-select of the words
	// its two reference characters pick
	uint32_t *qprof = reinterpret_cast<uint32_t *>(sm0 + 2 * perProb);
	const int rdgapo = sc.rdgap_const + sc.rdgap_linear, rdgape = sc.rdgap_linear;
	const int rfgapo = sc.rfgap_const + sc.rfgap_linear, rfgape = sc.rfgap_linear;
	const int bonus = sc.match_bonus;
	// OFFDOM (match bonus 0, the end-to-end default): every increment is <= 0, so clamping each intermediate value
	// at floor commutes with the recurrences (clamp(x) + s clamps to the same value as clamp(x + s) for s <= 0) and the
	// whole fill can run in the stored domain H - floor with 0 as its lower clamp: the H register IS the byte to store.
	const uint32_t FLOORP = OFFDOM ? L.zeroP : dpx_both(DPX_FLOOR);
	const uint32_t bonusP = dpx_both(bonus), nrdeP = dpx_both(-rdgape);

	for(uint64_t pw = slot; pw < nPairs; pw += nSlots) {
		uint64_t w[2] = {2 * pw, 2 * pw + 1};
		bool live[2] = {true, w[1] < nProb};
		if(!live[1]) w[1] = w[0];
		bt2g_dp_problem p[2] = {L.probs[chunkStart + w[0]], L.probs[chunkStart + w[1]]};
		hb[0] = L.codes + w[0] * L.codeStride; hb[1] = L.codes + w[1] * L.codeStride;
		const uint8_t *rs[2], *rq[2]; int rdlen[2], ncol[2], floorv[2];
		__syncwarp();
#pragma unroll
		for(int x = 0; x < 2; x++) {
			rs[x] = L.seq + L.roff[p[x].read_idx]; rq[x] = L.qual + L.roff[p[x].read_idx];
			rdlen[x] = (int)(L.roff[p[x].read_idx + 1] - L.roff[p[x].read_idx]);
			ncol[x] = (int)(p[x].refr - p[x].refl + 1);
			floorv[x] = p[x].minsc - bonus - 1;
			// shape, and the score range the byte encoding can hold (perfect - floor <= 127)
			if(ncol[x] <= 0 || ncol[x] > L.maxCol || rdlen[x] > 32 * R || rdlen[x] <= 0 ||
			   (int64_t)bonus * rdlen[x] - floorv[x] > 127 || floorv[x] < -DPX_LIMIT) {
				if(live[x] && lane == 0) {
					bt2g_dp_summary *sm = L.summ + chunkStart + w[x];
					sm->found = 0; sm->best = DP_NEG; sm->ncand = 0; sm->naln = 0; sm->flags = BT2G_DP_FLAG_BADSHAPE;
				}
				live[x] = false;
			}
		}
		if(!live[0] && !live[1]) continue;
		// a dead half mirrors the live one (its results are discarded)
		if(!live[0]) { p[0] = p[1]; rs[0] = rs[1]; rq[0] = rq[1]; rdlen[0] = rdlen[1]; ncol[0] = ncol[1]; floorv[0] = floorv[1]; }
		if(!live[1]) { p[1] = p[0]; rs[1] = rs[0]; rq[1] = rq[0]; rdlen[1] = rdlen[0]; ncol[1] = ncol[0]; floorv[1] = floorv[0]; }
		// reference windows (SwAligner::initRef, aligner_sw.cpp:155-271): codes 0..3, 4 = N / off-end
		const int ncolMax = ncol[0] > ncol[1] ? ncol[0] : ncol[1];
#pragma unroll
		for(int x = 0; x < 2; x++) {
			ref_window<OFF>(ix, p[x].tidx, p[x].refl, ncol[x], refw[x], lane);
			for(int k = ncol[x] + lane; k < ncolMax; k += 32) refw[x][k] = 4;      // padding read by the packed loop, never used
		}
		__syncwarp();

		// per-row constants of both problems (buildQueryProfileEnd2EndSseU8, aligner_swsse_ee_u8.cpp:75-142)
		uint32_t nrfoP[R], nrfeP[R], nrdoP[R];
#pragma unroll
		for(int r = 0; r < R; r++) {
			int v[2][6];
#pragma unroll
			for(int x = 0; x < 2; x++) {
				const int i = lane * R + r;
				bool bar = true;
				int c = 5, mm = 0, np = 0;
				if(i < rdlen[x]) {
					const int pos = p[x].fw ? i : rdlen[x] - 1 - i;
					c = rs[x][pos];
					c = p[x].fw ? c : (c > 3 ? 4 : 3 - c);
					int q = (int)rq[x][pos] - 33;
					q = q < 0 ? 0 : (q > 63 ? 63 : q);
					np = -(int)sc.npen[q];
					mm = c > 3 ? np : -(int)sc.mmpen[q];
					if(c > 3) c = 5;
					bar = (i < sc.gapbar) || (rdlen[x] - 1 - i < sc.gapbar);
				}
				// profile entries of this row: score against reference A, C, G, T and N
#pragma unroll
				for(int rf = 0; rf < 5; rf++)
					{
						const uint32_t v = (uint32_t)(uint16_t)(int16_t)(rf > 3 ? np : (c == rf ? bonus : mm));
						uint32_t &q = qprof[(rf * R + r) * 32 + lane];
						q = x == 0 ? v : (q | (v << 16));
					}
				v[x][3] = bar ? -DPX_BIG : -rfgapo; v[x][4] = bar ? -DPX_BIG : -rfgape; v[x][5] = bar ? -DPX_BIG : -rdgapo;
			}
			nrfoP[r] = dpx_pack(v[0][3], v[1][3]); nrfeP[r] = dpx_pack(v[0][4], v[1][4]); nrdoP[r] = dpx_pack(v[0][5], v[1][5]);
		}
		const int lastLane0 = (rdlen[0] - 1) / R, lastLane1 = (rdlen[1] - 1) / R;
		const int lastLaneMax = lastLane0 > lastLane1 ? lastLane0 : lastLane1;
		const uint32_t nfloorP = dpx_pack(-floorv[0], -floorv[1]);

		uint32_t Hleft[R], Earr[R];
#pragma unroll
		for(int r = 0; r < R; r++) { Hleft[r] = FLOORP; Earr[r] = FLOORP; }
		uint32_t botH = FLOORP, botF = FLOORP, prevInH = FLOORP;
		const int nsteps = ncolMax + lastLaneMax;
		// running store pointers: one per word plane and per byte plane of either problem
		const size_t P4 = (size_t)(L.maxCol + 32) * 128, P1 = (size_t)(L.maxCol + 32) * 32;
		uint8_t *w4A[R / 4 + 1], *w4B[R / 4 + 1], *w1A[R % 4 + 1], *w1B[R % 4 + 1];
#pragma unroll
		for(int g = 0; g < R / 4; g++) { w4A[g] = hb[0] + g * P4 + (size_t)lane * 4; w4B[g] = hb[1] + g * P4 + (size_t)lane * 4; }
#pragma unroll
		for(int g = 0; g < R % 4; g++) { w1A[g] = hb[0] + (R / 4) * P4 + g * P1 + lane; w1B[g] = hb[1] + (R / 4) * P4 + g * P1 + lane; }
		for(int t = 0; t < nsteps; t++) {
			uint32_t inH = __shfl_up_sync(0xffffffffu, botH, 1);
			uint32_t inF = __shfl_up_sync(0xffffffffu, botF, 1);
			if(lane == 0) { inH = FLOORP; inF = FLOORP; }
			const int j = t - lane;
			if(j >= 0 && j < ncolMax && lane <= lastLaneMax) {
				const uint32_t *qa = qprof + (int)refw[0][j] * (R * 32) + lane, *qb = qprof + (int)refw[1][j] * (R * 32) + lane;
				// H[i0-1][j-1]: row -1 is the free start row of end-to-end mode (vhilsw, :853,923-927)
				uint32_t diag = (lane == 0) ? (OFFDOM ? nfloorP : 0u) : prevInH;
				uint32_t upH = inH, upF = inF;
				uint32_t hs[DP_RP(R)];
#pragma unroll
				for(int r = R; r < DP_RP(R); r++) hs[r] = 0u;
#pragma unroll
				for(int r = 0; r < R; r++) {
					// F[i][j] = max(F[i-1][j]-rfgape, H[i-1][j]-rfgapo)
					const uint32_t F = __viaddmax_s16x2(upF, nrfeP[r], __viaddmax_s16x2(upH, nrfoP[r], FLOORP));
					const uint32_t sP = (qa[r * 32] & 0x0000ffffu) | (qb[r * 32] & 0xffff0000u);
					const uint32_t Hd = __viaddmax_s16x2(diag, sP, FLOORP);
					const uint32_t E = Earr[r];
					const uint32_t H = __vimax3_s16x2(Hd, E, F);
					// E[i][j+1] = max(E[i][j]-rdgape, H[i][j]-rdgapo)
					Earr[r] = __viaddmax_s16x2(E, nrdeP, __viaddmax_s16x2(H, nrdoP[r], FLOORP));
					hs[r] = OFFDOM ? H : __viaddmax_s16x2(H, nfloorP, 0u);  // max(H - floor, 0): the stored byte
					diag = Hleft[r]; Hleft[r] = H;
					upH = H; upF = F;
				}
				botH = upH; botF = upF;
				prevInH = inH;
				// byte 0 of every word is problem A's cell, byte 2 problem B's
#pragma unroll
				for(int q4 = 0; q4 < R / 4; q4++) {
					const uint32_t t01 = __byte_perm(hs[4 * q4], hs[4 * q4 + 1], 0x6240), t23 = __byte_perm(hs[4 * q4 + 2], hs[4 * q4 + 3], 0x6240);
					*reinterpret_cast<uint32_t *>(w4A[q4]) = __byte_perm(t01, t23, 0x5410);
					*reinterpret_cast<uint32_t *>(w4B[q4]) = __byte_perm(t01, t23, 0x7632);
				}
#pragma unroll
				for(int g = 0; g < R % 4; g++) {
					*w1A[g] = (uint8_t)(hs[(R / 4) * 4 + g] & 0xffu);
					*w1B[g] = (uint8_t)((hs[(R / 4) * 4 + g] >> 16) & 0xffu);
				}
			} else if(j >= ncolMax) {
				botH = FLOORP; botF = FLOORP;
			}
#pragma unroll
			for(int g = 0; g < R / 4; g++) { w4A[g] += 128; w4B[g] += 128; }
#pragma unroll
			for(int g = 0; g < R % 4; g++) { w1A[g] += 32; w1B[g] += 32; }
		}
	} // persistent loop over problem pairs
}

template <typename OFF, int R>
__global__ void __launch_bounds__(256) k_dp_tail_h(DevIndex<OFF> ix, bt2g_scoring sc, DpLaunch L, uint64_t chunkStart, uint64_t chunkMax) {
	extern __shared__ uint8_t smem[];
	const int warpInBlock = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const uint64_t nAll = L.nDev ? (uint64_t)*L.nDev : L.n;
	if(chunkStart >= nAll) return;
	const uint64_t nProb = (nAll - chunkStart < chunkMax) ? nAll - chunkStart : chunkMax;
	const size_t perWarp = dp_smem_per_warp(L.maxCol) + DP_PROF_BYTES(R);
	int32_t *lastH = reinterpret_cast<int32_t *>(smem + (size_t)warpInBlock * perWarp);
	uint16_t *candCol = reinterpret_cast<uint16_t *>(lastH + L.maxCol);
	uint8_t *refw = reinterpret_cast<uint8_t *>(candCol + L.maxCol);
	uint8_t *prof = smem + (size_t)warpInBlock * perWarp + dp_smem_per_warp(L.maxCol);
	const int bonus = sc.match_bonus;
	const uint64_t nWarps = (uint64_t)gridDim.x * (blockDim.x >> 5);
	for(uint64_t wl = blockIdx.x * (uint64_t)(blockDim.x >> 5) + warpInBlock; wl < nProb; wl += nWarps) {
		const uint64_t w = chunkStart + wl;
		const bt2g_dp_problem p = L.probs[w];
		const uint8_t *rs = L.seq + L.roff[p.read_idx], *rq = L.qual + L.roff[p.read_idx];
		const int rdlen = (int)(L.roff[p.read_idx + 1] - L.roff[p.read_idx]);
		const int ncol = (int)(p.refr - p.refl + 1);
		const int floorv = p.minsc - bonus - 1;
		__syncwarp();
		// the fill kernel flagged the same shapes as BADSHAPE
		if(ncol <= 0 || ncol > L.maxCol || rdlen > 32 * R || rdlen <= 0 || (int64_t)bonus * rdlen - floorv > 127 || floorv < -DPX_LIMIT) continue;
		uint8_t *hb = L.codes + wl * L.codeStride;
		ref_window<OFF>(ix, p.tidx, p.refl, ncol, refw, lane);
		for(int i = lane; i < rdlen; i += 32) {
			const int pos = p.fw ? i : rdlen - 1 - i;
			int c = rs[pos]; c = p.fw ? c : (c > 3 ? 4 : 3 - c);
			int q = (int)rq[pos] - 33; q = q < 0 ? 0 : (q > 63 ? 63 : q);
			prof[i] = (uint8_t)c; prof[rdlen + i] = sc.mmpen[q]; prof[2 * rdlen + i] = sc.npen[q];
		}
		// last row -> scores (candidates are the cells >= minsc; a clamped byte reads as floor < minsc)
		const int lr = rdlen - 1, kk = lr / R;
		for(int j = lane; j < ncol; j += 32) lastH[j] = (int)hb[hb_index<R>(L.maxCol + 32, lr, j)] + floorv;
		dp_e2e_tail<R, true>(L, sc, p, w, rs, rq, rdlen, ncol, lastH, candCol, refw, hb, L.summ + w, lane, prof);
	}
}

// ----------------------------------------------------------------------------------------
// "H-byte" end-to-end kernel: the fill stores ONE byte per cell that is the cell's H score itself
// (offset by floor = minsc - bonus - 1, clamped to [0,127]; bit 7 = reported-through mark), not a
// move code.  The fill then is just the three recurrences (13 DPX/logic instructions per row for two
// problems).  The backtrace re-derives each move from the stored scores, in the reference's
// preference order (aligner_swsse_ee_u8.cpp:1468-1520):
//   diag      H[i][j] == H[i-1][j-1] + score(i,j)          tested for a whole diagonal run at once;
//   ref gap   H[i][j] == H[i-k][j] - rfgapo - (k-1) rfgape  smallest k  (open first, then extensions:
//             exactly the F-state walk of the reference, because F[i][j] is the max of those terms);
//   read gap  H[i][j] == H[i][j-k] - rdgapo - (k-1) rdgape  smallest k,
// with the gap barrier of the recurrences (no F in barrier rows, no E opened from a barrier row).
// A clamped (zero) byte is a cell below floor: floor + bonus < minsc, so it can never satisfy an
// equality with a cell on a valid path.  Usable when perfect - floor <= 127 (dp_hbyte_ok).
template <int R>
__device__ __forceinline__ void dp_backtrace_h(const DpLaunch &L, const bt2g_scoring &sc, const bt2g_dp_problem &p, uint64_t w,
                                               const uint8_t *rs, const uint8_t *rq, int rdlen, const uint8_t *refw,
                                               uint8_t *hb, bt2g_dp_cand *cands, int ncand, bt2g_dp_summary *summ, int lane,
                                               const uint8_t *prof) {
	// prof (optional, shared memory): per read row the strand-adjusted base code, its mismatch and its N penalty
	const int rdgapo = sc.rdgap_const + sc.rdgap_linear, rdgape = sc.rdgap_linear;
	const int rfgapo = sc.rfgap_const + sc.rfgap_linear, rfgape = sc.rfgap_linear;
	const int bonus = sc.match_bonus, gapbar = sc.gapbar;
	const int vmax = bonus * rdlen - (p.minsc - bonus - 1);   // the largest byte a cell can hold: perfect score - floor
	bt2g_dp_aln *alns = L.alns + w * (uint64_t)L.maxAlns;
	uint8_t *ops = L.ops + w * (uint64_t)L.maxAlns * L.maxOps;
	int naln = 0, flags = 0;
	bool screened = false;
	const int S = L.maxCol + 32;
	auto cell = [&](int rr, int cc) -> uint8_t * { return hb + hb_index<R>(S, rr, cc); };
	auto rdchar = [&](int rr) -> int { const int pos = p.fw ? rr : rdlen - 1 - rr; int c = rs[pos]; return p.fw ? c : (c > 3 ? 4 : 3 - c); };
	auto rdqual = [&](int rr) -> int { const int pos = p.fw ? rr : rdlen - 1 - rr; int q = (int)rq[pos] - 33; return q < 0 ? 0 : (q > 63 ? 63 : q); };
	auto inCore = [&](int dlo, int dhi) -> bool { return dhi >= p.corel && dlo <= p.corer; };   // some diagonal of [dlo,dhi] is a core diagonal
	for(int ci = 0; ci < ncand; ci++) {
		int row = cands[ci].row, col = cands[ci].col;
		const int startRow = row, origCol = col;
		uint8_t *o = ops + (size_t)naln * L.maxOps;
		const bool room = naln < L.maxAlns;
		int nops = 0, ns = 0, gaps = 0;
		bool fail = false, core = false, done = false, first = true, filtStart = false;
		while(!done && !fail) {
			// ---- H state at (row, col): the diagonal run.  Lane k holds cell (row-k, col-k).
			// Every lane's byte sits in a different 32 B sector of the wavefront-major workspace, so a round costs as many
			// sectors as lanes that load.  Candidates after the best one usually leave their diagonal (and die on a
			// reported-through cell) within a few cells: their first round looks at 8 cells only.
			const int wd = (ci > 0 && first) ? 8 : 32;
			const int rk = row - lane, ck = col - lane;
			uint8_t *cp = (lane < wd && rk >= 0 && ck >= 0) ? cell(rk, ck) : nullptr;
			const int mine = cp ? (int)*cp : 0x80;
			const int v = mine & 0x7f;
			const int vn = __shfl_down_sync(0xffffffffu, v, 1);       // H of my diagonal predecessor (last loading lane: not loaded)
			int sck = 0, refc = 4; bool isN = false, isMatch = false;
			if(cp) {
				refc = refw[ck];
				if(prof) {
					const int c = prof[rk];
					isN = c > 3 || refc > 3;
					isMatch = !isN && c == refc;
					sck = isN ? -(int)prof[2 * rdlen + rk] : (isMatch ? bonus : -(int)prof[rdlen + rk]);
				} else {
					const int c = rdchar(rk), q = rdqual(rk);
					isN = c > 3 || refc > 3;
					isMatch = !isN && c == refc;
					sck = isN ? -(int)sc.npen[q] : (isMatch ? bonus : -(int)sc.mmpen[q]);
				}
			}
			const bool cont = lane < wd - 1 && !(mine & 0x80) && rk > 0 && ck > 0 && vn > 0 && v == vn + sck;
			const int run = __ffs(~__ballot_sync(0xffffffffu, cont)) - 1;   // 0..wd-1
			if(run > 0) {
				first = false;
				const int diagi = col - row + p.triml;
				if(inCore(diagi, diagi)) core = true;
				if(lane < run) {
					const uint8_t op = (uint8_t)((isMatch ? BT2G_OP_MATCH : BT2G_OP_MM) | (refc << 2));
					if(room && nops + lane < L.maxOps) o[nops + lane] = op;
					*cp = (uint8_t)(mine | 0x80);                      // setReportedThrough (:1555)
				}
				ns += __popc(__ballot_sync(0xffffffffu, lane < run && isN));
				nops += run; row -= run; col -= run;
			}
			const int endBits = __shfl_sync(0xffffffffu, mine, run);   // the cell at (row, col) now
			if(run == wd - 1 && !(endBits & 0x80) && row > 0 && col > 0) { __syncwarp(); continue; }   // last loaded cell: decide next round
			// ---- the cell that ends the run
			if(endBits & 0x80) {
				// start cell already reported through -> BT_CAND_FATE_FILT_START (:771-789); elsewhere the backtrace fails
				if(first) filtStart = true;
				fail = true; break;
			}
			first = false;
			if(lane == run) *cp = (uint8_t)(mine | 0x80);
			{
				const int diagi = col - row + p.triml;
				if(inCore(diagi, diagi)) core = true;
			}
			if(row == 0) { done = true; break; }
			const int cur = endBits & 0x7f;
			__syncwarp();
			// ---- which gap?  decided from scores only; reference gap (vertical) before read gap (horizontal)
			int klen = 0, gapKind = 0;                                 // 1 ref gap (rows), 2 read gap (columns)
			if(row >= gapbar && rdlen - 1 - row >= gapbar) {
				for(int k0 = 0; k0 < row; k0 += 32) {
					if(vmax - rfgapo - k0 * rfgape < cur) break;       // longer gaps cannot reach cur any more
					const int k = k0 + lane + 1, r2 = row - k;
					bool ok = false;
					if(r2 >= 0 && row - k + 1 >= gapbar && vmax - rfgapo - (k - 1) * rfgape >= cur) {   // rows row-k+1..row outside the barrier
						const int u = *cell(r2, col) & 0x7f;
						ok = u > 0 && u - rfgapo - (k - 1) * rfgape == cur;
					}
					const uint32_t mk = __ballot_sync(0xffffffffu, ok);
					if(mk) { klen = k0 + __ffs(mk); gapKind = 1; break; }
				}
				if(gapKind == 0) {
					for(int k0 = 0; k0 < col; k0 += 32) {
						if(vmax - rdgapo - k0 * rdgape < cur) break;
						const int k = k0 + lane + 1, c2 = col - k;
						bool ok = false;
						if(c2 >= 0 && vmax - rdgapo - (k - 1) * rdgape >= cur) {
							const int u = *cell(row, c2) & 0x7f;
							ok = u > 0 && u - rdgapo - (k - 1) * rdgape == cur;
						}
						const uint32_t mk = __ballot_sync(0xffffffffu, ok);
						if(mk) { klen = k0 + __ffs(mk); gapKind = 2; break; }
					}
				}
			}
			if(gapKind == 0) { fail = true; break; }                   // no legal move (cannot happen for a cell >= minsc)
			// ---- the klen-1 gap-state cells in between: reported-through check in walking order, then mark
			for(int m0 = 1; m0 < klen && !fail; m0 += 32) {
				const int mth = m0 + lane;
				uint8_t *q2 = nullptr; int b = 0;
				if(mth < klen) { q2 = gapKind == 1 ? cell(row - mth, col) : cell(row, col - mth); b = *q2; }
				const uint32_t vm = __ballot_sync(0xffffffffu, (b & 0x80) != 0);
				const int lim = vm ? __ffs(vm) - 1 : 32;
				if(q2 && lane < lim) *q2 = (uint8_t)(b | 0x80);
				if(vm) fail = true;
			}
			if(fail) break;
			{
				const int d0 = col - row + p.triml, ni = klen - 1;
				if(ni > 0 && (gapKind == 1 ? inCore(d0 + 1, d0 + ni) : inCore(d0 - ni, d0 - 1))) core = true;
			}
			if(room) {
				for(int k = lane; k < klen; k += 32) {
					const int idx = nops + k;
					if(idx < L.maxOps) o[idx] = gapKind == 1 ? (uint8_t)BT2G_OP_REFGAP : (uint8_t)(BT2G_OP_READGAP | (refw[col - k] << 2));
				}
			}
			nops += klen; gaps += klen;
			if(gapKind == 1) row -= klen; else col -= klen;
			__syncwarp();
		}
		if(filtStart) { if(lane == 0) cands[ci].fate = BT2G_CAND_FILT_START; continue; }
		if(!fail) {
			// the alignment's first cell (row, col) (:1797-1813)
			const int c = rdchar(row), refc = refw[col];
			const bool isN = c > 3 || refc > 3;
			ns += isN;
			const uint8_t op = (uint8_t)(((!isN && c == refc) ? BT2G_OP_MATCH : BT2G_OP_MM) | (refc << 2));
			if(!core) fail = true;                   // core-diagonal rejection (:1764-1795)
			else if(ns > p.nceil) fail = true;       // N ceiling (:1813-1818)
			else {
				if(room && lane == 0 && nops < L.maxOps) o[nops] = op;
				nops++;
			}
		}
		const bool opOverflow = nops > L.maxOps;
		if(fail) { if(lane == 0) cands[ci].fate = BT2G_CAND_FAILED; continue; }
		if(lane == 0) cands[ci].fate = BT2G_CAND_SUCCEEDED;
		if(room) {
			int refns = 0;
			for(int k = col + lane; k <= origCol; k += 32) refns += refw[k] > 3;
			refns = __reduce_add_sync(0xffffffffu, refns);
			if(lane == 0) {
				bt2g_dp_aln &a = alns[naln];
				a.cand_idx = ci; a.score = cands[ci].score; a.ns = ns; a.gaps = gaps; a.col0 = col; a.row0 = row;
				a.trim_beg = 0; a.trim_end = rdlen - 1 - startRow; a.nops = nops;
				a.refns = refns;
			}
			if(opOverflow) flags |= BT2G_DP_FLAG_OPS_OVERFLOW;
		} else {
			flags |= BT2G_DP_FLAG_ALN_OVERFLOW;
		}
		naln++;
		// ---- screening of the remaining candidates, one per lane.  After the first alignment almost every other
		// candidate is a shifted variant that runs into its reported-through cells within a few moves.  A read-only
		// walk against the marks that exist NOW decides each of them independently: marks added later (by other
		// failing candidates) can only make a walk stop earlier, so "fails now" implies "fails in sequence", and a
		// failing candidate changes nothing but marks.  Only if some walk gets through to row 0 is the sequential
		// procedure above needed for the rest (it then runs unchanged, from the next candidate).
		if(naln == 1 && !screened && ci + 1 < ncand) {
			screened = true;
			bool needSeq = false;
			for(int base = ci + 1; base < ncand; base += 32) {
				const int cj = base + lane;
				int verdict = 0;                               // 0 fails, 1 start cell already reported through, 2 might succeed
				if(cj < ncand) {
					int r2 = cands[cj].row, c2 = cands[cj].col;
					int b = *cell(r2, c2);
					if(b & 0x80) verdict = 1;
					else {
						for(int guard = 0; guard < 4 * rdlen + 8; guard++) {
							const int curv = b & 0x7f;
							if(r2 == 0) { verdict = 2; break; }
							if(c2 > 0) {
								const int pb = *cell(r2 - 1, c2 - 1), pv = pb & 0x7f;
								const int rf = refw[c2];
								int c, mm, np;
								if(prof) { c = prof[r2]; mm = prof[rdlen + r2]; np = prof[2 * rdlen + r2]; }
								else { c = rdchar(r2); const int q = rdqual(r2); mm = sc.mmpen[q]; np = sc.npen[q]; }
								const int sc2 = (c > 3 || rf > 3) ? -np : (c == rf ? bonus : -mm);
								if(pv > 0 && curv == pv + sc2) {
									if(pb & 0x80) break;              // runs into a reported-through cell
									r2--; c2--; b = pb;
									continue;
								}
							}
							if(r2 < gapbar || rdlen - 1 - r2 < gapbar) break;         // no legal move
							bool moved = false, dead = false, marked = false;
							for(int k = 1; k <= r2 && r2 - k + 1 >= gapbar && vmax - rfgapo - (k - 1) * rfgape >= curv; k++) {
								const int ub = *cell(r2 - k, c2), u = ub & 0x7f;
								if(u > 0 && u - rfgapo - (k - 1) * rfgape == curv) {
									if(marked || (ub & 0x80)) dead = true; else { r2 -= k; b = ub; moved = true; }
									break;
								}
								marked = marked || (ub & 0x80);
							}
							if(!moved && !dead) {
								marked = false;
								for(int k = 1; k <= c2 && vmax - rdgapo - (k - 1) * rdgape >= curv; k++) {
									const int ub = *cell(r2, c2 - k), u = ub & 0x7f;
									if(u > 0 && u - rdgapo - (k - 1) * rdgape == curv) {
										if(marked || (ub & 0x80)) dead = true; else { c2 -= k; b = ub; moved = true; }
										break;
									}
									marked = marked || (ub & 0x80);
								}
							}
							if(!moved) break;                      // dead end or no legal move: fails
						}
					}
				}
				if(__any_sync(0xffffffffu, verdict == 2)) { needSeq = true; break; }
				if(cj < ncand) cands[cj].fate = verdict == 1 ? BT2G_CAND_FILT_START : BT2G_CAND_FAILED;
			}
			__syncwarp();
			if(!needSeq) break;
			// some fates were written by lanes of completed groups; the sequential pass below rewrites all of them
		}
	}
	if(lane == 0) { summ->naln = naln; summ->flags |= flags; }
}

// persistent grid = resident blocks only (a second, partial wave would double the makespan)
template <typename K>
static unsigned dp_resident_grid(K kernel, int threads, size_t smem, uint64_t numSlots, int warpsPerBlock) {
	int dev = 0, sms = 148, nb = 1;
	cudaGetDevice(&dev);
	cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
	if(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, threads, smem) != cudaSuccess || nb < 1) nb = 1;
	uint64_t g = (uint64_t)nb * sms, cap = numSlots / warpsPerBlock;
	return (unsigned)(g < cap ? g : cap);
}

template <typename OFF, int R>
static void launch_dp_e2e_r(const DevIndex<OFF> &ix, const bt2g_scoring &sc, const DpLaunch &L, cudaStream_t st) {
	const int warpsPerBlock = 4;
	if(L.packed == 3) {
		// split: chunks of L.chunk problems through fill then tail (workspace = L.chunk * codeStride bytes)
		int dev = 0, sms = 148; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
		const size_t smF = (size_t)warpsPerBlock * (2 * (((size_t)L.maxCol + 15) & ~(size_t)15) + DP_QPROF_BYTES(R));
		const size_t smT = (size_t)8 * (dp_smem_per_warp(L.maxCol) + DP_PROF_BYTES(R));
		auto kfill = sc.match_bonus == 0 ? k_dp_fill_h<OFF, R, true> : k_dp_fill_h<OFF, R, false>;
		if(smF > 48 * 1024) cudaFuncSetAttribute(kfill, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smF);
		if(smT > 48 * 1024) cudaFuncSetAttribute(k_dp_tail_h<OFF, R>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smT);
		int nbF = 1, nbT = 1;
		if(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nbF, kfill, warpsPerBlock * 32, smF) != cudaSuccess || nbF < 1) nbF = 1;
		if(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nbT, k_dp_tail_h<OFF, R>, 256, smT) != cudaSuccess || nbT < 1) nbT = 1;
		auto mark = [&]() { if(L.tev && L.tevN && *L.tevN < L.tevCap) cudaEventRecord(L.tev[(*L.tevN)++], st); };
		mark();
		for(uint64_t c0 = 0; c0 < L.n; c0 += L.chunk) {
			kfill<<<(unsigned)(nbF * sms), warpsPerBlock * 32, smF, st>>>(ix, sc, L, c0, L.chunk);
			mark();
			k_dp_tail_h<OFF, R><<<(unsigned)(nbT * sms), 256, smT, st>>>(ix, sc, L, c0, L.chunk);
			mark();
		}
	} else if(L.packed) {
		const size_t smem = (size_t)warpsPerBlock * 2 * dp_smem_per_warp(L.maxCol);
		if(smem > 48 * 1024) cudaFuncSetAttribute(k_dp_e2e_x2<OFF, R>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
		const unsigned grid = dp_resident_grid(k_dp_e2e_x2<OFF, R>, warpsPerBlock * 32, smem, L.numSlots, warpsPerBlock);
		k_dp_e2e_x2<OFF, R><<<grid, warpsPerBlock * 32, smem, st>>>(ix, sc, L);
	} else {
		const size_t smem = (size_t)warpsPerBlock * dp_smem_per_warp(L.maxCol);
		if(smem > 48 * 1024) cudaFuncSetAttribute(k_dp_e2e<OFF, R>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
		const unsigned grid = dp_resident_grid(k_dp_e2e<OFF, R>, warpsPerBlock * 32, smem, L.numSlots, warpsPerBlock);
		k_dp_e2e<OFF, R><<<grid, warpsPerBlock * 32, smem, st>>>(ix, sc, L);
	}
}

// L.packed selects the two-problems-per-warp s16x2 kernel; the caller guarantees the score range
// (dp_packed_ok) and a workspace of 2 * codeStride bytes per slot.
template <typename OFF>
int launch_dp_e2e(const DevIndex<OFF> &ix, const bt2g_scoring &sc, const DpLaunch &L, int maxRdLen, cudaStream_t st) {
	if(L.n == 0) return 0;
	switch(dp_rows_per_lane(maxRdLen, L.packed)) {
		case 4: launch_dp_e2e_r<OFF, 4>(ix, sc, L, st); break;
		case 5: launch_dp_e2e_r<OFF, 5>(ix, sc, L, st); break;
		case 6: launch_dp_e2e_r<OFF, 6>(ix, sc, L, st); break;
		case 8: launch_dp_e2e_r<OFF, 8>(ix, sc, L, st); break;
		case 10: launch_dp_e2e_r<OFF, 10>(ix, sc, L, st); break;
		case 12: launch_dp_e2e_r<OFF, 12>(ix, sc, L, st); break;
		case 16: launch_dp_e2e_r<OFF, 16>(ix, sc, L, st); break;
		default: return -1;
	}
	return 0;
}
template int launch_dp_e2e<uint32_t>(const DevIndex<uint32_t> &, const bt2g_scoring &, const DpLaunch &, int, cudaStream_t);
template int launch_dp_e2e<uint64_t>(const DevIndex<uint64_t> &, const bt2g_scoring &, const DpLaunch &, int, cudaStream_t);

// ----------------------------------------------------------------------------------------
// Local mode (alignNucleotidesLocalSseU8/I16, aligner_swsse_loc_i16.cpp:938-1367; gather
// :1420-1535; backtrace :1615-2218).  Same wavefront; differences from end-to-end:
//   * every score is floored at 0 (the reference stores score-0x8000 and lets signed saturation
//     clamp, :1004-1017,1107), row -1 and column -1 are 0;
//   * a move is legal only from a source cell whose score is > 0 (floorsc = 0, :1683-1840), so the
//     move codes are computed from the explicit equality tests, and "no legal move" ends the
//     alignment (soft trimming);
//   * candidates are all cells with score >= minsc in rows >= minrow whose own base matches and
//     whose diagonal successor does not (:1497-1518), collected during the fill.
// The u8 -> i16 rerun of the reference (aligner_sw.cpp:569-605) has no counterpart: scores are exact.
// ----------------------------------------------------------------------------------------
template <typename OFF, int R>
__global__ void __launch_bounds__(128) k_dp_local(DevIndex<OFF> ix, bt2g_scoring sc, DpLaunch L) {
	extern __shared__ uint8_t smem[];
	const int warpInBlock = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const uint64_t slot = blockIdx.x * (uint64_t)(blockDim.x >> 5) + warpInBlock;
	const uint64_t nSlots = (uint64_t)gridDim.x * (blockDim.x >> 5);
	const uint64_t nProb = L.nDev ? (uint64_t)*L.nDev : L.n;
	const size_t perWarp = dp_smem_per_warp(L.maxCol);
	int32_t *wsm = reinterpret_cast<int32_t *>(smem + (size_t)warpInBlock * perWarp);   // [0] = raw candidate counter
	uint8_t *refw = reinterpret_cast<uint8_t *>(wsm + L.maxCol) + 2 * (size_t)L.maxCol;
	uint8_t *codes = L.codes + slot * L.codeStride;
	uint64_t *raw = L.rawKeys + slot * (uint64_t)L.maxRaw;
	const int rdgapo = sc.rdgap_const + sc.rdgap_linear, rdgape = sc.rdgap_linear;
	const int rfgapo = sc.rfgap_const + sc.rfgap_linear, rfgape = sc.rfgap_linear;
	const int bonus = sc.match_bonus;

	for(uint64_t w = slot; w < nProb; w += nSlots) {
		const bt2g_dp_problem p = L.probs[w];
		const uint8_t *rs = L.seq + L.roff[p.read_idx];
		const uint8_t *rq = L.qual + L.roff[p.read_idx];
		const int rdlen = (int)(L.roff[p.read_idx + 1] - L.roff[p.read_idx]);
		const int ncol = (int)(p.refr - p.refl + 1);
		bt2g_dp_summary *summ = L.summ + w;
		__syncwarp();
		if(ncol <= 0 || ncol + 1 > L.maxCol || rdlen > 32 * R || rdlen <= 0 || bonus <= 0) {
			if(lane == 0) { summ->found = 0; summ->best = DP_NEG; summ->ncand = 0; summ->naln = 0; summ->flags = BT2G_DP_FLAG_BADSHAPE; }
			continue;
		}
		// reference window plus the one extra character initRef captures (aligner_sw.cpp:170-173)
		for(int k = lane; k <= ncol; k += 32) refw[k] = (uint8_t)ref_base<OFF>(ix, p.tidx, p.refl + k);
		if(lane == 0) wsm[0] = 0;
		__syncwarp();

		int rc[R + 1], mmp[R], npn[R];
		bool bar[R];
#pragma unroll
		for(int r = 0; r <= R; r++) {
			int i = lane * R + r;
			int c = 6;                                   // beyond the read: matches nothing
			if(i < rdlen) {
				int pos = p.fw ? i : rdlen - 1 - i;
				c = rs[pos];
				c = p.fw ? c : (c > 3 ? 4 : 3 - c);
				if(r < R) {
					int q = (int)rq[pos] - 33;
					q = q < 0 ? 0 : (q > 63 ? 63 : q);
					npn[r] = sc.npen[q];
					mmp[r] = c > 3 ? npn[r] : sc.mmpen[q];
					bar[r] = (i < sc.gapbar) || (rdlen - 1 - i < sc.gapbar);
				}
			} else if(r < R) { mmp[r] = 0; npn[r] = 0; bar[r] = true; }
			rc[r] = c;                                   // raw code 0..4 (N = 4 matches a reference N in the gather test)
		}
		const int lastLane = (rdlen - 1) / R;
		const int minrow = (int)(((int64_t)p.minsc + bonus - 1) / bonus) - 1;   // aligner_swsse_loc_i16.cpp:1437

		int Hleft[R], Earr[R], Eprev[R];
#pragma unroll
		for(int r = 0; r < R; r++) { Hleft[r] = 0; Earr[r] = 0; Eprev[r] = 0; }
		int botH = 0, botF = 0, prevInH = 0, lmax = 0;
		const int nsteps = ncol + lastLane;
		for(int t = 0; t < nsteps; t++) {
			int inH = __shfl_up_sync(0xffffffffu, botH, 1);
			int inF = __shfl_up_sync(0xffffffffu, botF, 1);
			if(lane == 0) { inH = 0; inF = 0; }
			const int j = t - lane;
			if(j >= 0 && j < ncol && lane <= lastLane) {
				const int refc = refw[j], refn = refw[j + 1];
				const bool refN = refc > 3;
				int diag = (lane == 0) ? 0 : prevInH;
				int upH = inH, upF = inF;
				uint32_t packed[(R + 3) / 4];
#pragma unroll
				for(int q4 = 0; q4 < (R + 3) / 4; q4++) packed[q4] = 0;
#pragma unroll
				for(int r = 0; r < R; r++) {
					const int i = lane * R + r;
					const int fo = upH - rfgapo, fe = upF - rfgape;
					int F = bar[r] ? 0 : dp_max(dp_max(fo, fe), 0);
					const int fsel = (upH > 0 && fo == F) ? 1 : ((upF > 0 && fe == F) ? 2 : 0);
					int s = (rc[r] == refc && !refN) ? bonus : -mmp[r];
					s = (refN || rc[r] > 3) ? -npn[r] : s;
					const int Hd = diag + s;
					const int E = Earr[r];
					const int H = dp_max(__vimax3_s32(Hd, E, F), 0);
					int hsel = 0;
					if(diag > 0 && H == Hd) hsel = 1;
					else if(!bar[r]) {
						if(upH > 0 && H == fo) hsel = 2;
						else if(upF > 0 && H == fe) hsel = 3;
						else if(Hleft[r] > 0 && H == Hleft[r] - rdgapo) hsel = 4;
						else if(Eprev[r] > 0 && H == Eprev[r] - rdgape) hsel = 5;
					}
					const int esel = (Hleft[r] > 0 && Hleft[r] - rdgapo == E) ? 1 : ((Eprev[r] > 0 && Eprev[r] - rdgape == E) ? 2 : 0);
					const uint32_t code = (uint32_t)(hsel | (esel << 3) | (fsel << 5));
					packed[r >> 2] |= code << ((r & 3) * 8);
					const int eo = bar[r] ? 0 : H - rdgapo, ee = E - rdgape;
					// candidate cell (gatherCellsNucleotidesLocalSseI16, :1485-1518)
					if(i < rdlen && i >= minrow && H >= p.minsc && rc[r] == refc && !(i < rdlen - 1 && rc[r + 1] == refn)) {
						const int pos = atomicAdd(&wsm[0], 1);
						if(pos < L.maxRaw) raw[pos] = ((uint64_t)(uint32_t)H << 32) | ((uint64_t)i << 16) | (uint64_t)j;
					}
					lmax = dp_max(lmax, i < rdlen ? H : 0);
					diag = Hleft[r]; Hleft[r] = H; Eprev[r] = E; Earr[r] = dp_max(dp_max(eo, ee), 0);
					upH = H; upF = F;
				}
				botH = upH; botF = upF;
				prevInH = inH;
				uint8_t *dst = codes + ((size_t)t * 32 + lane) * R;
				if(R == 4) *reinterpret_cast<uint32_t *>(dst) = packed[0];
				else if(R == 8) *reinterpret_cast<uint2 *>(dst) = make_uint2(packed[0], packed[1]);
				else {
#pragma unroll
					for(int q4 = 0; q4 < (R + 3) / 4; q4++) reinterpret_cast<uint32_t *>(dst)[q4] = packed[q4];
				}
			} else if(j >= ncol) {
				botH = 0; botF = 0;
			}
		}
		__syncwarp();
		int best = lmax;
#pragma unroll
		for(int o = 16; o > 0; o >>= 1) best = dp_max(best, __shfl_xor_sync(0xffffffffu, best, o));
		if(lane == 0) { summ->best = best; summ->flags = 0; summ->naln = 0; summ->ncand = 0; summ->found = 0; }
		if(best < p.minsc) continue;
		// sort: DpBtCandidate::operator< = score desc, row desc, col desc = key desc
		const int nrawAll = wsm[0];
		const int nraw = nrawAll < L.maxRaw ? nrawAll : L.maxRaw;
		bt2g_dp_cand *cands = L.cands + w * (uint64_t)L.maxCands;
		for(int a0 = 0; a0 < nraw; a0 += 32) {
			const int a = a0 + lane;
			if(a < nraw) {
				const uint64_t key = raw[a];
				int rank = 0;
				for(int k = 0; k < nraw; k++) rank += raw[k] > key;
				if(rank < L.maxCands) {
					cands[rank].score = (int32_t)(key >> 32); cands[rank].row = (int32_t)((key >> 16) & 0xffff);
					cands[rank].col = (int32_t)(key & 0xffff); cands[rank].fate = 0;
				}
			}
		}
		const int ncand = nraw < L.maxCands ? nraw : L.maxCands;
		if(lane == 0) {
			summ->ncand = nrawAll; summ->found = nrawAll > 0;
			if(nrawAll > L.maxCands || nrawAll > L.maxRaw) summ->flags |= BT2G_DP_FLAG_CAND_OVERFLOW;
		}
		__syncwarp();
		dp_backtrace_all<R>(L, sc, p, w, rs, rq, rdlen, refw, codes, cands, ncand, summ, lane, true);
	}
}

template <typename OFF>
int launch_dp_local(const DevIndex<OFF> &ix, const bt2g_scoring &sc, const DpLaunch &L, int maxRdLen, cudaStream_t st) {
	if(L.n == 0) return 0;
	const int warpsPerBlock = 4;
	const size_t perWarp = dp_smem_per_warp(L.maxCol);
	size_t smem = (size_t)warpsPerBlock * perWarp;
	unsigned grid = (unsigned)(L.numSlots / warpsPerBlock);
	if(maxRdLen <= 128) {
		if(smem > 48 * 1024) cudaFuncSetAttribute(k_dp_local<OFF, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
		k_dp_local<OFF, 4><<<grid, warpsPerBlock * 32, smem, st>>>(ix, sc, L);
	} else if(maxRdLen <= 256) {
		if(smem > 48 * 1024) cudaFuncSetAttribute(k_dp_local<OFF, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
		k_dp_local<OFF, 8><<<grid, warpsPerBlock * 32, smem, st>>>(ix, sc, L);
	} else if(maxRdLen <= 512) {
		if(smem > 48 * 1024) cudaFuncSetAttribute(k_dp_local<OFF, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
		k_dp_local<OFF, 16><<<grid, warpsPerBlock * 32, smem, st>>>(ix, sc, L);
	} else {
		return -1;
	}
	return 0;
}
template int launch_dp_local<uint32_t>(const DevIndex<uint32_t> &, const bt2g_scoring &, const DpLaunch &, int, cudaStream_t);
template int launch_dp_local<uint64_t>(const DevIndex<uint64_t> &, const bt2g_scoring &, const DpLaunch &, int, cudaStream_t);
