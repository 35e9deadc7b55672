// dp_device.cuh -- launch descriptor shared by api.cu and dp_kernels.cu (DP types: include/bt2g.h)
#pragma once
#include "bt2g_internal.h"
#include <cstdlib>

// the s16x2 kernel needs every reachable score within +-DPX_LIMIT (dp_kernels.cu): end-to-end mode,
// minimum score >= -8000 and perfect score <= 8000
static inline bool dp_packed_ok(const bt2g_scoring &sc, int64_t minMinsc, int maxLen) {
	return !sc.local && minMinsc >= -8000 && (int64_t)sc.match_bonus * maxLen <= 8000 && sc.match_bonus >= 0;
}

// DpLaunch.packed: 0 = k_dp_e2e (32-bit, move codes), 1 = k_dp_e2e_x2 (s16x2, move codes),
// 3 = k_dp_fill_h + k_dp_tail_h (s16x2, H bytes: needs perfect - (minsc - bonus - 1) <= 127 for every problem)
//     over chunks of DpLaunch.chunk problems (workspace: chunk * codeStride bytes).
// The result is the highest of these modes that the batch allows and that is <= `cap` (bt2g_ctx::dpModeCap, set by
// bt2g_set_dp_mode), so a cap of 2 picks mode 1.
static inline int dp_kernel_mode(const bt2g_scoring &sc, int64_t minMinsc, int maxLen, int cap = 3) {
	if(cap < 0 || cap > 3) cap = 3;
	if(cap == 0 || !dp_packed_ok(sc, minMinsc, maxLen)) return 0;
	const int64_t range = (int64_t)sc.match_bonus * maxLen - (minMinsc - sc.match_bonus - 1);
	return (cap >= 3 && range <= 127) ? 3 : 1;
}

// rows per lane: the H-byte kernels (mode 3) take the smallest R of {4,5,6,8,10,12,16} with 32 R >= rdlen
// (a 150 bp read fills 30 lanes at R = 5 instead of 19 at R = 8); the move-code kernels use 4 / 8 / 16.
static inline int dp_rows_per_lane(int maxLen, int mode) {
	if(mode == 3) {
		const int rs[7] = {4, 5, 6, 8, 10, 12, 16};
		for(int i = 0; i < 7; i++) if(32 * rs[i] >= maxLen) return rs[i];
		return 0;
	}
	return maxLen <= 128 ? 4 : (maxLen <= 256 ? 8 : (maxLen <= 512 ? 16 : 0));
}
// bytes of workspace per problem (per warp slot in modes 0 and 1): (maxCol + 32) steps x 32 lanes x R rows
static inline uint64_t dp_code_stride(int maxCol, int maxLen, int mode) {
	const int R = dp_rows_per_lane(maxLen, mode);
	return (((uint64_t)(maxCol + 32) * 32 * (uint64_t)R) + 255) & ~(uint64_t)255;   // planes of hb_index, 256 B aligned
}

// mode 3 workspace: as many problems per chunk as fit a byte budget (default 6 GiB; BT2G_DP_CHUNK_MB overrides)
static inline uint64_t dp_chunk_problems(uint64_t codeStride, uint64_t nMax, uint64_t budget = 6ull << 30) {
	if(const char *e = getenv("BT2G_DP_CHUNK_MB")) { uint64_t v = strtoull(e, nullptr, 10); if(v) budget = v << 20; }
	uint64_t c = budget / (codeStride ? codeStride : 1);
	if(c < 1024) c = 1024;
	if(c > nMax) c = nMax;
	return c ? c : 1;
}

struct DpLaunch {
	const uint8_t  *seq, *qual;
	const uint64_t *roff;
	const bt2g_dp_problem *probs;
	uint64_t        n;
	const uint32_t *nDev;         // optional: problem count produced on the device
	uint64_t        numSlots;     // persistent warp slots (multiple of 4)
	uint8_t        *codes;        // workspace: n * codeStride bytes
	int32_t        *lastH;
	uint64_t       *rawKeys;      // local mode: per-slot candidate keys (score<<32 | row<<16 | col)
	int             maxRaw;        // workspace: n * maxCol ints (e2e last-row scores)
	uint64_t        codeStride;
	int             maxCol;
	int             maxCands, maxAlns, maxOps;
	uint64_t        chunk = 0;    // mode 3: problems per fill/tail chunk
	int             packed = 0;   // e2e: two problems per warp as s16x2 pairs (codes workspace: 2 * codeStride per slot)
	cudaEvent_t    *tev = nullptr;  // optional timing marks (mode 3): one before the first fill, then one after every fill and every tail
	int             tevCap = 0;
	int            *tevN = nullptr;
	uint32_t        zeroP = 0;    // always 0: a zero the compiler cannot see through, so that it stays in ONE register (a literal 0 as
	                              // the third operand of VIADDMNMX is re-materialised with a PRMT before every use: 13 per step)
	bt2g_dp_summary *summ;
	bt2g_dp_cand    *cands;
	bt2g_dp_aln     *alns;
	uint8_t         *ops;
};
