// fm_seed2.cu -- K1 v2: exact multiseed search with full lanes.
//
// The first version gave every (read, strand, seed) its own thread and let it run to
// completion; ncu showed 6.5 of 32 lanes active per instruction (seeds die at different steps,
// reverse-strand seeds of a forward read die after ~6 steps, and the range>1 / range==1 paths
// serialised), so the kernel was issue-bound at 20 % of HBM bandwidth (profiles/r01_*).
// This version keeps lanes full:
//   * reads are first packed to 2 bits/base (+ an N bit mask) by k_pack_reads, so a whole seed
//     (<= 32 bases) lives in one 64-bit register: no byte loads or strand branches per step;
//   * ONE uniform step for every range size: ranks are taken at top and bot whatever the width.
//     For a width-1 range this equals Ebwt::mapLF1 (bt2_idx.h:2420): rank_c(top+1)-rank_c(top) is
//     1 exactly when BWT[top] == c and top is not the "$" row (the "$" adjustment of
//     countBt2Side removes it), and the mirror range is unchanged because every other width is 0;
//     when top and bot fall in the same side the side is fetched once;
//   * persistent lanes: a lane whose seed finished or died pulls the next task from a global
//     counter (one warp-aggregated atomic per refill), so a warp keeps 32 searches in flight.
#include "fm_device.cuh"
#include "launch.cuh"

#define REFILL_MIN 8

// 2-bit packing of a read batch.  Word w of read r holds bases 32w..32w+31 (base i at bits 2(i&31)),
// nmask has the same word structure with one bit per base.  Word offset of read r is
// (roff[r] >> 5) + r, which needs no extra offset array and never overlaps the next read.
__global__ void k_pack_reads(const uint8_t *seq, const uint64_t *roff, uint64_t nReads, int maxWords,
                             uint64_t *packed, uint32_t *nmask) {
	uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if(t >= nReads * (uint64_t)maxWords) return;
	const uint64_t rd = t / maxWords;
	const int w = (int)(t - rd * maxWords);
	const int len = (int)(roff[rd + 1] - roff[rd]);
	if(w * 32 >= len) return;
	const uint8_t *s = seq + roff[rd] + (uint64_t)w * 32;
	const int n = len - w * 32 < 32 ? len - w * 32 : 32;
	uint64_t p = 0; uint32_t m = 0;
	for(int i = 0; i < n; i++) {
		const uint32_t c = s[i];
		if(c > 3) m |= 1u << i; else p |= (uint64_t)c << (2 * i);
	}
	const uint64_t wb = (roff[rd] >> 5) + rd + (uint64_t)w;
	packed[wb] = p; nmask[wb] = m;
}

// reverse the order of the n 2-bit groups held in the low 2n bits of x
__device__ __forceinline__ uint64_t rev_pairs(uint64_t x, int n) {
	uint64_t r = __brevll(x);
	r = ((r >> 1) & 0x5555555555555555ull) | ((r & 0x5555555555555555ull) << 1);
	return r >> (64 - 2 * n);
}

template <typename OFF>
__device__ __forceinline__ void rank4_loaded(const DevEbwt<OFF> &e, const SideRegs<OFF> &s, uint64_t sideNum, uint32_t charOff, uint64_t out[4]) {
	uint32_t nC, nG, nT;
	count_cgt<OFF>(s, charOff, nC, nG, nT);
	uint32_t nA = charOff - nC - nG - nT;
	if(sideNum == e.zSide && charOff > e.zChar) nA--;
	out[0] = nA + s.occ[0] + e.fchr[0];
	out[1] = nC + s.occ[1] + e.fchr[1];
	out[2] = nG + s.occ[2] + e.fchr[2];
	out[3] = nT + s.occ[3] + e.fchr[3];
}

// Task = (read, strand); the lane walks through that strand's seeds one after another, so the per-read
// loads (offsets, interval, packed words) are paid once per strand instead of once per seed.  With the extended
// seed table a seed is only a table lookup plus L - K steps, and with one task per seed the refill chain (task id ->
// offsets -> packed words -> table -> first side) had become the bulk of the kernel.
template <typename OFF>
__global__ void __launch_bounds__(256) k_seed_search3(DevIndex<OFF> ix, const uint64_t *packed, const uint32_t *nmask,
                                                      const uint64_t *roff, uint64_t nReads, int seedLen, int maxSeeds,
                                                      int nofw, int norc, const int32_t *interval, const int32_t *offset,
                                                      uint64_t *out, int32_t *nseedsOut, unsigned long long *next,
                                                      unsigned long long *cnt, const uint8_t *actv) {
	// actv != nullptr: only reads with actv[rd] != 0 are searched (their output slots are rewritten; the others stay untouched)
	constexpr uint32_t BL = SideGeom<OFF>::BWT_LEN;
	const unsigned FULL = 0xffffffffu;
	const int lane = threadIdx.x & 31;
	const uint64_t total = nReads * 2;
	const DevEbwt<OFF> &fw = ix.fw;
	const DevEbwt<OFF> &bw = ix.bw;
	const int ftabLen = fw.ftabChars;
	bool haveTask = false, exhausted = false, active = false;
	uint64_t topf = 0, botf = 0, topb = 0, botb = 0, bits = 0, wb = 0;
	uint64_t *o = nullptr, *obase = nullptr;
	int sl = 0, step = 0, k = 0, nseeds = 0, per = 1, off0 = 0, len = 0, strand = 0;
	unsigned nside = 0;
	for(;;) {
		const unsigned need = __ballot_sync(FULL, !haveTask && !exhausted);
		if(need && (__popc(need) >= REFILL_MIN || __ballot_sync(FULL, haveTask) == 0)) {
			unsigned long long base = 0;
			const int leader = __ffs(need) - 1;
			if(lane == leader) base = atomicAdd(next, (unsigned long long)__popc(need));
			base = __shfl_sync(FULL, base, leader);
			if(!haveTask && !exhausted) {
				const uint64_t t = base + (unsigned)__popc(need & ((1u << lane) - 1u));
				if(t >= total) exhausted = true;
				else if(actv && !actv[t >> 1]) { }               // not requested: take another task next round
				else {
					const uint64_t rd = t >> 1;
					strand = (int)(t & 1);
					const uint64_t r0 = roff[rd];
					len = (int)(roff[rd + 1] - r0);
					per = interval[rd]; off0 = offset[rd];
					nseeds = 1;                                       // instantiateSeeds (aligner_seed.cpp:523-526)
					if(len - off0 > seedLen) nseeds += (len - off0 - seedLen) / per;
					if(strand == 0 && nseedsOut) nseedsOut[rd] = nseeds;
					sl = seedLen < len ? seedLen : len;
					wb = (r0 >> 5) + rd;
					obase = out + (rd * 2ull + strand) * (uint64_t)maxSeeds * 4;
					k = 0; haveTask = true; active = false;
				}
			}
		}
		if(__ballot_sync(FULL, haveTask) == 0) {
			if(__all_sync(FULL, exhausted)) break;
			continue;
		}
		// ---- seed set-up for the lanes between seeds
		if(haveTask && !active) {
			if(k >= maxSeeds) haveTask = false;
			else {
				o = obase + (uint64_t)k * 4;
				reinterpret_cast<uint4 *>(o)[0] = make_uint4(0, 0, 0, 0);
				reinterpret_cast<uint4 *>(o)[1] = make_uint4(0, 0, 0, 0);
				const int depth = k * per + off0;
				bool ok = k < nseeds && !((strand == 0 && nofw) || (strand == 1 && norc)) && depth + sl <= len && sl >= 1;
				if(ok) {
					const int w = depth >> 5, sh = depth & 31;
					const bool two = sh + sl > 32;
					const uint64_t p0 = packed[wb + w], p1 = two ? packed[wb + w + 1] : 0;
					const uint64_t n0 = nmask[wb + w], n1 = two ? nmask[wb + w + 1] : 0;
					const uint64_t m2 = sl == 32 ? ~0ull : ((1ull << (2 * sl)) - 1);
					bits = (sh ? ((p0 >> (2 * sh)) | (p1 << (64 - 2 * sh))) : p0) & m2;
					const uint64_t nb = ((n0 | (n1 << 32)) >> sh) & (sl == 32 ? 0xffffffffull : ((1ull << sl) - 1));
					if(nb) ok = false;                               // exact seeds cannot absorb an N (aligner_seed.cpp:326-352)
					if(strand == 1) bits = rev_pairs(bits, sl) ^ m2;   // reverse complement of the window
				}
				if(ok) {
					if(ix.ktab != nullptr && ix.ktabChars <= sl) {
						const OFF *e3 = ix.ktab + 3ull * (bits >> (2 * (sl - ix.ktabChars)));
						topf = e3[0]; botf = e3[1]; topb = e3[2]; botb = topb + (botf - topf);
						if(botf <= topf) ok = false;
						step = ix.ktabChars;
					} else if(ftabLen > 1 && ftabLen <= sl) {
						const uint64_t top20 = bits >> (2 * (sl - ftabLen));
						const uint64_t fwi = rev_pairs(top20, ftabLen), bwi = top20;
						topf = ftab_hi<OFF>(fw, fwi); botf = ftab_lo<OFF>(fw, fwi + 1);
						if(botf <= topf) ok = false;
						else if(bw.ebwt != nullptr) { topb = ftab_hi<OFF>(bw, bwi); botb = topb + (botf - topf); }
						else { topb = botb = 0; }
						step = ftabLen;
					} else {
						const int c = (int)((bits >> (2 * (sl - 1))) & 3);
						topf = topb = fw.fchr[c]; botf = botb = fw.fchr[c + 1];
						if(botf <= topf) ok = false;
						step = 1;
					}
				}
				if(ok) {
					if(step >= sl) { o[0] = topf; o[1] = botf; o[2] = topb; o[3] = botb; }
					else active = true;
				}
				k++;
				// the remaining slots of this strand (k >= nseeds) only need their zero fill: finish them in this pass
				if(!active && k >= nseeds) {
					for(; k < maxSeeds; k++) {
						uint64_t *z = obase + (uint64_t)k * 4;
						reinterpret_cast<uint4 *>(z)[0] = make_uint4(0, 0, 0, 0);
						reinterpret_cast<uint4 *>(z)[1] = make_uint4(0, 0, 0, 0);
					}
					haveTask = false;
				}
			}
		}
		// ---- one LF step for the lanes inside a seed
		if(active) {
			const int c = (int)((bits >> (2 * (sl - step - 1))) & 3);
			const uint64_t sideT = topf / BL, sideB = botf / BL;
			const uint32_t offT = (uint32_t)(topf - sideT * BL), offB = (uint32_t)(botf - sideB * BL);
			nside += (botf - topf > 1) ? 2 : 1;                     // algorithmic count (mapBiLFEx = 2, mapLF1 = 1)
			uint64_t tt[4], bb[4];
			SideRegs<OFF> s;
			load_side<OFF>(fw.ebwt, sideT, s);
			rank4_loaded<OFF>(fw, s, sideT, offT, tt);
			if(sideB != sideT) load_side<OFF>(fw.ebwt, sideB, s);
			rank4_loaded<OFF>(fw, s, sideB, offB, bb);
			const uint64_t w0 = bb[0] - tt[0], w1 = bb[1] - tt[1], w2 = bb[2] - tt[2];
			const uint64_t tp = topb + (c > 0 ? w0 : 0) + (c > 1 ? w1 : 0) + (c > 2 ? w2 : 0);
			const uint64_t nt = c == 0 ? tt[0] : (c == 1 ? tt[1] : (c == 2 ? tt[2] : tt[3]));
			const uint64_t nb = c == 0 ? bb[0] : (c == 1 ? bb[1] : (c == 2 ? bb[2] : bb[3]));
			if(nb <= nt) {
				active = false;
			} else {
				topf = nt; botf = nb; topb = tp; botb = tp + (nb - nt);
				if(++step == sl) { o[0] = topf; o[1] = botf; o[2] = topb; o[3] = botb; active = false; }
			}
		}
	}
	if(cnt && nside) atomicAdd(cnt, (unsigned long long)nside);
}

template <typename OFF>
void launch_seed_search2(const DevIndex<OFF> &ix, const uint8_t *seq, const uint64_t *roff, uint64_t nReads, int maxLen,
                         int seedLen, int maxSeeds, int nofw, int norc, const int32_t *interval, const int32_t *offset,
                         uint64_t *out, int32_t *nseeds, uint64_t *packed, uint32_t *nmask, unsigned long long *next,
                         int numSMs, cudaStream_t st, unsigned long long *cnt) {
	if(nReads == 0) return;
	(void)seq; (void)maxLen;          // reads arrive packed (launch_pack_reads)
	cudaMemsetAsync(next, 0, sizeof(unsigned long long), st);
	// persistent grid: exactly as many blocks as can be resident (no second wave, no tail)
	int perSM = 4;
	cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, k_seed_search3<OFF>, 256, 0);
	if(perSM < 1) perSM = 1;
	k_seed_search3<OFF><<<(unsigned)(numSMs * perSM), 256, 0, st>>>(ix, packed, nmask, roff, nReads, seedLen, maxSeeds, nofw, norc,
	                                                              interval, offset, out, nseeds, next, cnt, nullptr);
}
// the same over the reads flagged in actv[] (re-seeding rounds of the exact engine, csrc/xengine.cu)
template <typename OFF>
void launch_seed_search_active(const DevIndex<OFF> &ix, const uint64_t *roff, uint64_t nReads, int seedLen, int maxSeeds,
                               const int32_t *interval, const int32_t *offset, const uint8_t *actv, uint64_t *out, int32_t *nseeds,
                               const uint64_t *packed, const uint32_t *nmask, unsigned long long *next, int numSMs, cudaStream_t st) {
	if(nReads == 0) return;
	cudaMemsetAsync(next, 0, sizeof(unsigned long long), st);
	int perSM = 4;
	cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, k_seed_search3<OFF>, 256, 0);
	if(perSM < 1) perSM = 1;
	uint64_t blocks = (uint64_t)numSMs * perSM, want = (nReads * 2 + 255) / 256;
	if(want < blocks) blocks = want ? want : 1;
	k_seed_search3<OFF><<<(unsigned)blocks, 256, 0, st>>>(ix, packed, nmask, roff, nReads, seedLen, maxSeeds, 0, 0, interval, offset, out, nseeds, next, nullptr, actv);
}
template void launch_seed_search_active<uint32_t>(const DevIndex<uint32_t> &, const uint64_t *, uint64_t, int, int, const int32_t *, const int32_t *, const uint8_t *, uint64_t *, int32_t *, const uint64_t *, const uint32_t *, unsigned long long *, int, cudaStream_t);
template void launch_seed_search_active<uint64_t>(const DevIndex<uint64_t> &, const uint64_t *, uint64_t, int, int, const int32_t *, const int32_t *, const uint8_t *, uint64_t *, int32_t *, const uint64_t *, const uint32_t *, unsigned long long *, int, cudaStream_t);
template void launch_seed_search2<uint32_t>(const DevIndex<uint32_t> &, const uint8_t *, const uint64_t *, uint64_t, int, int, int, int, int, const int32_t *, const int32_t *, uint64_t *, int32_t *, uint64_t *, uint32_t *, unsigned long long *, int, cudaStream_t, unsigned long long *);
template void launch_seed_search2<uint64_t>(const DevIndex<uint64_t> &, const uint8_t *, const uint64_t *, uint64_t, int, int, int, int, int, const int32_t *, const int32_t *, uint64_t *, int32_t *, uint64_t *, uint32_t *, unsigned long long *, int, cudaStream_t, unsigned long long *);

// ----------------------------------------------------------------------------------------
// Extended seed table (include/bt2g.h: bt2g_build_seed_table): one thread per K-mer replays the first K
// characters of k_seed_search3's chain: ftab lookup for the first ftabChars, then K - ftabChars
// bidirectional LF steps.  Entry index = the K characters in the order the search consumes them,
// first character in the most significant pair.
template <typename OFF>
__global__ void k_build_ktab(DevIndex<OFF> ix, int K, OFF *out) {
	constexpr uint32_t BL = SideGeom<OFF>::BWT_LEN;
	const uint64_t x = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if(x >> (2 * K)) return;
	const DevEbwt<OFF> &fw = ix.fw;
	const DevEbwt<OFF> &bw = ix.bw;
	const int F = fw.ftabChars;
	OFF *o = out + 3ull * x;
	o[0] = 0; o[1] = 0; o[2] = 0;
	const uint64_t top20 = x >> (2 * (K - F));
	const uint64_t fwi = rev_pairs(top20, F), bwi = top20;
	uint64_t topf = ftab_hi<OFF>(fw, fwi), botf = ftab_lo<OFF>(fw, fwi + 1);
	if(botf <= topf) return;
	uint64_t topb = ftab_hi<OFF>(bw, bwi);
	for(int step = F; step < K; step++) {
		const int c = (int)((x >> (2 * (K - step - 1))) & 3);
		const uint64_t sideT = topf / BL, sideB = botf / BL;
		const uint32_t offT = (uint32_t)(topf - sideT * BL), offB = (uint32_t)(botf - sideB * BL);
		uint64_t tt[4], bb[4];
		SideRegs<OFF> s;
		load_side<OFF>(fw.ebwt, sideT, s);
		rank4_loaded<OFF>(fw, s, sideT, offT, tt);
		if(sideB != sideT) load_side<OFF>(fw.ebwt, sideB, s);
		rank4_loaded<OFF>(fw, s, sideB, offB, bb);
		const uint64_t w0 = bb[0] - tt[0], w1 = bb[1] - tt[1], w2 = bb[2] - tt[2];
		const uint64_t tp = topb + (c > 0 ? w0 : 0) + (c > 1 ? w1 : 0) + (c > 2 ? w2 : 0);
		const uint64_t nt = c == 0 ? tt[0] : (c == 1 ? tt[1] : (c == 2 ? tt[2] : tt[3]));
		const uint64_t nb = c == 0 ? bb[0] : (c == 1 ? bb[1] : (c == 2 ? bb[2] : bb[3]));
		if(nb <= nt) return;
		topf = nt; botf = nb; topb = tp;
	}
	o[0] = (OFF)topf; o[1] = (OFF)botf; o[2] = (OFF)topb;
}

template <typename OFF>
void launch_build_ktab(const DevIndex<OFF> &ix, int K, OFF *out, cudaStream_t st) {
	const uint64_t n = 1ull << (2 * K);
	k_build_ktab<OFF><<<(unsigned)((n + 255) / 256), 256, 0, st>>>(ix, K, out);
}
template void launch_build_ktab<uint32_t>(const DevIndex<uint32_t> &, int, uint32_t *, cudaStream_t);
template void launch_build_ktab<uint64_t>(const DevIndex<uint64_t> &, int, uint64_t *, cudaStream_t);

// ----------------------------------------------------------------------------------------
// Denser SA sample (include/bt2g.h: bt2g_build_dense_sa): one thread per sampled row walks to the index's own
// sample (Ebwt::getOffset) and records the offset.
template <typename OFF>
__global__ void k_build_dense_sa(DevIndex<OFF> ix, int rate, uint64_t entries, OFF *out) {
	const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if(i >= entries) return;
	DevIndex<OFF> base = ix;
	base.saOffs = ix.offs; base.saRate = ix.offRate;            // always walk against the index's own sample
	unsigned nside = 0;
	const uint64_t row = i << rate;
	out[i] = row < ix.fw.len + 1 ? (OFF)get_offset<OFF>(base, row, nside) : (OFF)0;
}

template <typename OFF>
void launch_build_dense_sa(const DevIndex<OFF> &ix, int rate, OFF *out, cudaStream_t st) {
	const uint64_t entries = ((ix.fw.len + 1) + ((1ull << rate) - 1)) >> rate;
	if(entries == 0) return;
	k_build_dense_sa<OFF><<<(unsigned)((entries + 255) / 256), 256, 0, st>>>(ix, rate, entries, out);
}
template void launch_build_dense_sa<uint32_t>(const DevIndex<uint32_t> &, int, uint32_t *, cudaStream_t);
template void launch_build_dense_sa<uint64_t>(const DevIndex<uint64_t> &, int, uint64_t *, cudaStream_t);

// ----------------------------------------------------------------------------------------
// K1' v2: exact end-to-end sweep (SeedAligner::exactSweep, aligner_seed.cpp:856-970) with packed
// reads, single-character ranks, one uniform LF step and persistent lanes.  Task = (read, strand).
// ----------------------------------------------------------------------------------------
__device__ __forceinline__ int packed_char(const uint64_t *pk, const uint32_t *nm, uint64_t wb, int pos) {
	const int w = pos >> 5, b = pos & 31;
	if((nm[wb + w] >> b) & 1u) return 4;
	return (int)((pk[wb + w] >> (2 * b)) & 3);
}

// occurrences of nucleotide c among the first charOff characters of a loaded side
template <typename OFF>
__device__ __forceinline__ uint32_t count_one(const SideRegs<OFF> &s, uint32_t charOff, int c) {
	const uint64_t M = 0x5555555555555555ull, pat = (uint64_t)c * M;
	uint32_t n = 0;
#pragma unroll
	for(uint32_t i = 0; i < SideGeom<OFF>::WORDS; i++) {
		int k = (int)charOff - (int)(i * 32);
		k = k < 0 ? 0 : (k > 32 ? 32 : k);
		const uint64_t mask = (k == 32) ? M : (((1ull << (2 * k)) - 1) & M);
		const uint64_t z = ~(s.w[i] ^ pat);
		n += __popcll(z & (z >> 1) & mask);
	}
	return n;
}

template <typename OFF>
__device__ __forceinline__ uint64_t rank1_loaded(const DevEbwt<OFF> &e, const SideRegs<OFF> &s, uint64_t sideNum, uint32_t charOff, int c) {
	uint32_t n = count_one<OFF>(s, charOff, c);
	if(c == 0 && sideNum == e.zSide && charOff > e.zChar) n--;
	const uint64_t oc = c == 0 ? s.occ[0] : (c == 1 ? s.occ[1] : (c == 2 ? s.occ[2] : s.occ[3]));
	return n + oc + e.fchr[c];
}

template <typename OFF>
__global__ void __launch_bounds__(256) k_exact_sweep2(DevIndex<OFF> ix, const uint64_t *packed, const uint32_t *nmask,
                                                      const uint64_t *roff, uint64_t nReads, int nofw, int norc,
                                                      uint8_t *mine, uint64_t *ee, unsigned long long *next, unsigned long long *cnt,
                                                      int flags) {
	// flags bit 0, eeOnly (the pipeline): only the exact end-to-end range is wanted, so the search stops at the first failed
	// extension (mine = 1 then means "at least one edit") and may start from the extended seed table.
	// flags bit 1, text (the exact engine): once the range is ONE row the sweep continues in the joined text (ix.refBuf): a
	// single row's LF steps yield the text characters to the left of the occurrence, so the rest of the stretch is compared
	// with the text at the occurrence's joined offset; an end-to-end range found that way is returned as that offset with
	// BT2G_ROW_IS_OFFSET set (the engine resolves rows to offsets anyway; csrc/xengine.cu: DevSvc::resolve).
	const int eeOnly = flags & 1;
	const bool text = (flags & 2) != 0 && ix.refBuf != nullptr;
	constexpr uint32_t BL = SideGeom<OFF>::BWT_LEN;
	const unsigned FULL = 0xffffffffu;
	const int lane = threadIdx.x & 31;
	const uint64_t total = nReads * 2;
	const DevEbwt<OFF> &e = ix.fw;
	const int ftabLen = e.ftabChars;
	const int mineMax = 2;
	bool active = false, exhausted = false, doInit = true;
	uint64_t top = 0, bot = 0, wb = 0, task = 0;
	int len = 0, dep = 0, nedit = 0, strand = 0;
	int cacheW = -1; uint64_t cacheP = 0; uint32_t cacheM = 0;
	unsigned nside = 0;
	for(;;) {
		const unsigned need = __ballot_sync(FULL, !active && !exhausted);
		// refill in batches: the refill path is a chain of dependent loads that stalls the whole warp
		if(need && (__popc(need) >= REFILL_MIN || __ballot_sync(FULL, active) == 0)) {
			unsigned long long base = 0;
			const int leader = __ffs(need) - 1;
			if(lane == leader) base = atomicAdd(next, (unsigned long long)__popc(need));
			base = __shfl_sync(FULL, base, leader);
			if(!active && !exhausted) {
				cacheW = -1;
				task = base + (unsigned)__popc(need & ((1u << lane) - 1u));
				if(task >= total) exhausted = true;
				else {
					const uint64_t rd = task >> 1;
					strand = (int)(task & 1);
					if((strand == 0 && nofw) || (strand == 1 && norc)) {
						mine[task] = 0; ee[rd * 4 + strand * 2] = 0; ee[rd * 4 + strand * 2 + 1] = 0;
					} else {
						const uint64_t r0 = roff[rd];
						len = (int)(roff[rd + 1] - r0);
						wb = (r0 >> 5) + rd;
						dep = 0; nedit = 0; doInit = true; top = bot = 0;
						active = true;
						if(len <= 0) { mine[task] = 0; ee[rd * 4 + strand * 2] = 0; ee[rd * 4 + strand * 2 + 1] = 0; active = false; }
					}
				}
			}
		}
		if(__ballot_sync(FULL, active) == 0) {
			if(__all_sync(FULL, exhausted)) break;
			continue;
		}
		if(active) {
			bool done = false;
			// character of the strand-oriented read at position p: fw -> read[p]; rc -> comp(read[len-1-p])
			// the packed word holding the character is kept in registers: the sweep walks the read monotonically, so it
			// changes once every 32 characters
			auto rawchr = [&](int pos) -> int {
				const int w = pos >> 5, b = pos & 31;
				if(w != cacheW) { cacheW = w; cacheP = packed[wb + w]; cacheM = nmask[wb + w]; }
				if((cacheM >> b) & 1u) return 4;
				return (int)((cacheP >> (2 * b)) & 3);
			};
			auto chr = [&](int p) -> int {
				if(strand == 0) return rawchr(p);
				const int c = rawchr(len - 1 - p);
				return c > 3 ? 4 : 3 - c;
			};
			bool stepNow = true;
			if(doInit) {
				// exactSweepInit (aligner_seed.cpp:760-800)
				const int left = len - dep;
				bool doFtab = ftabLen > 1 && left >= ftabLen;
				uint64_t fi = 0;
				bool viaTable = false;
				if(eeOnly && ix.ktab != nullptr && left >= ix.ktabChars) {
					const int K = ix.ktabChars;
					uint64_t x = 0;
					bool clean = true;
					for(int i = 0; i < K; i++) {
						const int c = chr(left - 1 - i);
						if(c > 3) { clean = false; break; }
						x = (x << 2) | (uint64_t)c;
					}
					if(clean) {
						const OFF *e3 = ix.ktab + 3ull * x;
						top = e3[0]; bot = e3[1]; dep += K;
						viaTable = true; doFtab = false;
					}
				}
				if(viaTable) {
				} else if(doFtab) {
					for(int i = 0; i < ftabLen; i++) {
						const int c = chr(left - ftabLen + i);
						if(c > 3) { doFtab = false; break; }
						fi = (fi << 2) | (uint64_t)c;
					}
				}
				if(!viaTable) top = bot = 0;
				if(viaTable) {
				} else if(doFtab) { top = ftab_hi<OFF>(e, fi); bot = ftab_lo<OFF>(e, fi + 1); dep += ftabLen; }
				else {
					const int c = chr(len - dep - 1);
					if(c < 4) { top = e.fchr[c]; bot = e.fchr[c + 1]; }
					dep++;
				}
				if(bot <= top) {
					nedit++;
					if(nedit >= mineMax || eeOnly) done = true;
					stepNow = false;                    // the reference `continue`s: re-init from the new depth
				} else doInit = false;
			}
			if(stepNow && !done && dep < len && text && bot - top == 1) {
				unsigned ns2 = 0;
				int64_t b = (int64_t)get_offset<OFF>(ix, top, ns2) - 1;
				nside += ns2;
				bool mism = false;
				while(dep < len) {
					const int c = chr(len - dep - 1);
					if(c > 3 || b < 0 || (int)((__ldg(ix.refBuf + (b >> 2)) >> ((b & 3) << 1)) & 3) != c) { mism = true; break; }
					b--; dep++;
				}
				if(mism) {
					top = bot = 0;
					nedit++;
					if(nedit >= mineMax || eeOnly) done = true;
					doInit = true;
					dep++;
				} else { top = BT2G_ROW_IS_OFFSET | (uint64_t)(b + 1); bot = top + 1; }
			} else if(stepNow && !done && dep < len) {
				const int c = chr(len - dep - 1);
				if(c > 3) { top = bot = 0; }
				else {
					nside += (bot - top > 1) ? 2 : 1;
					const uint64_t sideT = top / BL, sideB = bot / BL;
					SideRegs<OFF> s;
					load_side<OFF>(e.ebwt, sideT, s);
					const uint64_t nt = rank1_loaded<OFF>(e, s, sideT, (uint32_t)(top - sideT * BL), c);
					if(sideB != sideT) load_side<OFF>(e.ebwt, sideB, s);
					const uint64_t nb = rank1_loaded<OFF>(e, s, sideB, (uint32_t)(bot - sideB * BL), c);
					top = nt; bot = nb;
					if(bot <= top) { top = bot = 0; }
				}
				if(bot <= top) {
					nedit++;
					if(nedit >= mineMax || eeOnly) done = true;
					doInit = true;
				}
				dep++;
			}
			if(done || dep >= len) {
				const uint64_t rd = task >> 1;
				mine[task] = (uint8_t)nedit;
				uint64_t *eo = ee + rd * 4 + strand * 2;
				if(!done && nedit == 0 && bot > top) { eo[0] = top; eo[1] = bot; } else { eo[0] = eo[1] = 0; }
				active = false;
			}
		}
	}
	if(cnt && nside) atomicAdd(cnt, (unsigned long long)nside);
}

template <typename OFF>
void launch_exact_sweep2(const DevIndex<OFF> &ix, const uint64_t *roff, uint64_t nReads, int nofw, int norc,
                         uint8_t *mine, uint64_t *ee, const uint64_t *packed, const uint32_t *nmask, unsigned long long *next,
                         int numSMs, cudaStream_t st, unsigned long long *cnt, int flags) {
	if(nReads == 0) return;
	cudaMemsetAsync(next, 0, sizeof(unsigned long long), st);
	int perSM = 4;
	cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, k_exact_sweep2<OFF>, 256, 0);
	if(perSM < 1) perSM = 1;
	k_exact_sweep2<OFF><<<(unsigned)(numSMs * perSM), 256, 0, st>>>(ix, packed, nmask, roff, nReads, nofw, norc, mine, ee, next, cnt, flags);
}
template void launch_exact_sweep2<uint32_t>(const DevIndex<uint32_t> &, const uint64_t *, uint64_t, int, int, uint8_t *, uint64_t *, const uint64_t *, const uint32_t *, unsigned long long *, int, cudaStream_t, unsigned long long *, int);
template void launch_exact_sweep2<uint64_t>(const DevIndex<uint64_t> &, const uint64_t *, uint64_t, int, int, uint8_t *, uint64_t *, const uint64_t *, const uint32_t *, unsigned long long *, int, cudaStream_t, unsigned long long *, int);

void launch_pack_reads(const uint8_t *seq, const uint64_t *roff, uint64_t nReads, int maxLen, uint64_t *packed, uint32_t *nmask, cudaStream_t st) {
	if(nReads == 0) return;
	const int maxWords = (maxLen + 31) / 32;
	const uint64_t nw = nReads * (uint64_t)maxWords;
	k_pack_reads<<<(unsigned)((nw + 255) / 256), 256, 0, st>>>(seq, roff, nReads, maxWords, packed, nmask);
}

// ----------------------------------------------------------------------------------------
// K2 v2: SA-offset resolution over a DENSE row list with persistent lanes (v1 ran one thread per
// padded slot: 2.8 of 32 lanes active).  The row count lives on the device (written by the
// collect stage), so no host round trip is needed to size the launch.
// ----------------------------------------------------------------------------------------
template <typename OFF>
__global__ void __launch_bounds__(256) k_resolve2(DevIndex<OFF> ix, const uint64_t *rows, const uint32_t *hitlen, uint64_t nHost,
                                                  const uint32_t *nDev, int rejectStraddle, uint64_t *joined, uint64_t *tidx,
                                                  uint64_t *textoff, uint64_t *tlen, uint8_t *flags, unsigned long long *next,
                                                  unsigned long long *cnt) {
	const unsigned FULL = 0xffffffffu;
	const int lane = threadIdx.x & 31;
	const uint64_t total = nDev ? (uint64_t)*nDev : nHost;
	const uint64_t rateMask = (1ull << ix.saRate) - 1;
	bool active = false, exhausted = false;
	uint64_t row = 0, jumps = 0, task = 0;
	unsigned nside = 0;
	for(;;) {
		const unsigned need = __ballot_sync(FULL, !active && !exhausted);
		if(need && (__popc(need) >= REFILL_MIN || __ballot_sync(FULL, active) == 0)) {
			unsigned long long base = 0;
			const int leader = __ffs(need) - 1;
			if(lane == leader) base = atomicAdd(next, (unsigned long long)__popc(need));
			base = __shfl_sync(FULL, base, leader);
			if(!active && !exhausted) {
				task = base + (unsigned)__popc(need & ((1u << lane) - 1u));
				if(task >= total) exhausted = true;
				else {
					row = rows[task]; jumps = 0;
					if(row == BT2G_OFFMASK) { if(flags) flags[task] = 4; }
					else active = true;
				}
			}
		}
		if(__ballot_sync(FULL, active) == 0) {
			if(__all_sync(FULL, exhausted)) break;
			continue;
		}
		if(active) {
			// Ebwt::getOffset (bt2_idx.cpp:150-171), one LF step per iteration
			bool fin = false; uint64_t off = 0;
			if(row == ix.fw.zOff) { fin = true; off = jumps; }
			else if((row & rateMask) == 0) { fin = true; off = jumps + (uint64_t)__ldg(ix.saOffs + (row >> ix.saRate)); }
			else { int c; row = lf_step<OFF>(ix.fw, row, c); jumps++; nside++; }
			if(fin) {
				if(joined) joined[task] = off;
				if(tidx || textoff || tlen || flags) {
					uint64_t ti, to, tl; bool st;
					const bool ok = joined_to_text<OFF>(ix, hitlen ? hitlen[task] : 1, off, rejectStraddle != 0, ti, to, tl, st);
					if(tidx) tidx[task] = ti;
					if(textoff) textoff[task] = to;
					if(tlen) tlen[task] = tl;
					if(flags) flags[task] = (uint8_t)((st ? 1 : 0) | (ok ? 0 : 2));
				}
				active = false;
			}
		}
	}
	if(cnt && nside) atomicAdd(cnt, (unsigned long long)nside);
}

template <typename OFF>
void launch_resolve2(const DevIndex<OFF> &ix, const uint64_t *rows, const uint32_t *hitlen, uint64_t nHost, const uint32_t *nDev,
                     int rej, uint64_t *joined, uint64_t *tidx, uint64_t *textoff, uint64_t *tlen, uint8_t *flags,
                     unsigned long long *next, int numSMs, cudaStream_t st, unsigned long long *cnt) {
	if(nHost == 0 && nDev == nullptr) return;
	cudaMemsetAsync(next, 0, sizeof(unsigned long long), st);
	int perSM = 4;
	cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, k_resolve2<OFF>, 256, 0);
	if(perSM < 1) perSM = 1;
	k_resolve2<OFF><<<(unsigned)(numSMs * perSM), 256, 0, st>>>(ix, rows, hitlen, nHost, nDev, rej, joined, tidx, textoff, tlen, flags, next, cnt);
}
template void launch_resolve2<uint32_t>(const DevIndex<uint32_t> &, const uint64_t *, const uint32_t *, uint64_t, const uint32_t *, int, uint64_t *, uint64_t *, uint64_t *, uint64_t *, uint8_t *, unsigned long long *, int, cudaStream_t, unsigned long long *);
template void launch_resolve2<uint64_t>(const DevIndex<uint64_t> &, const uint64_t *, const uint32_t *, uint64_t, const uint32_t *, int, uint64_t *, uint64_t *, uint64_t *, uint64_t *, uint8_t *, unsigned long long *, int, cudaStream_t, unsigned long long *);
