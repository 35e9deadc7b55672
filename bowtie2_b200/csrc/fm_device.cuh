// fm_device.cuh -- device-side FM-index primitives for sm_100a.
//
// These are re-designs, not translations: the reference walks a side with 64-bit XOR/shift
// popcounts plus a 4x4x256 LUT tail (bt2_idx.h:518-530, :1933-2080, ccnt_lut.cpp).  Here one
// thread pulls the whole 64 B (.bt2) / 128 B (.bt2l) side with 128-bit loads (two / four 32 B
// sectors of one cache line, so one rank query = one line of HBM traffic) and counts three of
// the four nucleotides with masked __popcll on bit-plane combinations; the fourth count is
// char_off minus the others.  No lookup table, no byte loop, no divergence on char_off.
#pragma once
#include "bt2g_internal.h"

#define BT2G_OFFMASK (~(uint64_t)0)

template <typename OFF> struct SideGeom;
template <> struct SideGeom<uint32_t> {
	static constexpr uint32_t SIDE_SZ = 64, BWT_SZ = 48, BWT_LEN = 192, WORDS = 6, VECS = 4;
};
template <> struct SideGeom<uint64_t> {
	static constexpr uint32_t SIDE_SZ = 128, BWT_SZ = 96, BWT_LEN = 384, WORDS = 12, VECS = 8;
};

// One side in registers: WORDS 64-bit BWT words followed by the four Occ counters.
template <typename OFF>
struct SideRegs {
	uint64_t w[SideGeom<OFF>::WORDS];
	uint64_t occ[4];
};

// One 32-byte sector per instruction (sm_100 256-bit loads), read-only path, and an explicit
// L2 fetch granule equal to the side: tools/gather_bench.cu measured on B200 (random gathers over
// 1 GB) 4 x LDG.128 nc/no_allocate = 0.70 TB/s with 128 B of DRAM traffic per 64 B side, while
// 2 x LDG.256 with .L2::64B = 1.39 TB/s with 64 B of DRAM traffic per side.
__device__ __forceinline__ void ldg_sector(const uint8_t *p, uint64_t &a, uint64_t &b, uint64_t &c, uint64_t &d) {
	asm volatile("ld.global.nc.L1::no_allocate.L2::64B.v4.u64 {%0,%1,%2,%3}, [%4];"
	             : "=l"(a), "=l"(b), "=l"(c), "=l"(d) : "l"(p));
}
__device__ __forceinline__ void ldg_sector128(const uint8_t *p, uint64_t &a, uint64_t &b, uint64_t &c, uint64_t &d) {
	asm volatile("ld.global.nc.L1::no_allocate.L2::128B.v4.u64 {%0,%1,%2,%3}, [%4];"
	             : "=l"(a), "=l"(b), "=l"(c), "=l"(d) : "l"(p));
}

template <typename OFF>
__device__ __forceinline__ void load_side(const uint8_t *ebwt, uint64_t sideNum, SideRegs<OFF> &s);

template <>
__device__ __forceinline__ void load_side<uint32_t>(const uint8_t *ebwt, uint64_t sideNum, SideRegs<uint32_t> &s) {
	const uint8_t *p = ebwt + sideNum * 64;
	uint64_t o0, o1;
	ldg_sector(p, s.w[0], s.w[1], s.w[2], s.w[3]);
	ldg_sector(p + 32, s.w[4], s.w[5], o0, o1);
	s.occ[0] = (uint32_t)o0; s.occ[1] = o0 >> 32; s.occ[2] = (uint32_t)o1; s.occ[3] = o1 >> 32;
}

template <>
__device__ __forceinline__ void load_side<uint64_t>(const uint8_t *ebwt, uint64_t sideNum, SideRegs<uint64_t> &s) {
	const uint8_t *p = ebwt + sideNum * 128;
	ldg_sector128(p, s.w[0], s.w[1], s.w[2], s.w[3]);
	ldg_sector128(p + 32, s.w[4], s.w[5], s.w[6], s.w[7]);
	ldg_sector128(p + 64, s.w[8], s.w[9], s.w[10], s.w[11]);
	ldg_sector128(p + 96, s.occ[0], s.occ[1], s.occ[2], s.occ[3]);
}

// counts of C, G, T among the first charOff characters of the side (A = charOff - sum)
template <typename OFF>
__device__ __forceinline__ void count_cgt(const SideRegs<OFF> &s, uint32_t charOff,
                                          uint32_t &nC, uint32_t &nG, uint32_t &nT) {
	nC = nG = nT = 0;
	const uint64_t M = 0x5555555555555555ull;
#pragma unroll
	for(uint32_t i = 0; i < SideGeom<OFF>::WORDS; i++) {
		int n = (int)charOff - (int)(i * 32);           // characters of this word that count
		n = n < 0 ? 0 : (n > 32 ? 32 : n);
		uint64_t mask = (n == 32) ? M : (((1ull << (2 * n)) - 1) & M);
		uint64_t lo = s.w[i] & mask, hi = (s.w[i] >> 1) & mask;
		nC += __popcll(lo & ~hi);
		nG += __popcll(hi & ~lo);
		nT += __popcll(hi & lo);
	}
}

// Ebwt::countBt2SideEx (bt2_idx.h:1887-1919): all four ranks at `row`.
template <typename OFF>
__device__ __forceinline__ void rank4(const DevEbwt<OFF> &e, uint64_t row, uint64_t out[4]) {
	constexpr uint32_t BL = SideGeom<OFF>::BWT_LEN;
	uint64_t sideNum = row / BL;
	uint32_t charOff = (uint32_t)(row - sideNum * BL);
	SideRegs<OFF> s;
	load_side<OFF>(e.ebwt, sideNum, s);
	uint32_t nC, nG, nT;
	count_cgt<OFF>(s, charOff, nC, nG, nT);
	uint32_t nA = charOff - nC - nG - nT;
	// "$" is stored as an A at row zOff; do not count it (bt2_idx.h:1891-1899)
	if(sideNum == e.zSide && charOff > e.zChar) nA--;
	out[0] = nA + s.occ[0] + e.fchr[0];
	out[1] = nC + s.occ[1] + e.fchr[1];
	out[2] = nG + s.occ[2] + e.fchr[2];
	out[3] = nT + s.occ[3] + e.fchr[3];
}

// rowL + mapLF in one side fetch: returns LF(row) and the BWT char, for the SA walk
// (Ebwt::mapLF(l), bt2_idx.h:2313-2338).  Caller guarantees row != zOff.
template <typename OFF>
__device__ __forceinline__ uint64_t lf_step(const DevEbwt<OFF> &e, uint64_t row, int &cOut) {
	constexpr uint32_t BL = SideGeom<OFF>::BWT_LEN;
	uint64_t sideNum = row / BL;
	uint32_t charOff = (uint32_t)(row - sideNum * BL);
	SideRegs<OFF> s;
	load_side<OFF>(e.ebwt, sideNum, s);
	// character at charOff: select the word without dynamic register indexing
	uint64_t word = 0;
	uint32_t wi = charOff >> 5;
#pragma unroll
	for(uint32_t i = 0; i < SideGeom<OFF>::WORDS; i++) word = (wi == i) ? s.w[i] : word;
	int c = (int)((word >> ((charOff & 31) * 2)) & 3);
	uint32_t nC, nG, nT;
	count_cgt<OFF>(s, charOff, nC, nG, nT);
	uint32_t nA = charOff - nC - nG - nT;
	if(sideNum == e.zSide && charOff > e.zChar) nA--;
	uint32_t n = c == 0 ? nA : (c == 1 ? nC : (c == 2 ? nG : nT));
	uint64_t oc = c == 0 ? s.occ[0] : (c == 1 ? s.occ[1] : (c == 2 ? s.occ[2] : s.occ[3]));
	cOut = c;
	return n + oc + e.fchr[c];
}

// Ebwt::mapLF1(row, l, c) (bt2_idx.h:2420-2443)
template <typename OFF>
__device__ __forceinline__ uint64_t maplf1(const DevEbwt<OFF> &e, uint64_t row, int c) {
	if(row == e.zOff) return BT2G_OFFMASK;
	int cc;
	uint64_t r = lf_step<OFF>(e, row, cc);
	return cc == c ? r : BT2G_OFFMASK;
}

// Ebwt::ftabHi / ftabLo (bt2_idx.h:1428-1554)
template <typename OFF>
__device__ __forceinline__ uint64_t ftab_hi(const DevEbwt<OFF> &e, uint64_t i) {
	OFF v = __ldg(e.ftab + i);
	if((uint64_t)v <= e.len) return v;
	OFF ef = (OFF)(v ^ (OFF)~(OFF)0);
	return __ldg(e.eftab + (uint64_t)ef * 2 + 1);
}
template <typename OFF>
__device__ __forceinline__ uint64_t ftab_lo(const DevEbwt<OFF> &e, uint64_t i) {
	OFF v = __ldg(e.ftab + i);
	if((uint64_t)v <= e.len) return v;
	OFF ef = (OFF)(v ^ (OFF)~(OFF)0);
	return __ldg(e.eftab + (uint64_t)ef * 2);
}

// Ebwt::getOffset(row) (bt2_idx.cpp:150-171) == GroupWalk2S::advanceElement result
// (group_walk.h:517-520): LF-walk until a sampled row or the "$" row.
template <typename OFF>
__device__ __forceinline__ uint64_t get_offset(const DevIndex<OFF> &ix, uint64_t row, unsigned &nside) {
	const uint64_t rateMask = (1ull << ix.saRate) - 1;
	uint64_t jumps = 0;
	for(;;) {
		if(row == ix.fw.zOff) return jumps;
		if((row & rateMask) == 0) return jumps + (uint64_t)__ldg(ix.saOffs + (row >> ix.saRate));
		int c;
		row = lf_step<OFF>(ix.fw, row, c);
		jumps++; nside++;
	}
}

// Ebwt::joinedToTextOff (bt2_idx.cpp:54-124), forward index.  Returns false when rejected.
template <typename OFF>
__device__ __forceinline__ bool joined_to_text(const DevIndex<OFF> &ix, uint64_t qlen, uint64_t off,
                                               bool rejectStraddle, uint64_t &tidx, uint64_t &textoff,
                                               uint64_t &tlen, bool &straddled) {
	uint64_t top = 0, bot = ix.nFrag;
	straddled = false;
	// the reference would spin on an offset outside the joined text (its debug build asserts
	// progress, bt2_idx.cpp:70); a kernel must terminate, so such offsets are rejected
	if(off >= ix.fw.len || ix.nFrag == 0) { tidx = BT2G_OFFMASK; textoff = 0; tlen = 0; return false; }
	for(;;) {
		uint64_t elt = top + ((bot - top) >> 1);
		uint64_t lower = __ldg(ix.rstarts + elt * 3);
		uint64_t upper = (elt == ix.nFrag - 1) ? ix.fw.len : (uint64_t)__ldg(ix.rstarts + (elt + 1) * 3);
		if(lower <= off) {
			if(upper > off) {
				if(off + qlen > upper) {
					straddled = true;
					if(rejectStraddle) { tidx = BT2G_OFFMASK; textoff = 0; tlen = 0; return false; }
				}
				tidx = __ldg(ix.rstarts + elt * 3 + 1);
				textoff = (off - lower) + (uint64_t)__ldg(ix.rstarts + elt * 3 + 2);
				break;
			}
			top = elt;
		} else {
			bot = elt;
		}
	}
	tlen = __ldg(ix.plen + tidx);
	return true;
}

// BitPairReference::getBase (reference.cpp:330-358) with a binary search over the records of
// the target (the reference's getStretch does the same for > 16 records, reference.cpp:470-486).
template <typename OFF>
__device__ __forceinline__ int ref_base(const DevIndex<OFF> &ix, uint64_t tidx, int64_t toff) {
	if(toff < 0 || (uint64_t)toff >= ix.refLens[tidx]) return 4;
	uint64_t lo = ix.refRecOffs[tidx], hi = ix.refRecOffs[tidx + 1];
	// last record whose N-run starts at or before toff
	while(hi - lo > 1) {
		uint64_t mid = lo + ((hi - lo) >> 1);
		if(ix.recCumOff[mid] <= (uint64_t)toff) lo = mid; else hi = mid;
	}
	uint64_t start = ix.recCumOff[lo] + (uint64_t)ix.recOff[lo];
	if((uint64_t)toff < start) return 4;
	uint64_t k = (uint64_t)toff - start;
	if(k >= (uint64_t)ix.recLen[lo]) return 4;
	uint64_t b = ix.recCumUnamb[lo] + k;
	return (ix.refBuf[b >> 2] >> ((b & 3) << 1)) & 3;
}

// ref_base for runs of nearby positions: remembers the unambiguous stretch that held the last position, so that consecutive
// look-ups (ungapped alignment, edit lists) cost one packed-byte load instead of a binary search over the records each
template <typename OFF>
struct RefCursor {
	uint64_t tidx = ~0ull, b0 = 0;
	int64_t s = 0, e = 0;                                // positions [s, e) of reference tidx lie at packed offsets b0 ...
	__device__ __forceinline__ int get(const DevIndex<OFF> &ix, uint64_t t, int64_t toff) {
		if(t == tidx && toff >= s && toff < e) { const uint64_t b = b0 + (uint64_t)(toff - s); return (__ldg(ix.refBuf + (b >> 2)) >> ((b & 3) << 1)) & 3; }
		if(toff < 0 || (uint64_t)toff >= ix.refLens[t]) return 4;
		uint64_t lo = ix.refRecOffs[t], hi = ix.refRecOffs[t + 1];
		while(hi - lo > 1) {
			const uint64_t mid = lo + ((hi - lo) >> 1);
			if(ix.recCumOff[mid] <= (uint64_t)toff) lo = mid; else hi = mid;
		}
		const uint64_t start = ix.recCumOff[lo] + (uint64_t)ix.recOff[lo];
		if((uint64_t)toff < start) return 4;
		const uint64_t k = (uint64_t)toff - start;
		if(k >= (uint64_t)ix.recLen[lo]) return 4;
		tidx = t; s = (int64_t)start; e = (int64_t)(start + (uint64_t)ix.recLen[lo]); b0 = ix.recCumUnamb[lo];
		const uint64_t b = b0 + k;
		return (__ldg(ix.refBuf + (b >> 2)) >> ((b & 3) << 1)) & 3;
	}
};

// A whole reference window [refl, refl+ncol) into out[] (one warp; lane k fills columns k, k+32, ...).
// Fast path: the window lies inside one unambiguous stretch, found once per window instead of once
// per column; otherwise every column goes through ref_base (N runs, reference ends).
template <typename OFF>
__device__ __forceinline__ void ref_window(const DevIndex<OFF> &ix, uint64_t tidx, int64_t refl, int ncol, uint8_t *out, int lane) {
	bool fast = false;
	uint64_t b0 = 0;
	if(refl >= 0 && (uint64_t)(refl + ncol) <= ix.refLens[tidx]) {
		uint64_t lo = ix.refRecOffs[tidx], hi = ix.refRecOffs[tidx + 1];
		while(hi - lo > 1) {
			const uint64_t mid = lo + ((hi - lo) >> 1);
			if(ix.recCumOff[mid] <= (uint64_t)refl) lo = mid; else hi = mid;
		}
		const uint64_t start = ix.recCumOff[lo] + (uint64_t)ix.recOff[lo];
		if((uint64_t)refl >= start && (uint64_t)(refl + ncol) <= start + (uint64_t)ix.recLen[lo]) {
			fast = true;
			b0 = ix.recCumUnamb[lo] + ((uint64_t)refl - start);
		}
	}
	if(fast) {
		for(int k = lane; k < ncol; k += 32) {
			const uint64_t b = b0 + (uint64_t)k;
			out[k] = (uint8_t)((ix.refBuf[b >> 2] >> ((b & 3) << 1)) & 3);
		}
	} else {
		for(int k = lane; k < ncol; k += 32) out[k] = (uint8_t)ref_base<OFF>(ix, tidx, refl + k);
	}
}

// read access helpers: strand 0 = read as given, strand 1 = reverse complement
__device__ __forceinline__ int read_char(const uint8_t *seq, int len, int strand, int pos) {
	if(strand == 0) return seq[pos];
	int c = seq[len - 1 - pos];
	return c > 3 ? 4 : 3 - c;
}

// SwDriver::extend (aligner_sw_driver.cpp:299-484), one direction: how many read positions the range [top, bot) extends
// without an edit and without shrinking (<= 255).  Used by k_extend (fm_kernels.cu) and inline by the exact engine.
template <typename OFF>
__device__ __forceinline__ uint32_t extend_one(const DevEbwt<OFF> &e, uint64_t top, uint64_t bot, const uint8_t *s, int len,
                                               int strand, int i0, int step, int lim) {
	uint32_t n = 0;
	for(int ii = 0; ii < lim; ii++) {
		const int rdc = read_char(s, len, strand, i0 + ii * step);
		if(bot - top > 1) {
			uint64_t t[4], b[4];
			rank4<OFF>(e, top, t);
			rank4<OFF>(e, bot, b);
			const uint64_t orig = bot - top;
			int nonz = -1; bool abort = false;
#pragma unroll
			for(int j = 0; j < 4; j++) {
				if(!abort && b[j] > t[j]) {
					if(nonz >= 0) abort = true;
					else { nonz = j; top = t[j]; bot = b[j]; }
				}
			}
			if(abort || (nonz != rdc && rdc <= 3) || bot - top < orig) break;
		} else {
			int c = -1;
			if(top != e.zOff) top = lf_step<OFF>(e, top, c);
			if(c != rdc && rdc <= 3) break;
			bot = top + 1;
		}
		if(++n == 255) break;
	}
	return n;
}

// The same for a range of ONE row, without the index: LF from row r yields BWT[r] = T[SA[r] - 1], the character of the joined
// text that precedes the suffix (in the mirror index: the one that follows the occurrence), so the walk of a unique seed hit is
// a comparison of the read with the joined text itself -- ix.refBuf, the 2-bit packed reference, holds exactly the joined
// text (every unambiguous base in order; index = joined offset).  `b` = joined offset of the first text character compared,
// `tstep` = -1 (left, forward index) / +1 (right, mirror index).  Off either end of the text the row is the "$" row: LF yields
// no character (c = -1) and does not move, which only a read N survives (bt2_idx.h:2451-2473).
template <typename OFF>
__device__ __forceinline__ uint32_t extend_one_text(const DevIndex<OFF> &ix, int64_t b, int tstep, const uint8_t *s, int len,
                                                    int strand, int i0, int step, int lim) {
	uint32_t n = 0;
	const int64_t tlen = (int64_t)ix.fw.len;
	for(int ii = 0; ii < lim; ii++) {
		const int rdc = read_char(s, len, strand, i0 + ii * step);
		int c = -1;
		if(b >= 0 && b < tlen) { c = (int)((__ldg(ix.refBuf + (b >> 2)) >> ((b & 3) << 1)) & 3); b += tstep; }
		if(c != rdc && rdc <= 3) break;
		if(++n == 255) break;
	}
	return n;
}
// ---- the same comparison 32 characters at a time, over the 2-bit packed read (k_pack_reads: word w of a read holds its bases
// 32w..32w+31, base i at bits 2(i & 31); N mask with the same word structure) and the 2-bit packed joined text.
__device__ __forceinline__ uint64_t swap_rev_pairs(uint64_t x) {       // reverse the order of the 32 2-bit groups of x
	const uint64_t y = __brevll(x);
	return ((y & 0x5555555555555555ull) << 1) | ((y >> 1) & 0x5555555555555555ull);
}
__device__ __forceinline__ uint64_t spread_bits(uint32_t m) {            // bit j -> bit 2j
	uint64_t x = m;
	x = (x | (x << 16)) & 0x0000ffff0000ffffull;
	x = (x | (x << 8)) & 0x00ff00ff00ff00ffull;
	x = (x | (x << 4)) & 0x0f0f0f0f0f0f0f0full;
	x = (x | (x << 2)) & 0x3333333333333333ull;
	x = (x | (x << 1)) & 0x5555555555555555ull;
	return x;
}
// 32 characters of a packed sequence in WALK order (character j of the walk at bits 2j): ascending from p (p, p+1, ...) or
// descending from p (p, p-1, ...); `ok` gets one bit per walk position that lies inside [0, n).  Words are fetched through
// `word(k)` (k >= 0) so that the read (two arrays) and the text (one byte array) share the code.
template <typename F>
__device__ __forceinline__ uint64_t walk_window(F word, int64_t p, bool asc, int64_t n, uint32_t &ok) {
	int64_t q = asc ? p : p - 31;                      // ascending window [q, q + 32)
	int lshift = 0;                                    // groups the window is moved up by when it starts before 0
	if(q < 0) { lshift = (int)(-q); q = 0; }
	uint64_t a = 0;
	if(lshift < 32 && q < n) {
		const int64_t w = q >> 5; const int sh = (int)(q & 31);
		a = word(w) >> (2 * sh);
		if(sh && ((w + 1) << 5) < n) a |= word(w + 1) << (64 - 2 * sh);
		if(lshift) a <<= 2 * lshift;
	}
	// validity of ascending position k of the (unshifted) window [p or p-31 ...): inside [0, n)
	const int64_t q0 = asc ? p : p - 31;
	uint32_t v = 0xffffffffu;
	if(q0 < 0) v = q0 <= -32 ? 0u : (v << (int)(-q0));
	if(q0 + 32 > n) { const int64_t keep = n - q0; v = keep <= 0 ? 0u : (keep >= 32 ? v : (v & ((1u << (int)keep) - 1u))); }
	if(asc) { ok = v; return a; }
	ok = __brev(v);
	return swap_rev_pairs(a);
}
// extend_one_text, word-parallel.  pk / nm: the read's packed words and N-mask words (word 0 = bases 0..31).
template <typename OFF>
__device__ __forceinline__ uint32_t extend_one_text_packed(const DevIndex<OFF> &ix, int64_t b, int tstep, const uint64_t *pk, const uint32_t *nm, int len,
                                                           int strand, int i0, int step, int lim) {
	const int64_t tlen = (int64_t)ix.fw.len;
	const uint64_t *tw = reinterpret_cast<const uint64_t *>(ix.refBuf);
	auto tword = [&](int64_t k) -> uint64_t { return __ldg(tw + k); };
	auto rword = [&](int64_t k) -> uint64_t { return pk[k]; };
	// raw read position and direction of the walk: strand 1 reads the reverse complement
	int64_t rp = strand == 0 ? i0 : len - 1 - i0;
	const bool rasc = strand == 0 ? step > 0 : step < 0;
	const uint64_t comp = strand == 0 ? 0ull : ~0ull;
	int n = 0;
	if(lim > 255) lim = 255;
	while(n < lim) {
		uint32_t okR, okT, okN;
		const uint64_t R = walk_window(rword, rp, rasc, (int64_t)len, okR) ^ comp;
		const uint64_t T = walk_window(tword, b, tstep > 0, tlen, okT);
		// N mask of the read in walk order (one bit per character)
		uint32_t nmk;
		{
			int64_t q = rasc ? rp : rp - 31; int lshift = 0;
			if(q < 0) { lshift = (int)(-q); q = 0; }
			uint32_t a = 0;
			if(lshift < 32 && q < len) {
				const int64_t w = q >> 5; const int sh = (int)(q & 31);
				a = nm[w] >> sh;
				if(sh && ((w + 1) << 5) < len) a |= nm[w + 1] << (32 - sh);
				if(lshift) a <<= lshift;
			}
			nmk = rasc ? a : __brev(a);
			okN = 0;
		}
		(void)okN;
		const uint64_t X = R ^ T;
		const uint64_t neq = (X | (X >> 1)) & 0x5555555555555555ull;
		// a walk position stops the extension when the read character is not N and (the text has no character there or differs)
		const uint64_t stop = (neq | spread_bits(~okT)) & ~spread_bits(nmk);
		const int chunk = lim - n < 32 ? lim - n : 32;
		int first = stop ? (__ffsll((long long)stop) - 1) >> 1 : 32;
		if(first < chunk) { n += first; break; }
		n += chunk;
		rp += rasc ? 32 : -32;
		b += tstep > 0 ? 32 : -32;
		(void)okR;
	}
	return (uint32_t)n;
}

// SwDriver::extend, both directions of one seed hit (range rng = topf, botf, topb, botb of the seed at 5' offset `off` of the
// strand-oriented read): unique hits through the text, the rest through the index
template <typename OFF>
__device__ __forceinline__ void extend_hit(const DevIndex<OFF> &ix, const uint64_t rng[4], const uint8_t *s, int len, bool fw, int off, int sl,
                                           bool left, bool right, uint32_t &nlex, uint32_t &nrex, const uint64_t *pk = nullptr, const uint32_t *nm = nullptr) {
	const int strand = fw ? 0 : 1;
	const int limL = fw ? off : len - sl - off, limR = fw ? len - sl - off : off;
	const int i0L = fw ? off - 1 : len - off - sl - 1, i0R = fw ? sl + off : len - off;
	nlex = nrex = 0;
	const bool unique = ix.extText && ix.refBuf != nullptr && rng[1] - rng[0] == 1;
	int64_t p = 0;
	if(unique && ((left && limL > 0) || (right && limR > 0))) { unsigned ns = 0; p = (int64_t)get_offset<OFF>(ix, rng[0], ns); }
	if(left && limL > 0)
		nlex = !unique ? extend_one<OFF>(ix.fw, rng[0], rng[1], s, len, strand, i0L, -1, limL)
		     : (pk ? extend_one_text_packed<OFF>(ix, p - 1, -1, pk, nm, len, strand, i0L, -1, limL) : extend_one_text<OFF>(ix, p - 1, -1, s, len, strand, i0L, -1, limL));
	if(right && limR > 0 && ix.bw.ebwt != nullptr)
		nrex = !unique ? extend_one<OFF>(ix.bw, rng[2], rng[3], s, len, strand, i0R, +1, limR)
		     : (pk ? extend_one_text_packed<OFF>(ix, p + sl, +1, pk, nm, len, strand, i0R, +1, limR) : extend_one_text<OFF>(ix, p + sl, +1, s, len, strand, i0R, +1, limR));
}

