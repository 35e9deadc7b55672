// fm_kernels.cu -- FM-index primitive kernels, SwDriver::extend of seed hits and reference stretches for sm_100a.
// The seed search and offset resolution kernels are in fm_seed2.cu.
#include "fm_device.cuh"
#include "launch.cuh"

// ----------------------------------------------------------------------------------------
// primitive kernels (used by the parity tests and by the host policy as pure functions)
// ----------------------------------------------------------------------------------------
template <typename OFF>
__global__ void k_rank4(DevEbwt<OFF> e, const uint64_t *rows, uint64_t n, uint64_t *out) {
	uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if(i >= n) return;
	uint64_t r[4];
	rank4<OFF>(e, rows[i], r);
	out[4 * i + 0] = r[0]; out[4 * i + 1] = r[1]; out[4 * i + 2] = r[2]; out[4 * i + 3] = r[3];
}

template <typename OFF>
__global__ void k_maplf1(DevEbwt<OFF> e, const uint64_t *rows, const uint8_t *chars, uint64_t n, uint64_t *out) {
	uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if(i >= n) return;
	out[i] = maplf1<OFF>(e, rows[i], chars[i]);
}

template <typename OFF>
__global__ void k_ftab(DevEbwt<OFF> e, const uint64_t *idx, uint64_t n, uint64_t *out) {
	uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	if(i >= n) return;
	out[2 * i] = ftab_hi<OFF>(e, idx[i]);
	out[2 * i + 1] = ftab_lo<OFF>(e, idx[i] + 1);
}

// ----------------------------------------------------------------------------------------
// SwDriver::extend (aligner_sw_driver.cpp:299-484): how far each seed hit extends without an
// edit, to the left with the forward index and to the right with the mirror index (<= 255).
// Two threads per seed hit (one per direction) so both walks run concurrently.
// ----------------------------------------------------------------------------------------
template <typename OFF>
__global__ void k_extend(DevIndex<OFF> ix, const uint8_t *seq, const uint64_t *roff, uint64_t nReads,
                         int seedLen, int maxSeeds, const int32_t *interval, const int32_t *offset,
                         const uint64_t *ranges, uint8_t *out) {
	uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
	const uint64_t perRead = 4ull * maxSeeds;     // [strand][seed][direction]
	if(t >= nReads * perRead) return;
	const uint64_t rd = t / perRead;
	int rem = (int)(t - rd * perRead);
	const int dir = rem & 1; rem >>= 1;
	const int strand = rem / maxSeeds, k = rem - strand * maxSeeds;
	out[t] = 0;
	const uint64_t *q = ranges + ((rd * 2 + strand) * maxSeeds + k) * 4;
	if(q[1] <= q[0]) return;
	const uint8_t *s = seq + roff[rd];
	const int len = (int)(roff[rd + 1] - roff[rd]);
	const int sl = seedLen < len ? seedLen : len;
	const int off = k * interval[rd] + offset[rd];
	const bool fw = strand == 0;
	uint32_t nl = 0, nr = 0;
	extend_hit<OFF>(ix, q, s, len, fw, off, sl, dir == 0, dir != 0, nl, nr);
	out[t] = (uint8_t)(dir == 0 ? nl : nr);
}

template <typename OFF>
void launch_extend(const DevIndex<OFF> &ix, const uint8_t *seq, const uint64_t *roff, uint64_t nReads, int seedLen, int maxSeeds,
                   const int32_t *interval, const int32_t *offset, const uint64_t *ranges, uint8_t *out, cudaStream_t st) {
	uint64_t n = nReads * 4ull * maxSeeds;
	if(n) k_extend<OFF><<<(unsigned)((n + 127) / 128), 128, 0, st>>>(ix, seq, roff, nReads, seedLen, maxSeeds, interval, offset, ranges, out);
}
template void launch_extend<uint32_t>(const DevIndex<uint32_t> &, const uint8_t *, const uint64_t *, uint64_t, int, int, const int32_t *, const int32_t *, const uint64_t *, uint8_t *, cudaStream_t);
template void launch_extend<uint64_t>(const DevIndex<uint64_t> &, const uint8_t *, const uint64_t *, uint64_t, int, int, const int32_t *, const int32_t *, const uint64_t *, uint8_t *, cudaStream_t);

template <typename OFF>
__global__ void k_get_stretch(DevIndex<OFF> ix, const uint64_t *tidx, const int64_t *off, const int32_t *count,
                              uint64_t n, int stride, uint8_t *out) {
	uint64_t i = blockIdx.x;
	if(i >= n) return;
	for(int k = threadIdx.x; k < count[i]; k += blockDim.x) {
		out[i * (uint64_t)stride + k] = (uint8_t)ref_base<OFF>(ix, tidx[i], off[i] + k);
	}
}

// ----------------------------------------------------------------------------------------
// launchers (called from api.cu)
// ----------------------------------------------------------------------------------------
static inline unsigned gridFor(uint64_t n, unsigned block) { return (unsigned)((n + block - 1) / block); }

// Ebwt::mapLFRange (bt2_idx.h:2268-2305) = countBt2SideRange (:1804-1865) + countBt2SideRange2 (:2177-2239): the GroupWalk step
// of a range that is still several rows wide (group_walk.h:897).  One warp per range.  Lane 0 takes the four ranks at `top`
// (one side fetch, as rank4).  The rows are then walked side by side: the first WORDS lanes pull the side's BWT words with one
// coalesced load, every lane decodes the characters of its rows out of the word it gets by shuffle, writes them (32 consecutive
// bytes per warp store) and tallies them; the tallies are reduced over the warp.  The reference's four bool lists are
// masks[c][j] == (chars[j] == c); like the reference (:2209) the "$" row counts as an A in `in`, and not in `upto`.
template <typename OFF>
__global__ void k_maplf_range(DevEbwt<OFF> e, const uint64_t *tops, const uint64_t *nums, const uint64_t *rowOff, uint64_t n,
                              uint64_t *upto, uint64_t *in, uint8_t *chars) {
	constexpr uint32_t BL = SideGeom<OFF>::BWT_LEN, WORDS = SideGeom<OFF>::WORDS, SIDE_SZ = SideGeom<OFF>::SIDE_SZ;
	const uint32_t lane = threadIdx.x & 31;
	const uint64_t w = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
	if(w >= n) return;
	const uint64_t top = tops[w], num = nums[w];
	uint8_t *out = chars + rowOff[w];
	if(lane == 0) {
		uint64_t r[4];
		rank4<OFF>(e, top, r);
		upto[4 * w + 0] = r[0]; upto[4 * w + 1] = r[1]; upto[4 * w + 2] = r[2]; upto[4 * w + 3] = r[3];
	}
	uint64_t nA = 0, nC = 0, nG = 0, nT = 0, done = 0;
	uint64_t sideNum = top / BL;
	uint32_t charOff = (uint32_t)(top - sideNum * BL);
	while(done < num) {
		const uint64_t left = num - done;
		const uint32_t take = left < (uint64_t)(BL - charOff) ? (uint32_t)left : BL - charOff;
		uint64_t word = 0;
		if(lane < WORDS) word = __ldg((const unsigned long long *)(e.ebwt + sideNum * SIDE_SZ) + lane);
		for(uint32_t base = 0; base < take; base += 32) {
			const uint32_t k = base + lane, pos = charOff + k;
			const uint32_t src = (pos >> 5) < WORDS ? (pos >> 5) : WORDS - 1;
			const uint64_t ww = __shfl_sync(0xffffffffu, word, src);
			if(k < take) {
				const uint32_t c = (uint32_t)(ww >> ((pos & 31) * 2)) & 3;
				out[done + k] = (uint8_t)c;
				nA += c == 0; nC += c == 1; nG += c == 2; nT += c == 3;
			}
		}
		done += take;
		sideNum++; charOff = 0;                          // SideLocus::nextSide (:1857)
	}
#pragma unroll
	for(int d = 16; d > 0; d >>= 1) {
		nA += __shfl_xor_sync(0xffffffffu, nA, d); nC += __shfl_xor_sync(0xffffffffu, nC, d);
		nG += __shfl_xor_sync(0xffffffffu, nG, d); nT += __shfl_xor_sync(0xffffffffu, nT, d);
	}
	if(lane == 0) { in[4 * w + 0] = nA; in[4 * w + 1] = nC; in[4 * w + 2] = nG; in[4 * w + 3] = nT; }
}

template <typename OFF>
void launch_rank4(const DevEbwt<OFF> &e, const uint64_t *rows, uint64_t n, uint64_t *out, cudaStream_t st) {
	if(n) k_rank4<OFF><<<gridFor(n, 256), 256, 0, st>>>(e, rows, n, out);
}
template <typename OFF>
void launch_maplf1(const DevEbwt<OFF> &e, const uint64_t *rows, const uint8_t *chars, uint64_t n, uint64_t *out, cudaStream_t st) {
	if(n) k_maplf1<OFF><<<gridFor(n, 256), 256, 0, st>>>(e, rows, chars, n, out);
}
template <typename OFF>
void launch_maplf_range(const DevEbwt<OFF> &e, const uint64_t *tops, const uint64_t *nums, const uint64_t *rowOff, uint64_t n,
                        uint64_t *upto, uint64_t *in, uint8_t *chars, cudaStream_t st) {
	if(n) k_maplf_range<OFF><<<gridFor(n * 32, 256), 256, 0, st>>>(e, tops, nums, rowOff, n, upto, in, chars);
}
template <typename OFF>
void launch_ftab(const DevEbwt<OFF> &e, const uint64_t *idx, uint64_t n, uint64_t *out, cudaStream_t st) {
	if(n) k_ftab<OFF><<<gridFor(n, 256), 256, 0, st>>>(e, idx, n, out);
}
template <typename OFF>
void launch_get_stretch(const DevIndex<OFF> &ix, const uint64_t *tidx, const int64_t *off, const int32_t *count,
                        uint64_t n, int stride, uint8_t *out, cudaStream_t st) {
	if(n) k_get_stretch<OFF><<<(unsigned)n, 64, 0, st>>>(ix, tidx, off, count, n, stride, out);
}

#define INSTANTIATE(OFF)                                                                                          \
	template void launch_rank4<OFF>(const DevEbwt<OFF> &, const uint64_t *, uint64_t, uint64_t *, cudaStream_t);  \
	template void launch_maplf1<OFF>(const DevEbwt<OFF> &, const uint64_t *, const uint8_t *, uint64_t, uint64_t *, cudaStream_t); \
	template void launch_maplf_range<OFF>(const DevEbwt<OFF> &, const uint64_t *, const uint64_t *, const uint64_t *, uint64_t, uint64_t *, uint64_t *, uint8_t *, cudaStream_t); \
	template void launch_ftab<OFF>(const DevEbwt<OFF> &, const uint64_t *, uint64_t, uint64_t *, cudaStream_t);   \
	template void launch_get_stretch<OFF>(const DevIndex<OFF> &, const uint64_t *, const int64_t *, const int32_t *, uint64_t, int, uint8_t *, cudaStream_t);
INSTANTIATE(uint32_t)
INSTANTIATE(uint64_t)
