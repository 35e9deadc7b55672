// launch.cuh -- the kernel launchers that one translation unit of libbt2g.so calls in another.  The defining files include it
// too, and the library is linked with --no-undefined, so a definition that drifts from its declaration fails the build.
// Default arguments are given here and nowhere else; the explicit instantiations stay next to the definitions.
#pragma once
#include "bt2g_internal.h"

struct DpLaunch;   // dp_device.cuh

// ---- fm_kernels.cu: FM-index primitives, SwDriver::extend, reference stretches ---------------
template <typename OFF> void launch_rank4(const DevEbwt<OFF> &e, const uint64_t *rows, uint64_t n, uint64_t *out, cudaStream_t st);
template <typename OFF> void launch_maplf1(const DevEbwt<OFF> &e, const uint64_t *rows, const uint8_t *chars, uint64_t n, uint64_t *out, cudaStream_t st);
template <typename OFF> void launch_maplf_range(const DevEbwt<OFF> &e, const uint64_t *tops, const uint64_t *nums, const uint64_t *rowOff, uint64_t n,
                                                uint64_t *upto, uint64_t *in, uint8_t *chars, cudaStream_t st);
template <typename OFF> void launch_ftab(const DevEbwt<OFF> &e, const uint64_t *idx, uint64_t n, uint64_t *out, cudaStream_t st);
template <typename OFF> void launch_extend(const DevIndex<OFF> &ix, const uint8_t *seq, const uint64_t *roff, uint64_t nReads, int seedLen, int maxSeeds,
                                           const int32_t *interval, const int32_t *offset, const uint64_t *ranges, uint8_t *out, cudaStream_t st);
template <typename OFF> void launch_get_stretch(const DevIndex<OFF> &ix, const uint64_t *tidx, const int64_t *off, const int32_t *count,
                                                uint64_t n, int stride, uint8_t *out, cudaStream_t st);

// ---- fm_seed2.cu: read packing, exact sweep, multiseed search, offset resolution, seed tables --
void launch_pack_reads(const uint8_t *seq, const uint64_t *roff, uint64_t nReads, int maxLen, uint64_t *packed, uint32_t *nmask, cudaStream_t st);
template <typename OFF> void launch_exact_sweep2(const DevIndex<OFF> &ix, const uint64_t *roff, uint64_t nReads, int nofw, int norc,
                                                 uint8_t *mine, uint64_t *ee, const uint64_t *packed, const uint32_t *nmask, unsigned long long *next,
                                                 int numSMs, cudaStream_t st, unsigned long long *cnt, int flags = 0);
template <typename OFF> void launch_seed_search2(const DevIndex<OFF> &ix, const uint8_t *seq, const uint64_t *roff, uint64_t nReads, int maxLen,
                                                 int seedLen, int maxSeeds, int nofw, int norc, const int32_t *interval, const int32_t *offset,
                                                 uint64_t *out, int32_t *nseeds, uint64_t *packed, uint32_t *nmask, unsigned long long *next,
                                                 int numSMs, cudaStream_t st, unsigned long long *cnt);
template <typename OFF> void launch_seed_search_active(const DevIndex<OFF> &ix, const uint64_t *roff, uint64_t nReads, int seedLen, int maxSeeds,
                                                       const int32_t *interval, const int32_t *offset, const uint8_t *actv, uint64_t *out, int32_t *nseeds,
                                                       const uint64_t *packed, const uint32_t *nmask, unsigned long long *next, int numSMs, cudaStream_t st);
template <typename OFF> void launch_resolve2(const DevIndex<OFF> &ix, const uint64_t *rows, const uint32_t *hitlen, uint64_t nHost, const uint32_t *nDev,
                                             int rej, uint64_t *joined, uint64_t *tidx, uint64_t *textoff, uint64_t *tlen, uint8_t *flags,
                                             unsigned long long *next, int numSMs, cudaStream_t st, unsigned long long *cnt);
template <typename OFF> void launch_build_ktab(const DevIndex<OFF> &ix, int K, OFF *out, cudaStream_t st);
template <typename OFF> void launch_build_dense_sa(const DevIndex<OFF> &ix, int rate, OFF *out, cudaStream_t st);

// ---- fm_onemm.cu: 1-mismatch end-to-end search ------------------------------------------------
template <typename OFF> void launch_one_mm(const DevIndex<OFF> &ix, const uint8_t *seq, const uint8_t *qual, const uint64_t *roff, uint64_t nReads,
                                           const int32_t *minsc, const uint8_t *strandMask, const bt2g_scoring &sc, int maxHits, bt2g_mm_hit *hits,
                                           int32_t *counts, cudaStream_t st);
template <typename OFF> void launch_one_mm_sel(const DevIndex<OFF> &ix, const uint8_t *seq, const uint8_t *qual, const uint64_t *roff, uint64_t nSlots,
                                               const uint32_t *sel, const int32_t *minsc, const uint8_t *strandMask, const bt2g_scoring &sc, int maxHits,
                                               bt2g_mm_hit *hits, int32_t *counts, cudaStream_t st, bool text);

// ---- dp_kernels.cu / dp_ungapped.cu: dynamic programming ----------------------------------------
template <typename OFF> int launch_dp_e2e(const DevIndex<OFF> &ix, const bt2g_scoring &sc, const DpLaunch &L, int maxRdLen, cudaStream_t st);
template <typename OFF> int launch_dp_local(const DevIndex<OFF> &ix, const bt2g_scoring &sc, const DpLaunch &L, int maxRdLen, cudaStream_t st);
template <typename OFF> void launch_ungapped(const DevIndex<OFF> &ix, const bt2g_scoring &sc, const uint8_t *seq, const uint8_t *qual, const uint64_t *roff,
                                             const bt2g_ungapped_problem *probs, uint64_t n, bt2g_ungapped_result *out, uint8_t *mask, uint32_t stride,
                                             cudaStream_t st);

// ---- pe_kernels.cu: paired-end framing -----------------------------------------------------------
void launch_frame_mate(const bt2g_pe_policy &pp, const bt2g_mate_anchor *anchors, uint64_t n, bt2g_mate_frame *out, cudaStream_t st);
void launch_pe_classify(const bt2g_pe_policy &pp, const int64_t *pairs, uint64_t n, int32_t *out, cudaStream_t st);
