/* include/bt2g.h -- C ABI of libbt2g.so, the B200 (sm_100a) drop-in for bowtie2's alignment
 * hot path (SURVEY.md section 8b).
 *
 * The reference (BenLangmead/bowtie2 2.5.5) has no FFI boundary for this path: the only
 * extern "C" symbol is `int bowtie(int, const char**)` (bt2_search.cpp:5223-5230) and the hot
 * path is reached through C++ member calls from multiseedSearchWorker (bt2_search.cpp:3094).
 * This header therefore DEFINES the boundary; every entry point names the reference call(s)
 * it replaces.  All arguments are plain pointers and sizes (no torch / C++ types).  Return
 * value: 0 on success, negative on error (mirroring the reference's "throw 1 -> return 1"
 * convention, bt2_search.cpp:5353-5362); bt2g_last_error() gives the message.
 *
 * Offsets ("OFF" = TIndexOffU, btypes.h:23-43) are 4 bytes for .bt2 and 8 bytes for .bt2l
 * indexes.  Across this ABI every BW row / text offset travels as uint64_t regardless; the
 * index arrays themselves stay in their on-disk width.
 *
 * Buffers passed to the host-pointer entry points are host memory (pinned preferred); the
 * "_dev" twins take device pointers and an explicit cudaStream_t (passed as void*), do not
 * copy and do not synchronise.
 */
#ifndef BT2G_H_
#define BT2G_H_
#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct bt2g_ctx bt2g_ctx;

/* ---------------------------------------------------------------- context ------------- */
/* one context per GPU (replaces the per-process Ebwt/BitPairReference singletons that
 * multiseedSearch() publishes to its worker threads, bt2_search.cpp:4774-4790). */
int         bt2g_create(int device, bt2g_ctx **out);
void        bt2g_destroy(bt2g_ctx *ctx);
const char *bt2g_last_error(const bt2g_ctx *ctx);
int         bt2g_abi_version(void);

/* ---------------------------------------------------------------- index --------------- */
/* Host-side description of one loaded index, arrays in their on-disk layout
 * (Ebwt::readIntoMemory, bt2_io.cpp:131-616; BitPairReference ctor, reference.cpp:96-260).
 * "fw" = <base>.{1,2}.bt2[l]; "bw" = mirror index <base>.rev.1.bt2[l] (needed because
 * do1mmUpFront / SwDriver::extend use it, bt2_search.cpp:5149). */
typedef struct {
	int32_t  off_size;           /* 4 or 8 */
	int32_t  line_rate, off_rate, ftab_chars;
	uint64_t len;                /* joined text length */
	uint64_t n_pat, n_frag;
	uint64_t z_off_fw, z_off_bw;
	uint64_t fchr[5];
	const void    *plen;         /* OFF[n_pat] */
	const void    *rstarts;      /* OFF[3*n_frag] */
	const uint8_t *ebwt_fw;      /* num_sides * side_sz bytes */
	const uint8_t *ebwt_bw;      /* may be NULL */
	const void    *ftab_fw, *eftab_fw;   /* OFF[4^ftab_chars+1], OFF[2*ftab_chars] */
	const void    *ftab_bw, *eftab_bw;   /* may be NULL */
	const void    *offs;         /* OFF[offs_len] SA sample of the forward index */
	/* packed reference (.3/.4) */
	uint64_t n_recs;
	const void    *rec_off, *rec_len;    /* OFF[n_recs] */
	const uint8_t *rec_first;            /* u8[n_recs] */
	const uint8_t *ref_buf;              /* 2-bit packed, ceil(sum(rec_len)/4) bytes */
} bt2g_index_host;

/* Read <base>.{1,2,3,4,rev.1}.bt2 or .bt2l from disk and upload (Ebwt ctor + loadIntoMemory,
 * bt2_search.cpp:4986-5005,4832-4853; BitPairReference, :4789). */
int bt2g_load_index_files(bt2g_ctx *ctx, const char *basename);
/* Upload from host arrays (same content). */
int bt2g_load_index_host(bt2g_ctx *ctx, const bt2g_index_host *ix);
/* Adopt arrays that are ALREADY in this GPU's memory (pointers in bt2g_index_host are device
 * pointers; the caller keeps ownership).  This is how a torch.distributed/NCCL broadcast
 * receiver, or a GPU-side index builder, hands its tensors over. */
int bt2g_load_index_device(bt2g_ctx *ctx, const bt2g_index_host *ix_dev);

typedef struct {
	int32_t  off_size, line_rate, off_rate, ftab_chars;
	uint64_t len, bwt_len, num_sides, side_sz, side_bwt_sz, side_bwt_len;
	uint64_t ebwt_tot_len, offs_len, ftab_len, eftab_len, n_pat, n_frag, n_recs, ref_buf_bytes;
	uint64_t z_off_fw, z_off_bw;
	uint64_t fchr[5];
	int32_t  has_bw, has_ref;
	uint64_t device_bytes;      /* total HBM held by the index */
} bt2g_index_info;
int bt2g_index_info_get(const bt2g_ctx *ctx, bt2g_index_info *out);

/* Enumerate the device arrays of the loaded index (for one ncclBroadcast per array from the
 * rank that read the files; SURVEY.md section 8e).  which: 0 ebwt_fw, 1 ebwt_bw, 2 offs, 3 ftab_fw,
 * 4 eftab_fw, 5 ftab_bw, 6 eftab_bw, 7 plen, 8 rstarts, 9 rec_off, 10 rec_len, 11 rec_first,
 * 12 ref_buf.  Returns device pointer + byte size. */
#define BT2G_N_INDEX_ARRAYS 13
int bt2g_index_array(const bt2g_ctx *ctx, int which, void **dev_ptr, uint64_t *bytes);

/* ---------------------------------------------------------------- reads --------------- */
/* A batch of reads as the hot path sees them (Read::patFw / Read::qual, read.h:39):
 * seq[] = nucleotide codes 0..3 = A,C,G,T, 4 = N, all reads concatenated; qual[] = Phred+33
 * bytes, same layout; off[i]..off[i+1] delimits read i. */
typedef struct {
	uint64_t        n_reads;
	const uint8_t  *seq;
	const uint8_t  *qual;        /* may be NULL where quality is not needed */
	const uint64_t *off;         /* n_reads + 1 entries */
} bt2g_reads;

/* ---------------------------------------------------------------- FM primitives ------- */
/* Ebwt::countBt2SideEx via SideLocus::initFromRow (bt2_idx.h:1887-1919, :369-397):
 * out[4*i+c] = rank of nucleotide c at rows[i] (fchr + occ + in-side count, "$" adjusted). */
int bt2g_rank4(bt2g_ctx *ctx, int mirror, const uint64_t *rows, uint64_t n, uint64_t *out);
/* Ebwt::mapLF1(row, l, c) (bt2_idx.h:2420-2443): next row, or UINT64_MAX. */
int bt2g_maplf1(bt2g_ctx *ctx, int mirror, const uint64_t *rows, const uint8_t *chars, uint64_t n, uint64_t *out);
/* Ebwt::mapLFRange(ltop, lbot, num, cntsUpto, cntsIn, masks) (bt2_idx.h:2268-2305; countBt2SideRange :1804-1865,
 * countBt2SideRange2 :2177-2239), called per GroupWalk step (group_walk.h:897), for n ranges [tops[i], tops[i]+nums[i]):
 * upto[4*i+c] = rank of c at tops[i] ("$" adjusted), in[4*i+c] = rows of the range whose BWT character is c (the "$" row
 * tallied as an A, as the reference does), chars = the BWT character of every row, the ranges back to back (range i starts
 * at nums[0]+...+nums[i-1]); the reference's masks[c][j] is chars[j] == c.  -1 for an empty range or one that leaves the BWT. */
int bt2g_maplf_range(bt2g_ctx *ctx, int mirror, const uint64_t *tops, const uint64_t *nums, uint64_t n,
                     uint64_t *upto, uint64_t *in, uint8_t *chars);
/* Ebwt::ftabLoHi(i, top, bot) (bt2_idx.h:1476-1485). out[2*i]=top, out[2*i+1]=bot. */
int bt2g_ftab_lohi(bt2g_ctx *ctx, int mirror, const uint64_t *idx, uint64_t n, uint64_t *out);

/* ---------------------------------------------------------------- K1: seed search ----- */
/* SeedAligner::exactSweep (aligner_seed.cpp:856-970) with mineMax=2, repex=true, as called
 * at bt2_search.cpp:3514.  Per read: mine[2*i+{0,1}] = min(#edits lower bound, 2) for the
 * forward / reverse-complement read (0 for a skipped strand); ee[4*i+..] = topFw,botFw,topRc,botRc
 * of the exact end-to-end hit ranges (0,0 when none). */
int bt2g_exact_sweep(bt2g_ctx *ctx, const bt2g_reads *reads, int nofw, int norc,
                     uint8_t *mine, uint64_t *ee);

/* Seed layout for one seeding round (SeedAligner::instantiateSeeds, aligner_seed.cpp:498-587;
 * round arithmetic bt2_search.cpp:3905-3945).  All seeds are exact (multiseedMms == 0,
 * presets.cpp:37-92 => SEED_TYPE_EXACT). */
typedef struct {
	int32_t seed_len;            /* -L */
	int32_t max_seeds;           /* stride of the output: per read 2*max_seeds ranges */
	int32_t nofw, norc;
	const int32_t *interval;     /* per read: msIval.f(len), paired boost already applied */
	const int32_t *offset;       /* per read: (interval*roundi)/nrounds */
} bt2g_seed_plan;

/* SeedAligner::searchAllSeeds -> searchSeedBi/startSearchSeedBi for exact seeds
 * (aligner_seed.cpp:597-720, :1637-1718, :1858-2037) using Ebwt::ftabLoHi, mapBiLFEx,
 * mapLF1.  out[((i*2+strand)*max_seeds+k)*4 + {0,1,2,3}] = topf,botf,topb,botb of seed k
 * (k-th offset from the 5' end) of read i, all zero when the seed does not occur.
 * nseeds[i] receives the number of seed offsets of read i. */
int bt2g_seed_search(bt2g_ctx *ctx, const bt2g_reads *reads, const bt2g_seed_plan *plan,
                     uint64_t *out, int32_t *nseeds);

/* SeedAligner::oneMmSearch (aligner_seed.cpp:975-1325) as called from bt2_search.cpp:3709
 * (repex = false, rep1mm = true; scoring / local flag from bt2g_set_scoring): end-to-end hits
 * with exactly one mismatch.  strand_mask[i] bit0 = search the read (yfw), bit1 = search its
 * reverse complement (yrc) (bt2_search.cpp:3704-3706).  Task order per read = the reference's
 * loop order: (fw, forward index), (fw, mirror index), (rc, forward), (rc, mirror); within a task
 * hits appear by increasing depth then substituted nucleotide, i.e. the order of
 * SeedResults::add1mmEe calls.  counts[4*i+task] hits are stored at hits[(4*i+task)*max_hits ..]. */
typedef struct {
	uint64_t top, bot;           /* BW range in the FORWARD index */
	int32_t  pos;                /* mismatch offset from the 5' end of the read (Edit::pos) */
	int32_t  chr, qchr;          /* reference / read nucleotide codes (Edit::chr, qchr) */
	int32_t  score;
} bt2g_mm_hit;
int bt2g_one_mm(bt2g_ctx *ctx, const bt2g_reads *reads, const int32_t *minsc, const uint8_t *strand_mask,
                int32_t max_hits, bt2g_mm_hit *hits, int32_t *counts);

/* SwDriver::extend (aligner_sw_driver.cpp:299-484): for every seed hit of bt2g_seed_search
 * (same plan, `ranges` = its output) the number of read positions the hit extends without an
 * edit to the left (forward index) and to the right (mirror index), each capped at 255.
 * out[(((i*2+strand)*max_seeds+k)*2 + {0,1}] = nlex, nrex. */
int bt2g_extend_exact(bt2g_ctx *ctx, const bt2g_reads *reads, const bt2g_seed_plan *plan,
                      const uint64_t *ranges, uint8_t *out);

/* ---------------------------------------------------------------- K2: offset resolve -- */
/* GroupWalk2S::advanceElement == Ebwt::getOffset(row) (group_walk.h:1160-1215,517-520;
 * bt2_idx.cpp:150-171) followed by Ebwt::joinedToTextOff (bt2_idx.cpp:54-124) as
 * SwDriver::extendSeeds does (aligner_sw_driver.cpp:1126-1147).
 * For each i: joined[i] = offset in the joined text; tidx/textoff/tlen as joinedToTextOff
 * returns them for a hit of length hitlen[i]; flags bit0 = straddled, bit1 = rejected
 * (tidx == OFF_MASK, only when reject_straddle). Any output pointer may be NULL. */
int bt2g_resolve(bt2g_ctx *ctx, const uint64_t *rows, const uint32_t *hitlen, uint64_t n,
                 int reject_straddle, uint64_t *joined, uint64_t *tidx, uint64_t *textoff,
                 uint64_t *tlen, uint8_t *flags);

/* BitPairReference::getStretch (reference.cpp:420-560) with the off-end N padding of
 * SwAligner::initRef (aligner_sw.cpp:196-245): out[i*stride + k] = code of reference tidx[i]
 * at position off[i]+k for k < count[i] (4 = N / outside the reference). */
int bt2g_get_stretch(bt2g_ctx *ctx, const uint64_t *tidx, const int64_t *off, const int32_t *count,
                     uint64_t n, int32_t stride, uint8_t *out);

/* ---------------------------------------------------------------- K3: extension DP ----- */
/* Scoring scheme (Scoring, scoring.h:96-173; defaults :28-84; built at bt2_search.cpp:5040).
 * mmpen[q] / npen[q] are the per-quality penalty tables Scoring::initPens fills (q = Phred,
 * clamped to 63); bt2g_scoring_default() reproduces the reference defaults for end-to-end
 * (MA 0, MMP 6/2 by quality, NP 1, RDG/RFG 5+3, gap barrier 4) or --local (MA 2). */
typedef struct {
	int32_t match_bonus;
	int32_t rdgap_const, rdgap_linear, rfgap_const, rfgap_linear;
	int32_t gapbar;
	int32_t local;               /* 0 end-to-end (sc.monotone), 1 local */
	uint8_t mmpen[64];
	uint8_t npen[64];
	double  nceil_const, nceil_linear;   /* N ceiling function L,const,linear (scoring.h:58-62; (double)0.15f) */
} bt2g_scoring;
void bt2g_scoring_default(bt2g_scoring *sc, int local);
int  bt2g_set_scoring(bt2g_ctx *ctx, const bt2g_scoring *sc);

/* Highest generation of the end-to-end DP kernels the launchers may select (0 32-bit move codes, 1 s16x2 move codes,
 * 3 H-byte fill + tail = default; a cap of 2 selects 1); all generations return identical results (tests/test_dp_gpu.py).
 * A per-context setting: no process-global state. */
int  bt2g_set_dp_mode(bt2g_ctx *ctx, int cap);

/* SwDriver::extend (aligner_sw_driver.cpp:299-484) of a seed hit whose range is ONE row: 1 (default) = compare the read with the
 * 2-bit packed reference at the hit's joined-text offset (the characters LF would yield are the text's own), 0 = walk the index
 * as the reference does.  Results are identical (tests/test_fm_gpu.py); ranges of several rows always walk the index. */
int  bt2g_set_extend_mode(bt2g_ctx *ctx, int through_text);

/* One DP problem = one SwAligner::initRef + align + nextAlignment* session as issued by
 * SwDriver::extendSeeds (aligner_sw_driver.cpp:1272-1376).  The rectangle comes from
 * DynProgFramer::frameSeedExtensionRect (dp_framer.cpp:81-129; DPRect, dp_framer.h:59). */
typedef struct {
	uint32_t read_idx;           /* index into the bt2g_reads batch */
	uint32_t fw;                 /* 1 = align the read, 0 = its reverse complement */
	uint64_t tidx;               /* reference id */
	int64_t  refl, refr;         /* DPRect.refl / refr (post-trim, inclusive) */
	int32_t  triml;              /* DPRect.triml */
	int32_t  corel, corer;       /* DPRect core diagonals (offsets in the untrimmed rectangle) */
	int32_t  minsc;              /* minimum valid score */
	int32_t  nceil;              /* SwAligner::nceil_ = nCeil.f(rdlen) (aligner_sw.cpp:43) */
	int32_t  reserved;
} bt2g_dp_problem;

#define BT2G_DP_FLAG_BADSHAPE      1
#define BT2G_DP_FLAG_CAND_OVERFLOW 2   /* more candidate cells than max_cands */
#define BT2G_DP_FLAG_ALN_OVERFLOW  4   /* more successful backtraces than max_alns */
#define BT2G_DP_FLAG_OPS_OVERFLOW  8   /* an alignment longer than max_ops */
typedef struct {
	int32_t found;               /* SwAligner::align return value */
	int32_t best;                /* best score seen (aligner_sw.cpp:500 "best") */
	int32_t ncand;               /* |btncand_| */
	int32_t naln;                /* successful nextAlignment calls when every candidate is tried */
	int32_t flags;
} bt2g_dp_summary;

/* candidate cell, in btncand_ order (score desc, row desc, col desc; aligner_sw_nuc.h:149-157) */
#define BT2G_CAND_FILT_START 1   /* BT_CAND_FATE_FILT_START: start cell already reported through */
#define BT2G_CAND_FAILED     2   /* backtrace attempted and failed (RNG was consumed) */
#define BT2G_CAND_SUCCEEDED  3
#define BT2G_CAND_FILT_DOMINATED 4  /* local mode: within rows/16 of an attempted candidate (aligner_sw.cpp:946-971) */
typedef struct { int32_t score, row, col, fate; } bt2g_dp_cand;

/* one alignment: ops[] lists the alignment columns from the LAST read row back to the first
 * (the order the backtrace discovers them).  op & 3: 0 match, 1 mismatch (or N), 2 reference
 * gap (read char inserted), 3 read gap (reference char deleted); (op >> 2) & 7 = reference
 * nucleotide code of the column (0..3, 4 = N) for types 0, 1, 3. */
#define BT2G_OP_MATCH   0
#define BT2G_OP_MM      1
#define BT2G_OP_REFGAP  2
#define BT2G_OP_READGAP 3
typedef struct {
	int32_t cand_idx;            /* index into the candidate list */
	int32_t score, ns, gaps, refns;
	int32_t row0, col0;          /* first aligned cell: read row (= soft trim at the upstream end) and window column */
	int32_t trim_beg, trim_end;  /* soft-trimmed read rows upstream / downstream (local mode) */
	int32_t nops;
} bt2g_dp_aln;

/* Fill + gather + backtrace for n problems.  Output strides: cands[n][max_cands],
 * alns[n][max_alns], ops[n][max_alns][max_ops].  The reference offset of an alignment is
 * problem.refl + aln.col0. */
int bt2g_dp_extend(bt2g_ctx *ctx, const bt2g_reads *reads, const bt2g_dp_problem *probs, uint64_t n,
                   int32_t max_cands, int32_t max_alns, int32_t max_ops,
                   bt2g_dp_summary *summ, bt2g_dp_cand *cands, bt2g_dp_aln *alns, uint8_t *ops);

/* ------------------------------------------------------------------ extended seed table ----- */
/* An acceleration structure derived from the loaded index, in the spirit of ftab (bt2_idx.h:1373-1554)
 * but for k-mers of k > ftab_chars characters (k <= 16): for every k-mer, the state (topf, botf, topb)
 * of the bidirectional backward search after its k characters, i.e. exactly what ftabLoHi + (k -
 * ftab_chars) mapBiLFEx steps of SeedAligner::searchSeedBi would produce.  The seed-search kernel then
 * starts at depth k instead of ftab_chars; its results are bit-identical with and without the table.
 * Costs 3 * off_size * 4^k bytes of HBM (k = 14: 3.2 GB for .bt2) and one pass of (k - ftab_chars)
 * LF steps per entry at build time.  k = 0 drops the table. */
int bt2g_build_seed_table(bt2g_ctx *ctx, int k);

/* A denser suffix-array sample derived from the loaded index: offs2[row >> rate] for every row with
 * row % 2^rate == 0 (rate < offRate; rate = 0 is the full suffix array, 4 bytes x bwt_len for .bt2), each
 * value obtained with the index's own Ebwt::getOffset walk (bt2_idx.cpp:150-171).  bt2g_resolve and the
 * pipeline then stop their LF walk after < 2^rate steps instead of < 2^offRate; the offsets they return are
 * the same numbers.  rate < 0 drops it. */
int bt2g_build_dense_sa(bt2g_ctx *ctx, int rate);

/* ------------------------------------------------------------------- ungapped alignment ----- */
/* SwAligner::ungappedAlign (aligner_sw.cpp:286-487): the single-diagonal alignment the driver takes when
 * neither read nor reference gaps fit under the minimum score (aligner_sw_driver.cpp:1189-1253).
 * status: 0 no alignment, -1 more than one local solution on the diagonal (defer to the DP), 1 found.
 * Rows are in strand orientation (row 0 = leftmost aligned read position on the reference); the
 * reference offset of the alignment is refoff + rowi; edit_mask (optional, n * mask_stride bytes) gets a
 * 1 for every row in [rowi, rowf] whose base differs from the reference or faces an N. */
typedef struct {
	uint32_t read_idx;
	uint32_t fw;
	uint64_t tidx;
	int64_t  refoff;             /* Coord::off(): may be negative / run past the end (overhang) */
	uint64_t reflen;             /* length of the reference sequence */
	int32_t  minsc;
	int32_t  ohang;              /* gReportOverhangs */
} bt2g_ungapped_problem;
typedef struct {
	int32_t status, score;
	int32_t rowi, rowf;
	int32_t ns, refns, nedits, pad;
} bt2g_ungapped_result;
int bt2g_ungapped(bt2g_ctx *ctx, const bt2g_reads *reads, const bt2g_ungapped_problem *probs, uint64_t n,
                  bt2g_ungapped_result *out, uint8_t *edit_mask, uint32_t mask_stride);

/* ------------------------------------------------------------- paired-end framing ----- */
/* PairedEndPolicy (pe.h:169-330): pol = PE_POLICY_FF 1 / RR 2 / FR 3 / RF 4 (pe.h:43-55);
 * defaults of the program (bt2_search.cpp:350-358): FR, maxfrag 500, minfrag 0, flags
 * BT2G_PE_CONTAIN_OK | BT2G_PE_OLAP_OK | BT2G_PE_EXPAND_TO_FIT. */
#define BT2G_PE_FLIPPING_OK   1
#define BT2G_PE_DOVETAIL_OK   2
#define BT2G_PE_CONTAIN_OK    4
#define BT2G_PE_OLAP_OK       8
#define BT2G_PE_EXPAND_TO_FIT 16
typedef struct {
	int32_t  pol;
	int32_t  flags;
	uint64_t maxfrag, minfrag;
} bt2g_pe_policy;

/* one anchor alignment for which the opposite mate is sought (aligner_sw_driver.cpp:2157-2256) */
typedef struct {
	int64_t  off;                /* reference offset of the anchor alignment (AlnRes::refoff) */
	uint64_t reflen;             /* length of the reference sequence (tlen) */
	uint32_t len1, len2;         /* mate lengths */
	int32_t  maxalcols;          /* orows + oreadGaps, or -1 */
	int32_t  maxrdgap, maxrfgap; /* Scoring::maxReadGaps / maxRefGaps of the opposite mate */
	int32_t  maxns;              /* nCeil of the opposite mate */
	int32_t  maxhalf;            /* maxhalf (bt2_search.cpp: 15) */
	uint8_t  is1, fw;            /* anchor is mate 1?  anchor aligned to Watson? */
	uint8_t  pad[2];
} bt2g_mate_anchor;

/* PairedEndPolicy::otherMate (pe.cpp:161-355) followed by DynProgFramer::frameFindMateRect
 * (dp_framer.h:155-197; dp_framer.cpp:177-361; trimToRef = !gReportOverhangs = true):
 * status 0 = no concordant placement possible, 1 = window found but the rectangle is entirely
 * trimmed, 2 = rectangle valid. */
typedef struct {
	int32_t status;
	uint8_t oleft, ofw;          /* opposite mate lies to the left?  must align to Watson? */
	uint8_t pad[2];
	int64_t oll, olr, orl, orr;  /* windows for the LHS / RHS extreme of the opposite mate */
	int64_t refl, refr, refl_pretrim, refr_pretrim;
	int64_t triml, trimr, corel, corer, maxgap;   /* DPRect (dp_framer.h:33-73) */
} bt2g_mate_frame;
int bt2g_frame_mate(bt2g_ctx *ctx, const bt2g_pe_policy *pol, const bt2g_mate_anchor *anchors, uint64_t n,
                    bt2g_mate_frame *out);

/* PairedEndPolicy::peClassifyPair (pe.cpp:37-137) for n pairs: pairs[6*i] = off1, len1, fw1,
 * off2, len2, fw2; out[i] = PE_ALS_NORMAL 1 / OVERLAP 2 / CONTAIN 3 / DOVETAIL 4 / DISCORD 5. */
int bt2g_pe_classify(bt2g_ctx *ctx, const bt2g_pe_policy *pol, const int64_t *pairs, uint64_t n, int32_t *out);

/* ---------------------------------------------------------------- batched hot path ----- */
/* One pass of the hot path over a batch: exactSweep -> searchAllSeeds (round 0) -> offset
 * resolution -> extension DP + backtrace -> best alignment per read.  This is the unit the
 * caller (the restated multiseedSearchWorker loop, bt2_search.cpp:3253-4199) schedules; the
 * per-length tables carry the policy arithmetic the caller owns (scoreMin.f :3352-3372, nCeil.f
 * :3427, msIval.f :3443-3450, Scoring::maxReadGaps/maxRefGaps scoring.cpp:42,73). */
typedef struct {
	int32_t seed_len;            /* -L */
	int32_t max_seeds;           /* seeds per strand the buffers are sized for */
	int32_t row_cap;             /* BW rows resolved per read (<= 32) */
	int32_t range_max;           /* seed ranges wider than this are skipped by the collect stage */
	int32_t max_len;             /* longest read (<= 512) */
	int32_t maxhalf;             /* DP half-width cap (bt2_search.cpp maxhalf = 15) */
	int32_t max_cands, max_alns, max_ops;
	int32_t max_probs;           /* DP problems the workspace holds per batch (0 = max_reads*row_cap) */
	const int32_t *minsc_by_len, *nceil_by_len, *nceil_raw_by_len, *interval_by_len;   /* [max_len+1] */
	const int32_t *rdgaps_by_len, *rfgaps_by_len;                                     /* [max_len+1] */
} bt2g_pipeline_params;

typedef struct {
	int32_t  found;              /* 0 none, 1 gapped DP alignment, 2 exact end-to-end hit */
	int32_t  score, score2;      /* best and runner-up score (INT32_MIN when none) */
	uint32_t fw;
	uint64_t tidx;
	int64_t  refoff;             /* 0-based offset of the leftmost aligned reference base */
	int32_t  nops;               /* ops (bt2g_dp_aln encoding) in the per-read op buffer */
	int32_t  ndp;                /* DP problems issued for this read */
	int32_t  trim_left, trim_right; /* read positions soft-trimmed left / right of the alignment in reference
	                                 * orientation (local mode; SwResult alres softTrimmed 5'/3' per strand) */
	int32_t  mapq;               /* BowtieMapq2::mapq (unique.h:170-392) from score / score2 and the read's minimum and
	                              * perfect scores; for a concordant pair from the pair's score sums (no second-best pair
	                              * is tracked: the "no second best" branch) */
	int32_t  pad;                /* reference Ns spanned by the alignment (AlnRes::refNs, the XN:i field) */
} bt2g_read_result;

typedef struct bt2g_pipeline bt2g_pipeline;
int  bt2g_pipeline_create(bt2g_ctx *ctx, const bt2g_pipeline_params *prm, uint64_t max_reads, uint64_t max_bases,
                          bt2g_pipeline **out);
void bt2g_pipeline_destroy(bt2g_pipeline *p);
/* inputs already in HBM; asynchronous on `stream` (a cudaStream_t, NULL = the context stream);
 * count != 0 additionally tallies side fetches / DP cells (see bt2g_pipeline_counters) */
int  bt2g_pipeline_run_dev(bt2g_pipeline *p, const uint8_t *d_seq, const uint8_t *d_qual, const uint64_t *d_off,
                           uint64_t n_reads, void *stream, int count);
/* host buffers in, host results out (copies + kernels + synchronise): ops may be NULL,
 * else n_reads * max_ops bytes */
int  bt2g_pipeline_run_host(bt2g_pipeline *p, const bt2g_reads *reads, bt2g_read_result *res, uint8_t *ops);
int  bt2g_pipeline_results_dev(bt2g_pipeline *p, bt2g_read_result **res, uint8_t **ops);
int  bt2g_pipeline_counters(bt2g_pipeline *p, uint64_t *out6);
/* kernels launched by one bt2g_pipeline_run_dev call */
int  bt2g_pipeline_kernel_launches(bt2g_pipeline *p);
/* ---- paired-end pass (SwDriver::extendSeedsPaired's mate finding, aligner_sw_driver.cpp:2157-2440) ----
 * Reads are interleaved: mate 1 of pair i is read 2i, mate 2 is read 2i+1.  The pass runs the
 * single-end stages on all 2n reads, then for every aligned mate (the anchor) whose opposite mate has
 * no alignment concordant with it, frames the mate-finding rectangle (bt2g_frame_mate arithmetic) and
 * runs the same DP kernel on the opposite mate inside that window; finally the best concordant
 * combination per pair is chosen (peClassifyPair) and the per-read results are updated with it.
 * The reference runs the mate DP for EVERY anchor alignment as it goes; skipping it when the two
 * independent alignments already form a concordant pair is this pipeline's speculation (DESIGN.md). */
typedef struct {
	int32_t pair_type;           /* 0 neither mate aligned, 1 concordant pair, 2 both aligned but not concordant,
	                              * 3 only one mate aligned */
	int32_t kind;                /* peClassifyPair of the reported pair (1..4) or 5 */
	int32_t source;              /* 0 independent alignments, 1 mate 2 found by mate DP, 2 mate 1 found by mate DP */
	int32_t score_sum;           /* sum of the two alignment scores when pair_type == 1 */
	int64_t fraglen;             /* fragment length (pe.cpp:89-92) when pair_type == 1 */
} bt2g_pair_result;
int  bt2g_pipeline_enable_pairs(bt2g_pipeline *p, const bt2g_pe_policy *pol);
int  bt2g_pipeline_run_paired_dev(bt2g_pipeline *p, const uint8_t *d_seq, const uint8_t *d_qual, const uint64_t *d_off,
                                  uint64_t n_pairs, void *stream, int count);
int  bt2g_pipeline_run_paired_host(bt2g_pipeline *p, const bt2g_reads *reads, bt2g_read_result *res, uint8_t *ops,
                                   bt2g_pair_result *pairs);
int  bt2g_pipeline_pairs_dev(bt2g_pipeline *p, bt2g_pair_result **pairs);
/* [0] mate DP problems, [1] mate DP cells of the last paired run made with count != 0 */
int  bt2g_pipeline_pair_counters(bt2g_pipeline *p, uint64_t *out2);
/* device milliseconds of the paired tail of the last run: [0] mate framing, [1] mate DP, [2] pair pick */
int  bt2g_pipeline_pair_stage_ms(bt2g_pipeline *p, float *out3);

/* device milliseconds of the 8 stages of the last run (CUDA events on the launching stream) */
int  bt2g_pipeline_stage_ms(bt2g_pipeline *p, float *out8);

/* ---------------------------------------------------------------------- SAM records ----- */
/* The reporting tail for the pipeline's one-alignment-per-read results (host code, no GPU work):
 * AlnSinkSam::appendMate (aln_sink.cpp:1889-2060), StackedAln with leftAlign(false) -> CIGAR / MD:Z
 * (aligner_result.cpp:520-880), optional fields in the order of SamConfig::printAlignedOptFlags
 * (sam.cpp:121-330): AS XS XN XM XO XG NM MD YS YT.  `ops` / `max_ops` as returned by
 * bt2g_pipeline_run_*_host; `pairs` NULL for unpaired reads.  Returns 0, or -3 with *written = bytes
 * needed when `cap` is too small, or 1 when the text is complete but some alignment had more edit ops than
 * `max_ops` (bt2g_read_result.nops > max_ops: the engine could not store the whole op string, so that record's
 * CIGAR / MD:Z miss their beginning -- align again with a larger max_ops; only scoring schemes with very cheap gaps
 * produce alignments with more than read length + 64 ops). */
typedef struct {
	const char *const *ref_names;   /* [n_refs] reference names as they should appear in RNAME */
	uint64_t           n_refs;
	const char *const *read_names;  /* [n_reads] or NULL: "r<index>" (pair index for paired input) */
	int32_t            threads;     /* host threads formatting disjoint ranges of records (0 or 1 = the calling thread) */
	int32_t            sc_filter_maxlen; /* reads up to this length cannot reach the minimum score (Scoring::scoreFilter,
	                                     * bt2_search.cpp:3385: --local with very short reads): unaligned ones carry YF:Z:SC; 0 = none */
	double             nceil_const, nceil_linear;   /* --n-ceil (0, 0.15): unaligned reads with more Ns carry YF:Z:NS
	                                                * (bt2_search.cpp:3427-3431, sam.cpp:331-345); both 0 = defaults */
	uint32_t           flags;       /* BT2G_SAM_XEQ: --xeq (=/X instead of M); BT2G_SAM_NO_UNAL: --no-unal */
	uint32_t           reserved2;
	const char        *rg_optflag;  /* "RG:Z:<id>" of --rg-id, appended to every record (sam.cpp:384-387), or NULL */
} bt2g_sam_opts;
#define BT2G_SAM_XEQ     1u
#define BT2G_SAM_NO_UNAL 2u
/* --no-discordant: a pair whose mates both aligned exactly once without a concordant pair (pair_type 2) is NOT a discordant pair
 * (ReportingParams::discord, aln_sink.h:305-307; ReportingState::nextRead starts with doneDiscord_ set, aln_sink.cpp:38): its mates are reported as unpaired
 * alignments of a paired read (YT:Z:UP, no YS:i, TLEN 0).  pair_type 2 alone cannot tell: the caller passes the option. */
#define BT2G_SAM_NO_DISCORDANT 4u
int bt2g_sam_format(const bt2g_sam_opts *opt, const bt2g_reads *reads, const bt2g_read_result *res, const uint8_t *ops,
                    uint32_t max_ops, const bt2g_pair_result *pairs, char *out, uint64_t cap, uint64_t *written);

/* Host evaluations of the policy arithmetic that the kernels run on the device (one source for both: the
 * __host__ __device__ functions of mapq_device.cuh / pe_device.cuh), for callers that need a single value and for
 * the CPU test suite: BowtieMapq2::mapq (unique.h:170-392), PairedEndPolicy::otherMate + frameFindMateRect,
 * PairedEndPolicy::peClassifyPair. */
int bt2g_mapq(int64_t best, int has_secbest, int64_t secbest, int64_t sc_min, int64_t sc_perfect, int monotone);
int bt2g_frame_mate_host(const bt2g_pe_policy *pol, const bt2g_mate_anchor *anchors, uint64_t n, bt2g_mate_frame *out);
int bt2g_pe_classify_host(const bt2g_pe_policy *pol, const int64_t *pairs, uint64_t n, int32_t *out);

/* FASTQ text -> read buffers (host code; FastqPatternSource::parse, pat.cpp:1130-1245, plain 4-line records,
 * Phred+33, no trimming).  Parses whole records until max_reads / max_bases / the end of `text`; *consumed is the
 * offset of the first unparsed byte (a truncated last record is left for the next call).  names: n * name_stride
 * bytes, NUL-terminated header lines (may be NULL).  Errors: -4 not FASTQ, -5 integer qualities, -6 / -7 fewer /
 * more qualities than bases. */
int bt2g_fastq_parse(const char *text, uint64_t len, uint64_t max_reads, uint64_t max_bases, uint8_t *seq, uint8_t *qual,
                     uint64_t *off, char *names, uint32_t name_stride, uint64_t *n_reads, uint64_t *consumed);

/* SAM header: @HD, one @SQ per reference (name up to the first whitespace), and @PG with the given command line
 * when pg_cl != NULL (SamConfig::printHeader, sam.cpp:54-111).  -3 with *written = bytes needed when cap is short. */
int bt2g_sam_header(const char *const *names, const uint64_t *lens, uint64_t n, const char *pg_cl,
                    char *out, uint64_t cap, uint64_t *written);
/* the same with the @RG line of --rg-id / --rg between @SQ and @PG: rg_line = "ID:<id>\t<field>..." or NULL */
int bt2g_sam_header_rg(const char *const *names, const uint64_t *lens, uint64_t n, const char *rg_line, const char *pg_cl,
                       char *out, uint64_t cap, uint64_t *written);

/* Alignment summary = what the reference prints on stderr at the end of a run (AlnSink::printAlSumm,
 * aln_sink.cpp:349-528), from the counters AlnSinkWrap::finishRead keeps (aln_sink.cpp:708-1046).  The ">1 times"
 * lines print uni2 + rep of the reference's ReportingMetrics (the -M mode both presets use).  counts_add derives
 * the counters from pipeline results: a read "aligned >1 times" when a second alignment was found (score2 valid);
 * a pair is discordant when both mates aligned exactly once without forming a concordant pair; a concordant pair
 * counts ">1" when both mates have a second alignment (the pipeline does not keep the second-best PAIR: an
 * approximation of the reference's bestUnchosenCScore test, aln_sink.cpp:838-842). */
typedef struct {
	uint64_t nread, npaired, nunpaired;
	uint64_t nconcord_0, nconcord_uni1, nconcord_gt1, ndiscord;
	uint64_t nunp_0_0, nunp_0_uni1, nunp_0_gt1;       /* mates of pairs that aligned neither concordantly nor discordantly */
	uint64_t nunp_0, nunp_uni1, nunp_gt1;             /* unpaired reads */
} bt2g_align_counts;
int bt2g_align_counts_add(bt2g_align_counts *c, const bt2g_read_result *res, uint64_t n_reads, const bt2g_pair_result *pairs);
/* the same with formatter flags: BT2G_SAM_NO_DISCORDANT counts such pairs' mates under the unpaired tallies */
int bt2g_align_counts_add_ex(bt2g_align_counts *c, const bt2g_read_result *res, uint64_t n_reads, const bt2g_pair_result *pairs, uint32_t flags);
int bt2g_align_summary(const bt2g_align_counts *c, int discord, int mixed, char *out, uint64_t cap, uint64_t *written);

/* ---------------------------------------------------------------------- index files on the host ----- */
/* Host image of <basename>.{1,2,3,4,rev.1}.bt2[l] (no GPU involved): Ebwt::readIntoMemory (bt2_io.cpp:131-616) incl.
 * its endian switch and --offrate override (offrate_override < 0: none; <= the stored offRate: ignored), the
 * reference names stored after eftab, BitPairReference's .3/.4 (reference.cpp:30-260).  The descriptor points
 * into the image and stays valid until close; hand it to bt2g_load_index_host (or broadcast its arrays first). */
typedef struct bt2g_index_file bt2g_index_file;
int  bt2g_index_file_open(const char *basename, int offrate_override, bt2g_index_file **out, char *err, uint32_t err_cap);
const bt2g_index_host *bt2g_index_file_desc(const bt2g_index_file *f);
uint64_t bt2g_index_file_n_refs(const bt2g_index_file *f);
const char *const *bt2g_index_file_ref_names(const bt2g_index_file *f);
const uint64_t *bt2g_index_file_ref_lens(const bt2g_index_file *f);      /* plen[]: the @SQ LN values */
void bt2g_index_file_close(bt2g_index_file *f);
/* bt2g_load_index_files with an --offrate override */
int  bt2g_load_index_files_ex(bt2g_ctx *ctx, const char *basename, int offrate_override);


/* ------------------------------------------------------------- the exact search policy, in waves ----- */
/* The reference's sequential, RNG-driven policy (multiseedSearchWorker + SwDriver::extendSeeds[Paired] + AlnSinkWrap) for a
 * whole batch: every read (pair) is a coroutine blocked on one hot-path request at a time; per wave the pending requests
 * are grouped by primitive and answered by ONE call of the entry point below (csrc/policy_engine.cpp; specification and
 * CPU pinning: bowtie2_b200/policy_engine.py).  The backend table holds those entry points; bt2g_policy_backend_gpu fills it
 * with this library's own (ctx = the bt2g_ctx), the CPU test-suite fills it with callbacks that answer from the oracle. */
typedef struct {
	void *ctx;
	int (*exact_sweep)(void *, const bt2g_reads *, int, int, uint8_t *, uint64_t *);
	int (*seed_search)(void *, const bt2g_reads *, const bt2g_seed_plan *, uint64_t *, int32_t *);
	int (*one_mm)(void *, const bt2g_reads *, const int32_t *, const uint8_t *, int32_t, bt2g_mm_hit *, int32_t *);
	int (*extend_exact)(void *, const bt2g_reads *, const bt2g_seed_plan *, const uint64_t *, uint8_t *);
	int (*resolve)(void *, const uint64_t *, const uint32_t *, uint64_t, int, uint64_t *, uint64_t *, uint64_t *, uint64_t *, uint8_t *);
	int (*get_stretch)(void *, const uint64_t *, const int64_t *, const int32_t *, uint64_t, int32_t, uint8_t *);
	int (*ungapped)(void *, const bt2g_reads *, const bt2g_ungapped_problem *, uint64_t, bt2g_ungapped_result *, uint8_t *, uint32_t);
	int (*dp_extend)(void *, const bt2g_reads *, const bt2g_dp_problem *, uint64_t, int32_t, int32_t, int32_t, bt2g_dp_summary *,
	                 bt2g_dp_cand *, bt2g_dp_aln *, uint8_t *);
	int32_t off_size;            /* 4 (.bt2) or 8 (.bt2l): width of the RNG draws of eeSaTups */
	int32_t reserved;
} bt2g_policy_backend;
void bt2g_policy_backend_gpu(bt2g_ctx *ctx, bt2g_policy_backend *be);

typedef struct {
	int32_t local, paired;
	int32_t seed_len, seed_rounds, dp_fail_streak;          /* -L -R -D (the preset's values) */
	int32_t ival_type; double ival_const, ival_coeff;       /* -i: 1 const, 2 linear, 3 sqrt, 4 log (simple_func.h) */
	int32_t smin_type; double smin_const, smin_coeff;       /* --score-min (defaults are FLOAT literals: pass (double)-0.6f) */
	double  nceil_const, nceil_coeff;                       /* --n-ceil L,const,coeff */
	int64_t khits;                                          /* -k; 0 with all_hits = -a */
	int64_t mhits;                                          /* -M (default 50) */
	int32_t mmode, all_hits;                                /* mmode = no -k / -a given */
	int32_t nofw, norc, discord, mixed;
	uint32_t seed; int32_t max_inflight;                    /* --seed; reads (pairs) advanced together (0 = 65536) */
	int32_t match_bonus, mmp_max, mmp_min, n_pen, rdgap_const, rdgap_linear, rfgap_const, rfgap_linear;
	bt2g_pe_policy pe;
	int32_t host_threads;                                   /* threads resuming the per-read state machines between waves (0 / 1 = caller) */
	int32_t reserved;
} bt2g_policy_params;

/* reads: the batch (mates interleaved when prm->paired); names[i]: read names (the RNG seed depends on them).  Outputs as
 * bt2g_pipeline_run_[paired_]host: res[n_reads], ops[n_reads * max_ops], pairs[n_reads / 2] (NULL if unpaired).
 * stats (optional, 3 entries): waves, backend calls, requests.  The primary alignment per read / pair is reported. */
int bt2g_policy_align(const bt2g_policy_backend *be, const bt2g_policy_params *prm, const bt2g_reads *reads, const char *const *names,
                      bt2g_read_result *res, uint8_t *ops, uint32_t max_ops, bt2g_pair_result *pairs, uint64_t *stats);

/* -k N / -a for unpaired reads (AlnSinkWrap::finishRead with khits > 1, aln_sink.cpp:643-1070; ReportingState::getReport,
 * aln_sink.cpp:300-330): up to max_per_read records per read, rows [i * max_per_read, i * max_per_read + n_reported[i]) of res / ops:
 * the primary first, then the secondaries in the reference's order (found bit 8 set -> FLAG 256, MAPQ 255, the read's XS:i).
 * An unaligned read has n_reported[i] = 0 and an unaligned row at i * max_per_read.  Returns 1 when a read had more alignments
 * than max_per_read (the extra ones are dropped), 0 otherwise, < 0 on error (paired parameters are an error). */
int bt2g_policy_align_k(const bt2g_policy_backend *be, const bt2g_policy_params *prm, const bt2g_reads *reads, const char *const *names,
                        uint32_t max_per_read, bt2g_read_result *res, uint8_t *ops, uint32_t max_ops, uint32_t *n_reported,
                        uint64_t *stats);
/* paired -k N / -a: up to max_per_pair ENTRIES per pair.  Entry e of pair i = rows 2 * (i * max_per_pair + e) + {0, 1} of res / ops
 * and pairs[i * max_per_pair + e]: entry 0 carries the primaries of both mates; the further entries are the other concordant pairs
 * in the reference's report order, or -- when the pair did not align concordantly and a mate has further alignments -- every record
 * of mate 1 and then of mate 2, each beside the opposite mate's primary (AlnSinkWrap::finishRead, aln_sink.cpp:930-1010).  bt2g_read_result.found bit 8 marks a secondary
 * (FLAG 256, MAPQ 255), bit 9 a row that is present only as its mate's mate (bt2g_sam_format skips it).  n_entries[n_pairs].
 * Returns 1 when a pair had more entries than max_per_pair. */
int bt2g_policy_align_pairs_k(const bt2g_policy_backend *be, const bt2g_policy_params *prm, const bt2g_reads *reads, const char *const *names,
                              uint32_t max_per_pair, bt2g_read_result *res, uint8_t *ops, uint32_t max_ops, bt2g_pair_result *pairs,
                              uint32_t *n_entries, uint64_t *stats);

/* ------------------------------------------------------------- the exact search policy ON THE DEVICE ----- */
/* The same policy as bt2g_policy_align (results identical to the reference program's), but the per-read state machines run as a
 * kernel (csrc/xengine.cuh / xengine.cu: one thread per read pair or read, state in HBM) and the batched primitives consume
 * device-side request queues once per wave: no host round trip per request, the host only reads the queue counters of each wave.
 * This is the entry point the restated multiseedSearchWorker loop (bt2_search.cpp:3094-4254) calls per block of reads.
 * Supported: the default reporting mode (-M; no -k / -a), end-to-end and --local, paired and unpaired, reads up to 512 bp.
 * A unit whose state outgrows its fixed capacity is re-run by bt2g_policy_align over bt2g_policy_backend_gpu (same results).
 * create installs the scoring scheme of `prm` in the context (bt2g_set_scoring). */
typedef struct bt2g_xengine bt2g_xengine;
int  bt2g_xengine_create(bt2g_ctx *ctx, const bt2g_policy_params *prm, uint64_t max_units /* pairs or reads per call */, uint32_t max_len,
                         bt2g_xengine **out);
void bt2g_xengine_destroy(bt2g_xengine *e);
/* host buffers in, host results out (mates interleaved when paired).  names: n_reads rows of name_stride bytes, NUL-terminated
 * (the per-read RNG seed depends on the name, pat.cpp:45-82), or NULL = "r<pair or read index>".  res[n_reads],
 * ops[n_reads * max_ops], pairs[n_reads / 2] (paired).  stats (optional, 8 entries): waves, fallback units, seed-extension DPs,
 * mate-finding DPs, their DP cells (2 entries), 1-mismatch searches, seed searches. */
int  bt2g_xengine_align(bt2g_xengine *e, const bt2g_reads *reads, const char *names, uint32_t name_stride, bt2g_read_result *res,
                        uint8_t *ops, uint32_t max_ops, bt2g_pair_result *pairs, uint64_t *stats);
/* inputs already in HBM (d_names as above or NULL); results stay on the device until fetched */
int  bt2g_xengine_run_dev(bt2g_xengine *e, const uint8_t *d_seq, const uint8_t *d_qual, const uint64_t *d_off, uint64_t n_reads,
                          const char *d_names, uint32_t name_stride, void *stream, uint64_t *stats);
int  bt2g_xengine_results_dev(bt2g_xengine *e, bt2g_read_result **res, uint8_t **ops, uint32_t *max_ops, bt2g_pair_result **pairs);
/* An engine owns two CUDA streams (cudaStream_t): its waves run on *stream, the small waves of a batch's tail on *stream_hi (high
 * priority, so that several engines of one context interleave: one engine's tail is not queued behind another's full waves).  They
 * are used when bt2g_xengine_run_dev is given stream = NULL, and always by bt2g_xengine_align.  Every call returns with both idle. */
int  bt2g_xengine_streams(bt2g_xengine *e, void **stream, void **stream_hi);
/* device time of the last batch per stage, milliseconds (CUDA events on the batch's stream), 10 entries: admission (read seeds,
 * 2-bit packing, exactSweep), state machine steps, 1-mismatch searches, seed searches, seed-extension DP, mate-finding DP,
 * host fallback (wall clock), whole batch, and the split of the two DP entries into their fill kernels and their tail
 * (candidates + backtrace) kernels; *launches (optional) = kernels of this library launched by that batch */
int  bt2g_xengine_stage_ms(bt2g_xengine *e, float *ms, uint64_t *launches);
/* the same state machine driven on the host over an entry-point table (no GPU: the CPU pinning of csrc/xengine.cuh) */
int  bt2g_xengine_align_host(const bt2g_policy_backend *be, const bt2g_policy_params *prm, const bt2g_reads *reads, const char *const *names,
                             bt2g_read_result *res, uint8_t *ops, uint32_t max_ops, bt2g_pair_result *pairs, uint64_t *stats);

/* bt2g_fastq_parse on `threads` host threads: the text is cut at record boundaries, the pieces parsed concurrently and
 * concatenated in input order; outputs, limits and error codes as bt2g_fastq_parse */
int bt2g_fastq_parse_mt(const char *text, uint64_t len, uint64_t max_reads, uint64_t max_bases, uint8_t *seq, uint8_t *qual,
                        uint64_t *off, char *names, uint32_t name_stride, uint64_t *n_reads, uint64_t *consumed, int threads);

/* The two mate files of paired input into ONE interleaved batch: mate 1 of pair i is read 2i, mate 2 read 2i + 1 (the layout of every
 * paired entry point here; DualPatternComposer::nextBatch, pat.cpp:222-300, hands the reference's aligner the two mates together).
 * Both texts are parsed concurrently on `threads` host threads and the records written straight to their interleaved places.
 * Stops after max_pairs pairs, max_bases bases (both mates), or when either text runs out of whole records; *consumed1 / *consumed2 =
 * offset of the first unparsed byte of each text (the caller feeds the rest with its next block; the reference's "fewer reads in
 * file specified with -1 / -2" is the caller's call at end of input).  seq / qual: max_bases bytes; off: 2 * max_pairs + 1;
 * names: 2 * max_pairs rows of name_stride bytes, every byte defined (may be NULL).  Error codes as bt2g_fastq_parse. */
int bt2g_fastq_parse_pairs_mt(const char *text1, uint64_t len1, const char *text2, uint64_t len2, uint64_t max_pairs, uint64_t max_bases,
                              uint8_t *seq, uint8_t *qual, uint64_t *off, char *names, uint32_t name_stride, uint64_t *n_pairs,
                              uint64_t *consumed1, uint64_t *consumed2, int threads);

/* ------------------------------------------------------------- FASTQ text in -> SAM text out, the whole batch loop ----- */
/* The loop of multiseedSearchWorker (bt2_search.cpp:3253-4254) around the engines with its reader (PatternComposer::nextBatch,
 * pat.cpp:222-300; FastqPatternSource::parse :1130) and its ordered sink (AlnSinkWrap::finishRead aln_sink.cpp:643 ->
 * AlnSinkSam::appendMate :1889; OutputQueue of --reorder, outq.cpp) as overlapped host stages in C++ (csrc/stream_host.cpp):
 * the reader thread calls next_block and parses (parse_threads), one thread per engine calls `align`, the writer thread formats
 * (format_threads), adds the block to the alignment counts and calls write -- blocks leave in input order, each block in flight
 * owns one set of reused host buffers (depth + n_engines + 1 sets).
 *   align: bt2g_xengine_align itself (cast; engines[j] = a bt2g_xengine*), or any function of that shape.
 *   next_block: 1 = a block of WHOLE records (at most max_units reads or pairs; paired: the same number of records in both texts,
 *     *text2 / *len2 ignored otherwise), 0 = end of input, < 0 = error; the texts must stay valid until the next call of next_block.
 *   write: SAM records (no header: bt2g_sam_header), valid until write returns; 0 = ok.  One call per block -- more for a block with solo
 *     reads (see solo_engine) --, blocks in input order.
 * opt: as for bt2g_sam_format (read_names and threads are set per block here).  count_flags: as bt2g_align_counts_add_ex.
 * Returns 0, 1 (complete, but some alignment had more edit ops than max_ops: see bt2g_sam_format), or the first error of a stage
 * (parser codes -4..-7, engine codes, -20 reader, -22 block does not hold whole records, -23 a pair with an empty mate 2 and no solo_engine, -24 read longer than max_len, -25 writer) with its text in err. */
typedef int (*bt2g_stream_align_fn)(void *engine, const bt2g_reads *reads, const char *names, uint32_t name_stride, bt2g_read_result *res,
                                    uint8_t *ops, uint32_t max_ops, bt2g_pair_result *pairs, uint64_t *stats);
typedef struct {
	void *user;
	int (*next_block)(void *user, const char **text1, uint64_t *len1, const char **text2, uint64_t *len2);
	int (*write)(void *user, const char *sam, uint64_t len);
	/* Instead of next_block (used when not NULL): the mate files as byte streams -- read(user, mate 0 | 1, dst, cap) copies up to cap bytes of
	 * that file to dst and returns their number, 0 at the end of the file, < 0 on error (fread / gzread behind it).  The reader keeps one
	 * text buffer per file, takes up to max_units records from their fronts per block and carries the rest: the files are read in step by
	 * RECORD (DualPatternComposer::nextBatch, pat.cpp:222-300), a last record needs no final newline, "fewer reads in file specified with
	 * -1 / -2" is error -26, input that ends inside a record -22, a read name longer than name_stride - 2 bytes -27. */
	int64_t (*read)(void *user, int mate, char *dst, uint64_t cap);
} bt2g_stream_io;
typedef struct {
	int32_t  paired, parse_threads, format_threads, depth /* parsed blocks waiting for an engine; 0 = 2 */;
	uint64_t max_units;          /* reads (pairs) per block = the engines' capacity */
	uint32_t max_len, max_ops, name_stride, count_flags;
	uint64_t chunk_bytes;        /* read callback: bytes of text kept per file at the start (0 = 32 MiB); grows to a little more than max_units records */
	void    *solo_engine;        /* an UNPAIRED engine of the same run (same preset and options), or NULL.  A pair whose mate 2 is empty is an
	                              * unpaired read for the reference (`paired = !read_b().empty()`, bt2_search.cpp:3326): its mate 1 goes through the
	                              * unpaired policy and leaves ONE record (YT:Z:UU), counted with the unpaired reads.  With a solo engine those
	                              * pairs are aligned and written that way (in place, input order kept); without one they are error -23. */
	uint64_t solo_max_units;     /* capacity of the solo engine (0 = max_units) */
} bt2g_stream_params;
int bt2g_stream_run(bt2g_stream_align_fn align, void *const *engines, int32_t n_engines, const bt2g_stream_params *sp,
                    const bt2g_sam_opts *opt, const bt2g_stream_io *io, bt2g_align_counts *counts, uint64_t *n_reads,
                    char *err, uint32_t err_cap);

#ifdef __cplusplus
}
#endif
#endif /* BT2G_H_ */
