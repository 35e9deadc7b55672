// api.cu -- C-ABI entry points of libbt2g.so (include/bt2g.h): context, index residency in HBM,
// and the host-buffer wrappers around the K1/K2 kernels.
#include "bt2g_internal.h"
#include "dp_device.cuh"
#include "launch.cuh"
#include <cstring>
#include <new>

namespace {

// RAII device buffer for the host-pointer wrappers
struct DBuf {
	void *p = nullptr;
	size_t bytes = 0;
	~DBuf() { if(p) cudaFree(p); }
	cudaError_t alloc(size_t n) { bytes = n; return cudaMalloc(&p, n ? n : 1); }
	template <typename T> T *as() { return (T *)p; }
};

void freeArr(DevArray &a) {
	if(a.owned && a.ptr) cudaFree(a.ptr);
	a = DevArray();
}

void freeIndex(bt2g_ctx *ctx) {
	for(int i = 0; i < BT2G_N_INDEX_ARRAYS; i++) freeArr(ctx->arr[i]);
	freeArr(ctx->recCumOff); freeArr(ctx->recCumUnamb); freeArr(ctx->refRecOffs); freeArr(ctx->refLens);
	freeArr(ctx->ktab); ctx->ktabChars = 0;
	freeArr(ctx->denseSa); ctx->denseRate = -1;
	ctx->loaded = false;
}

uint64_t readOffHost(const void *p, uint64_t i, int offSize) {
	return offSize == 4 ? ((const uint32_t *)p)[i] : ((const uint64_t *)p)[i];
}

// fills ctx->info from the header part of a bt2g_index_host (EbwtParams::init, bt2_idx.h:133-167)
void fillInfo(bt2g_ctx *ctx, const bt2g_index_host *ix) {
	bt2g_index_info &f = ctx->info;
	memset(&f, 0, sizeof(f));
	f.off_size = ix->off_size; f.line_rate = ix->line_rate; f.off_rate = ix->off_rate; f.ftab_chars = ix->ftab_chars;
	f.len = ix->len; f.bwt_len = ix->len + 1;
	f.side_sz = 1ull << ix->line_rate;
	f.side_bwt_sz = f.side_sz - 4ull * ix->off_size;
	f.side_bwt_len = f.side_bwt_sz * 4;
	uint64_t bwtSz = ix->len / 4 + 1;
	f.num_sides = (bwtSz + f.side_bwt_sz - 1) / f.side_bwt_sz;
	f.ebwt_tot_len = f.num_sides * f.side_sz;
	f.offs_len = (f.bwt_len + (1ull << ix->off_rate) - 1) >> ix->off_rate;
	f.ftab_len = (1ull << (2 * ix->ftab_chars)) + 1;
	f.eftab_len = 2ull * ix->ftab_chars;
	f.n_pat = ix->n_pat; f.n_frag = ix->n_frag; f.n_recs = ix->n_recs;
	f.z_off_fw = ix->z_off_fw; f.z_off_bw = ix->z_off_bw;
	for(int i = 0; i < 5; i++) f.fchr[i] = ix->fchr[i];
	f.has_bw = ix->ebwt_bw != nullptr;
	f.has_ref = ix->ref_buf != nullptr;
}

void arrayBytes(const bt2g_index_info &f, uint64_t refBases, uint64_t bytes[BT2G_N_INDEX_ARRAYS]) {
	uint64_t os = f.off_size;
	bytes[0] = f.ebwt_tot_len; bytes[1] = f.has_bw ? f.ebwt_tot_len : 0; bytes[2] = f.offs_len * os;
	bytes[3] = f.ftab_len * os; bytes[4] = f.eftab_len * os;
	bytes[5] = f.has_bw ? f.ftab_len * os : 0; bytes[6] = f.has_bw ? f.eftab_len * os : 0;
	bytes[7] = f.n_pat * os; bytes[8] = f.n_frag * 3 * os;
	bytes[9] = f.n_recs * os; bytes[10] = f.n_recs * os; bytes[11] = f.n_recs; bytes[12] = (refBases + 3) >> 2;
}

// derived per-record tables for device-side BitPairReference::getBase (reference.cpp:118-166)
int buildRefTables(bt2g_ctx *ctx, const void *recOff, const void *recLen, const uint8_t *recFirst, uint64_t nRecs,
                   int offSize, uint64_t &refBases) {
	std::vector<uint64_t> cumOff(nRecs), cumUnamb(nRecs), refRecOffs, refLens;
	uint64_t cumsz = 0, cumlen = 0;
	for(uint64_t i = 0; i < nRecs; i++) {
		if(recFirst[i]) {
			if(!refRecOffs.empty()) refLens.push_back(cumlen);
			refRecOffs.push_back(i);
			cumlen = 0;
		}
		cumOff[i] = cumlen; cumUnamb[i] = cumsz;
		cumsz += readOffHost(recLen, i, offSize);
		cumlen += readOffHost(recOff, i, offSize) + readOffHost(recLen, i, offSize);
	}
	refRecOffs.push_back(nRecs);
	refLens.push_back(cumlen);
	refBases = cumsz;
	ctx->nRefs = refLens.size();
	auto up = [&](DevArray &a, const std::vector<uint64_t> &v) -> int {
		a.bytes = v.size() * 8; a.owned = true;
		BT2G_CUDA_TRY(ctx, cudaMalloc(&a.ptr, a.bytes ? a.bytes : 8));
		BT2G_CUDA_TRY(ctx, cudaMemcpy(a.ptr, v.data(), a.bytes, cudaMemcpyHostToDevice));
		return 0;
	};
	if(up(ctx->recCumOff, cumOff) || up(ctx->recCumUnamb, cumUnamb) || up(ctx->refRecOffs, refRecOffs) || up(ctx->refLens, refLens)) return -2;
	return 0;
}

const void *hostArr(const bt2g_index_host *ix, int which) {
	switch(which) {
		case 0: return ix->ebwt_fw; case 1: return ix->ebwt_bw; case 2: return ix->offs;
		case 3: return ix->ftab_fw; case 4: return ix->eftab_fw; case 5: return ix->ftab_bw; case 6: return ix->eftab_bw;
		case 7: return ix->plen; case 8: return ix->rstarts; case 9: return ix->rec_off; case 10: return ix->rec_len;
		case 11: return ix->rec_first; case 12: return ix->ref_buf;
	}
	return nullptr;
}

int loadCommon(bt2g_ctx *ctx, const bt2g_index_host *ix, bool fromDevice) {
	if(!ctx || !ix) return -1;
	if(ix->off_size != 4 && ix->off_size != 8) { ctx->err = "off_size must be 4 or 8"; return -1; }
	if(ix->line_rate != (ix->off_size == 4 ? 6 : 7)) { ctx->err = "line_rate must be 6 (.bt2) / 7 (.bt2l)"; return -1; }
	BT2G_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
	freeIndex(ctx);
	fillInfo(ctx, ix);
	// record tables need host copies of the (small) record arrays
	uint64_t refBases = 0;
	if(ix->n_recs) {
		uint64_t os = ix->off_size;
		std::vector<uint8_t> ro(ix->n_recs * os), rl(ix->n_recs * os), rf(ix->n_recs);
		if(fromDevice) {
			BT2G_CUDA_TRY(ctx, cudaMemcpy(ro.data(), ix->rec_off, ro.size(), cudaMemcpyDeviceToHost));
			BT2G_CUDA_TRY(ctx, cudaMemcpy(rl.data(), ix->rec_len, rl.size(), cudaMemcpyDeviceToHost));
			BT2G_CUDA_TRY(ctx, cudaMemcpy(rf.data(), ix->rec_first, rf.size(), cudaMemcpyDeviceToHost));
		} else {
			memcpy(ro.data(), ix->rec_off, ro.size()); memcpy(rl.data(), ix->rec_len, rl.size()); memcpy(rf.data(), ix->rec_first, rf.size());
		}
		int rc = buildRefTables(ctx, ro.data(), rl.data(), rf.data(), ix->n_recs, ix->off_size, refBases);
		if(rc) return rc;
	}
	uint64_t bytes[BT2G_N_INDEX_ARRAYS];
	arrayBytes(ctx->info, refBases, bytes);
	ctx->info.ref_buf_bytes = bytes[12];
	uint64_t total = 0;
	for(int i = 0; i < BT2G_N_INDEX_ARRAYS; i++) {
		const void *src = hostArr(ix, i);
		if(!src || bytes[i] == 0) continue;
		DevArray &a = ctx->arr[i];
		a.bytes = bytes[i];
		if(fromDevice) {
			a.ptr = const_cast<void *>(src); a.owned = false;
		} else {
			a.owned = true;
			BT2G_CUDA_TRY(ctx, cudaMalloc(&a.ptr, a.bytes));
			BT2G_CUDA_TRY(ctx, cudaMemcpy(a.ptr, src, a.bytes, cudaMemcpyHostToDevice));
		}
		total += a.bytes;
	}
	ctx->info.device_bytes = total + ctx->recCumOff.bytes + ctx->recCumUnamb.bytes + ctx->refRecOffs.bytes + ctx->refLens.bytes;
	ctx->loaded = true;
	return 0;
}

template <typename OFF>
DevEbwt<OFF> devEbwt(const bt2g_ctx *ctx, bool mirror) {
	DevEbwt<OFF> e;
	const bt2g_index_info &f = ctx->info;
	e.ebwt = (const uint8_t *)ctx->arr[mirror ? 1 : 0].ptr;
	e.ftab = (const OFF *)ctx->arr[mirror ? 5 : 3].ptr;
	e.eftab = (const OFF *)ctx->arr[mirror ? 6 : 4].ptr;
	e.len = f.len;
	e.zOff = mirror ? f.z_off_bw : f.z_off_fw;
	e.zSide = e.zOff / f.side_bwt_len;
	e.zChar = (uint32_t)(e.zOff % f.side_bwt_len);
	for(int i = 0; i < 5; i++) e.fchr[i] = f.fchr[i];
	e.ftabChars = f.ftab_chars;
	return e;
}

} // namespace

template <typename OFF>
DevIndex<OFF> bt2g_dev_index(const bt2g_ctx *ctx) {
	DevIndex<OFF> ix;
	ix.fw = devEbwt<OFF>(ctx, false);
	ix.bw = devEbwt<OFF>(ctx, true);
	ix.offs = (const OFF *)ctx->arr[2].ptr;
	ix.ktab = (const OFF *)ctx->ktab.ptr; ix.ktabChars = ctx->ktab.ptr ? ctx->ktabChars : 0;
	if(ctx->denseSa.ptr) { ix.saOffs = (const OFF *)ctx->denseSa.ptr; ix.saRate = ctx->denseRate; }
	else { ix.saOffs = ix.offs; ix.saRate = ctx->info.off_rate; }
	ix.extText = ctx->extendText;
	ix.offRate = ctx->info.off_rate;
	ix.rstarts = (const OFF *)ctx->arr[8].ptr;
	ix.nFrag = ctx->info.n_frag;
	ix.plen = (const OFF *)ctx->arr[7].ptr;
	ix.nPat = ctx->info.n_pat;
	ix.recOff = (const OFF *)ctx->arr[9].ptr;
	ix.recLen = (const OFF *)ctx->arr[10].ptr;
	ix.recCumOff = (const uint64_t *)ctx->recCumOff.ptr;
	ix.recCumUnamb = (const uint64_t *)ctx->recCumUnamb.ptr;
	ix.refRecOffs = (const uint64_t *)ctx->refRecOffs.ptr;
	ix.refLens = (const uint64_t *)ctx->refLens.ptr;
	ix.refBuf = (const uint8_t *)ctx->arr[12].ptr;
	ix.nRecs = ctx->info.n_recs;
	ix.nRefs = ctx->nRefs;
	return ix;
}
template DevIndex<uint32_t> bt2g_dev_index<uint32_t>(const bt2g_ctx *);
template DevIndex<uint64_t> bt2g_dev_index<uint64_t>(const bt2g_ctx *);

#define REQUIRE_LOADED(ctx)                                         \
	do {                                                            \
		if(!(ctx)) return -1;                                       \
		if(!(ctx)->loaded) { (ctx)->err = "no index loaded"; return -1; } \
		BT2G_CUDA_TRY(ctx, cudaSetDevice((ctx)->device));           \
	} while(0)

// dispatch on offset width
#define DISPATCH(ctx, CALL32, CALL64) do { if((ctx)->info.off_size == 4) { CALL32; } else { CALL64; } } while(0)

extern "C" {

int bt2g_abi_version(void) { return 1; }

int bt2g_create(int device, bt2g_ctx **out) {
	if(!out) return -1;
	*out = nullptr;
	int n = 0;
	if(cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) return -3;  // no CUDA device: fail loudly
	bt2g_ctx *ctx = new(std::nothrow) bt2g_ctx();
	if(!ctx) return -4;
	ctx->device = device;
	if(cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) {
		delete ctx; return -2;
	}
	*out = ctx;
	return 0;
}

void bt2g_destroy(bt2g_ctx *ctx) {
	if(!ctx) return;
	cudaSetDevice(ctx->device);
	freeIndex(ctx);
	for(auto &s : ctx->scratch) freeArr(s);
	if(ctx->stream) cudaStreamDestroy(ctx->stream);
	delete ctx;
}

const char *bt2g_last_error(const bt2g_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int bt2g_load_index_files(bt2g_ctx *ctx, const char *basename) {
	if(!ctx || !basename) return -1;
	HostIndex h;
	if(bt2g_read_index_files(basename, h, ctx->err)) return -1;
	return loadCommon(ctx, &h.d, false);
}

int bt2g_load_index_host(bt2g_ctx *ctx, const bt2g_index_host *ix) { return loadCommon(ctx, ix, false); }
int bt2g_load_index_device(bt2g_ctx *ctx, const bt2g_index_host *ix) { return loadCommon(ctx, ix, true); }

int bt2g_index_info_get(const bt2g_ctx *ctx, bt2g_index_info *out) {
	if(!ctx || !out || !ctx->loaded) return -1;
	*out = ctx->info;
	return 0;
}

int bt2g_index_array(const bt2g_ctx *ctx, int which, void **devPtr, uint64_t *bytes) {
	if(!ctx || !ctx->loaded || which < 0 || which >= BT2G_N_INDEX_ARRAYS) return -1;
	if(devPtr) *devPtr = ctx->arr[which].ptr;
	if(bytes) *bytes = ctx->arr[which].bytes;
	return 0;
}

// ---- FM primitives -----------------------------------------------------------------------
int bt2g_rank4(bt2g_ctx *ctx, int mirror, const uint64_t *rows, uint64_t n, uint64_t *out) {
	REQUIRE_LOADED(ctx);
	if(mirror && !ctx->info.has_bw) { ctx->err = "mirror index not loaded"; return -1; }
	DBuf dr, dout;
	BT2G_CUDA_TRY(ctx, dr.alloc(n * 8)); BT2G_CUDA_TRY(ctx, dout.alloc(n * 32));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(dr.p, rows, n * 8, cudaMemcpyHostToDevice, ctx->stream));
	DISPATCH(ctx, launch_rank4<uint32_t>(devEbwt<uint32_t>(ctx, mirror), dr.as<uint64_t>(), n, dout.as<uint64_t>(), ctx->stream),
	              launch_rank4<uint64_t>(devEbwt<uint64_t>(ctx, mirror), dr.as<uint64_t>(), n, dout.as<uint64_t>(), ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaGetLastError());
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(out, dout.p, n * 32, cudaMemcpyDeviceToHost, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
	return 0;
}

int bt2g_maplf1(bt2g_ctx *ctx, int mirror, const uint64_t *rows, const uint8_t *chars, uint64_t n, uint64_t *out) {
	REQUIRE_LOADED(ctx);
	if(mirror && !ctx->info.has_bw) { ctx->err = "mirror index not loaded"; return -1; }
	DBuf dr, dc, dout;
	BT2G_CUDA_TRY(ctx, dr.alloc(n * 8)); BT2G_CUDA_TRY(ctx, dc.alloc(n)); BT2G_CUDA_TRY(ctx, dout.alloc(n * 8));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(dr.p, rows, n * 8, cudaMemcpyHostToDevice, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(dc.p, chars, n, cudaMemcpyHostToDevice, ctx->stream));
	DISPATCH(ctx, launch_maplf1<uint32_t>(devEbwt<uint32_t>(ctx, mirror), dr.as<uint64_t>(), dc.as<uint8_t>(), n, dout.as<uint64_t>(), ctx->stream),
	              launch_maplf1<uint64_t>(devEbwt<uint64_t>(ctx, mirror), dr.as<uint64_t>(), dc.as<uint8_t>(), n, dout.as<uint64_t>(), ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaGetLastError());
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(out, dout.p, n * 8, cudaMemcpyDeviceToHost, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
	return 0;
}

int bt2g_maplf_range(bt2g_ctx *ctx, int mirror, const uint64_t *tops, const uint64_t *nums, uint64_t n, uint64_t *upto, uint64_t *in, uint8_t *chars) {
	REQUIRE_LOADED(ctx);
	if(mirror && !ctx->info.has_bw) { ctx->err = "mirror index not loaded"; return -1; }
	if(n == 0) return 0;
	const uint64_t bwtLen = ctx->info.len + 1;
	std::vector<uint64_t> rowOff(n + 1, 0);
	for(uint64_t i = 0; i < n; i++) {
		if(nums[i] == 0 || tops[i] >= bwtLen || nums[i] > bwtLen - tops[i]) { ctx->err = "bt2g_maplf_range: a range is empty or leaves the BWT"; return -1; }
		rowOff[i + 1] = rowOff[i] + nums[i];
	}
	const uint64_t rows = rowOff[n];
	DBuf dt, dn, dro, du, di, dc;
	BT2G_CUDA_TRY(ctx, dt.alloc(n * 8)); BT2G_CUDA_TRY(ctx, dn.alloc(n * 8)); BT2G_CUDA_TRY(ctx, dro.alloc((n + 1) * 8));
	BT2G_CUDA_TRY(ctx, du.alloc(n * 32)); BT2G_CUDA_TRY(ctx, di.alloc(n * 32)); BT2G_CUDA_TRY(ctx, dc.alloc(rows));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(dt.p, tops, n * 8, cudaMemcpyHostToDevice, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(dn.p, nums, n * 8, cudaMemcpyHostToDevice, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(dro.p, rowOff.data(), (n + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
	DISPATCH(ctx, launch_maplf_range<uint32_t>(devEbwt<uint32_t>(ctx, mirror), dt.as<uint64_t>(), dn.as<uint64_t>(), dro.as<uint64_t>(), n, du.as<uint64_t>(), di.as<uint64_t>(), dc.as<uint8_t>(), ctx->stream),
	              launch_maplf_range<uint64_t>(devEbwt<uint64_t>(ctx, mirror), dt.as<uint64_t>(), dn.as<uint64_t>(), dro.as<uint64_t>(), n, du.as<uint64_t>(), di.as<uint64_t>(), dc.as<uint8_t>(), ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaGetLastError());
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(upto, du.p, n * 32, cudaMemcpyDeviceToHost, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(in, di.p, n * 32, cudaMemcpyDeviceToHost, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(chars, dc.p, rows, cudaMemcpyDeviceToHost, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
	return 0;
}

int bt2g_ftab_lohi(bt2g_ctx *ctx, int mirror, const uint64_t *idx, uint64_t n, uint64_t *out) {
	REQUIRE_LOADED(ctx);
	if(mirror && !ctx->info.has_bw) { ctx->err = "mirror index not loaded"; return -1; }
	DBuf di, dout;
	BT2G_CUDA_TRY(ctx, di.alloc(n * 8)); BT2G_CUDA_TRY(ctx, dout.alloc(n * 16));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(di.p, idx, n * 8, cudaMemcpyHostToDevice, ctx->stream));
	DISPATCH(ctx, launch_ftab<uint32_t>(devEbwt<uint32_t>(ctx, mirror), di.as<uint64_t>(), n, dout.as<uint64_t>(), ctx->stream),
	              launch_ftab<uint64_t>(devEbwt<uint64_t>(ctx, mirror), di.as<uint64_t>(), n, dout.as<uint64_t>(), ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaGetLastError());
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(out, dout.p, n * 16, cudaMemcpyDeviceToHost, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
	return 0;
}

// ---- K1 ------------------------------------------------------------------------------------
static int uploadReads(bt2g_ctx *ctx, const bt2g_reads *r, DBuf &dseq, DBuf &dqual, DBuf &doff, bool wantQual) {
	uint64_t nb = r->off[r->n_reads];
	BT2G_CUDA_TRY(ctx, dseq.alloc(nb)); BT2G_CUDA_TRY(ctx, doff.alloc((r->n_reads + 1) * 8));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(dseq.p, r->seq, nb, cudaMemcpyHostToDevice, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(doff.p, r->off, (r->n_reads + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
	if(wantQual && r->qual) {
		BT2G_CUDA_TRY(ctx, dqual.alloc(nb));
		BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(dqual.p, r->qual, nb, cudaMemcpyHostToDevice, ctx->stream));
	}
	return 0;
}

int bt2g_exact_sweep(bt2g_ctx *ctx, const bt2g_reads *reads, int nofw, int norc, uint8_t *mine, uint64_t *ee) {
	REQUIRE_LOADED(ctx);
	if(!reads || !mine || !ee) return -1;
	uint64_t n = reads->n_reads;
	if(n == 0) return 0;
	DBuf dseq, dqual, doff, dmine, dee;
	int rc = uploadReads(ctx, reads, dseq, dqual, doff, false);
	if(rc) return rc;
	BT2G_CUDA_TRY(ctx, dmine.alloc(n * 2)); BT2G_CUDA_TRY(ctx, dee.alloc(n * 32));
	int maxLen = 1;
	for(uint64_t i = 0; i < n; i++) { int l = (int)(reads->off[i + 1] - reads->off[i]); if(l > maxLen) maxLen = l; }
	DBuf dpack, dnm, dnext;
	const uint64_t nWords = (reads->off[n] >> 5) + n + 2;
	BT2G_CUDA_TRY(ctx, dpack.alloc(nWords * 8)); BT2G_CUDA_TRY(ctx, dnm.alloc(nWords * 4)); BT2G_CUDA_TRY(ctx, dnext.alloc(8));
	int sms = 148; cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
	launch_pack_reads(dseq.as<uint8_t>(), doff.as<uint64_t>(), n, maxLen, dpack.as<uint64_t>(), dnm.as<uint32_t>(), ctx->stream);
	DISPATCH(ctx, launch_exact_sweep2<uint32_t>(bt2g_dev_index<uint32_t>(ctx), doff.as<uint64_t>(), n, nofw, norc, dmine.as<uint8_t>(), dee.as<uint64_t>(), dpack.as<uint64_t>(), dnm.as<uint32_t>(), dnext.as<unsigned long long>(), sms, ctx->stream, nullptr),
	              launch_exact_sweep2<uint64_t>(bt2g_dev_index<uint64_t>(ctx), doff.as<uint64_t>(), n, nofw, norc, dmine.as<uint8_t>(), dee.as<uint64_t>(), dpack.as<uint64_t>(), dnm.as<uint32_t>(), dnext.as<unsigned long long>(), sms, ctx->stream, nullptr));
	BT2G_CUDA_TRY(ctx, cudaGetLastError());
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(mine, dmine.p, n * 2, cudaMemcpyDeviceToHost, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(ee, dee.p, n * 32, cudaMemcpyDeviceToHost, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
	return 0;
}

int bt2g_seed_search(bt2g_ctx *ctx, const bt2g_reads *reads, const bt2g_seed_plan *plan, uint64_t *out, int32_t *nseeds) {
	REQUIRE_LOADED(ctx);
	if(!reads || !plan || !out || plan->max_seeds <= 0 || plan->seed_len <= 0) return -1;
	uint64_t n = reads->n_reads;
	if(n == 0) return 0;
	DBuf dseq, dqual, doff, dint, doffs, dout, dns;
	int rc = uploadReads(ctx, reads, dseq, dqual, doff, false);
	if(rc) return rc;
	uint64_t outBytes = n * 2ull * plan->max_seeds * 4 * 8;
	BT2G_CUDA_TRY(ctx, dint.alloc(n * 4)); BT2G_CUDA_TRY(ctx, doffs.alloc(n * 4));
	BT2G_CUDA_TRY(ctx, dout.alloc(outBytes)); BT2G_CUDA_TRY(ctx, dns.alloc(n * 4));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(dint.p, plan->interval, n * 4, cudaMemcpyHostToDevice, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(doffs.p, plan->offset, n * 4, cudaMemcpyHostToDevice, ctx->stream));
	if(plan->seed_len > 32) { ctx->err = "seed length must be <= 32 (as in bowtie2 -L)"; return -1; }
	int maxLen = 1;
	for(uint64_t i = 0; i < n; i++) { int l = (int)(reads->off[i + 1] - reads->off[i]); if(l > maxLen) maxLen = l; }
	DBuf dpack, dnm, dnext;
	const uint64_t nWords = (reads->off[n] >> 5) + n + 2;
	BT2G_CUDA_TRY(ctx, dpack.alloc(nWords * 8)); BT2G_CUDA_TRY(ctx, dnm.alloc(nWords * 4)); BT2G_CUDA_TRY(ctx, dnext.alloc(8));
	int sms = 148; cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
	launch_pack_reads(dseq.as<uint8_t>(), doff.as<uint64_t>(), n, maxLen, dpack.as<uint64_t>(), dnm.as<uint32_t>(), ctx->stream);
	DISPATCH(ctx, launch_seed_search2<uint32_t>(bt2g_dev_index<uint32_t>(ctx), dseq.as<uint8_t>(), doff.as<uint64_t>(), n, maxLen, plan->seed_len, plan->max_seeds, plan->nofw, plan->norc, dint.as<int32_t>(), doffs.as<int32_t>(), dout.as<uint64_t>(), dns.as<int32_t>(), dpack.as<uint64_t>(), dnm.as<uint32_t>(), dnext.as<unsigned long long>(), sms, ctx->stream, nullptr),
	              launch_seed_search2<uint64_t>(bt2g_dev_index<uint64_t>(ctx), dseq.as<uint8_t>(), doff.as<uint64_t>(), n, maxLen, plan->seed_len, plan->max_seeds, plan->nofw, plan->norc, dint.as<int32_t>(), doffs.as<int32_t>(), dout.as<uint64_t>(), dns.as<int32_t>(), dpack.as<uint64_t>(), dnm.as<uint32_t>(), dnext.as<unsigned long long>(), sms, ctx->stream, nullptr));
	BT2G_CUDA_TRY(ctx, cudaGetLastError());
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(out, dout.p, outBytes, cudaMemcpyDeviceToHost, ctx->stream));
	if(nseeds) BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(nseeds, dns.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
	return 0;
}

int bt2g_one_mm(bt2g_ctx *ctx, const bt2g_reads *reads, const int32_t *minsc, const uint8_t *strandMask, int32_t maxHits,
                bt2g_mm_hit *hits, int32_t *counts) {
	REQUIRE_LOADED(ctx);
	if(!reads || !reads->qual || !minsc || !strandMask || !hits || !counts || maxHits < 1) return -1;
	if(!ctx->info.has_bw) { ctx->err = "mirror index not loaded"; return -1; }
	if(ctx->scoring.gapbar < 1) bt2g_scoring_default(&ctx->scoring, 0);
	uint64_t n = reads->n_reads;
	if(n == 0) return 0;
	DBuf dseq, dqual, doff, dms, dmask, dhits, dcnt;
	int rc = uploadReads(ctx, reads, dseq, dqual, doff, true);
	if(rc) return rc;
	BT2G_CUDA_TRY(ctx, dms.alloc(n * 4)); BT2G_CUDA_TRY(ctx, dmask.alloc(n));
	BT2G_CUDA_TRY(ctx, dhits.alloc(n * 4 * (uint64_t)maxHits * sizeof(bt2g_mm_hit))); BT2G_CUDA_TRY(ctx, dcnt.alloc(n * 16));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(dms.p, minsc, n * 4, cudaMemcpyHostToDevice, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(dmask.p, strandMask, n, cudaMemcpyHostToDevice, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaMemsetAsync(dhits.p, 0, dhits.bytes, ctx->stream));
	DISPATCH(ctx, launch_one_mm<uint32_t>(bt2g_dev_index<uint32_t>(ctx), dseq.as<uint8_t>(), dqual.as<uint8_t>(), doff.as<uint64_t>(), n, dms.as<int32_t>(), dmask.as<uint8_t>(), ctx->scoring, maxHits, dhits.as<bt2g_mm_hit>(), dcnt.as<int32_t>(), ctx->stream),
	              launch_one_mm<uint64_t>(bt2g_dev_index<uint64_t>(ctx), dseq.as<uint8_t>(), dqual.as<uint8_t>(), doff.as<uint64_t>(), n, dms.as<int32_t>(), dmask.as<uint8_t>(), ctx->scoring, maxHits, dhits.as<bt2g_mm_hit>(), dcnt.as<int32_t>(), ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaGetLastError());
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(hits, dhits.p, dhits.bytes, cudaMemcpyDeviceToHost, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(counts, dcnt.p, n * 16, cudaMemcpyDeviceToHost, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
	return 0;
}

int bt2g_ungapped(bt2g_ctx *ctx, const bt2g_reads *reads, const bt2g_ungapped_problem *probs, uint64_t n,
                  bt2g_ungapped_result *out, uint8_t *editMask, uint32_t maskStride) {
	REQUIRE_LOADED(ctx);
	if(!ctx->info.has_ref) { ctx->err = "packed reference (.3/.4) not loaded"; return -1; }
	if(!reads || !reads->qual || !probs || !out) { ctx->err = "null argument"; return -1; }
	if(ctx->scoring.gapbar < 1) bt2g_scoring_default(&ctx->scoring, 0);
	if(n == 0) return 0;
	for(uint64_t i = 0; i < n; i++) if(probs[i].read_idx >= reads->n_reads) { ctx->err = "read_idx out of range"; return -1; }
	DBuf dseq, dqual, doff, dprob, dout, dmask;
	int rc = uploadReads(ctx, reads, dseq, dqual, doff, true);
	if(rc) return rc;
	BT2G_CUDA_TRY(ctx, dprob.alloc(n * sizeof(bt2g_ungapped_problem))); BT2G_CUDA_TRY(ctx, dout.alloc(n * sizeof(bt2g_ungapped_result)));
	if(editMask) { BT2G_CUDA_TRY(ctx, dmask.alloc(n * (uint64_t)maskStride)); BT2G_CUDA_TRY(ctx, cudaMemsetAsync(dmask.p, 0, dmask.bytes, ctx->stream)); }
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(dprob.p, probs, dprob.bytes, cudaMemcpyHostToDevice, ctx->stream));
	DISPATCH(ctx, launch_ungapped<uint32_t>(bt2g_dev_index<uint32_t>(ctx), ctx->scoring, dseq.as<uint8_t>(), dqual.as<uint8_t>(), doff.as<uint64_t>(), dprob.as<bt2g_ungapped_problem>(), n, dout.as<bt2g_ungapped_result>(), editMask ? dmask.as<uint8_t>() : nullptr, maskStride, ctx->stream),
	              launch_ungapped<uint64_t>(bt2g_dev_index<uint64_t>(ctx), ctx->scoring, dseq.as<uint8_t>(), dqual.as<uint8_t>(), doff.as<uint64_t>(), dprob.as<bt2g_ungapped_problem>(), n, dout.as<bt2g_ungapped_result>(), editMask ? dmask.as<uint8_t>() : nullptr, maskStride, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaGetLastError());
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(out, dout.p, dout.bytes, cudaMemcpyDeviceToHost, ctx->stream));
	if(editMask) BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(editMask, dmask.p, dmask.bytes, cudaMemcpyDeviceToHost, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
	return 0;
}

int bt2g_build_seed_table(bt2g_ctx *ctx, int k) {
	REQUIRE_LOADED(ctx);
	BT2G_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
	BT2G_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
	freeArr(ctx->ktab); ctx->ktabChars = 0;
	if(k == 0) return 0;
	const int F = ctx->info.ftab_chars;
	if(k <= F || k > 16 || F < 1) { ctx->err = "seed table: k must be in (ftab_chars, 16]"; return -1; }
	if(!ctx->info.has_bw) { ctx->err = "seed table: mirror index not loaded"; return -1; }
	const uint64_t entries = 1ull << (2 * k), bytes = entries * 3ull * (uint64_t)ctx->info.off_size;
	void *p = nullptr;
	cudaError_t e = cudaMalloc(&p, bytes);
	if(e != cudaSuccess) { ctx->err = std::string("seed table cudaMalloc: ") + cudaGetErrorString(e); return -2; }
	if(ctx->info.off_size == 4) launch_build_ktab<uint32_t>(bt2g_dev_index<uint32_t>(ctx), k, (uint32_t *)p, ctx->stream);
	else launch_build_ktab<uint64_t>(bt2g_dev_index<uint64_t>(ctx), k, (uint64_t *)p, ctx->stream);
	e = cudaStreamSynchronize(ctx->stream);
	if(e == cudaSuccess) e = cudaGetLastError();
	if(e != cudaSuccess) { cudaFree(p); ctx->err = std::string("seed table build: ") + cudaGetErrorString(e); return -2; }
	ctx->ktab.ptr = p; ctx->ktab.bytes = bytes; ctx->ktab.owned = true; ctx->ktabChars = k;
	return 0;
}

int bt2g_build_dense_sa(bt2g_ctx *ctx, int rate) {
	REQUIRE_LOADED(ctx);
	BT2G_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
	BT2G_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
	freeArr(ctx->denseSa); ctx->denseRate = -1;
	if(rate < 0) return 0;
	if(rate >= ctx->info.off_rate) { ctx->err = "dense SA: rate must be below the index's offRate"; return -1; }
	const uint64_t entries = (ctx->info.bwt_len + ((1ull << rate) - 1)) >> rate, bytes = entries * (uint64_t)ctx->info.off_size;
	void *p = nullptr;
	cudaError_t e = cudaMalloc(&p, bytes ? bytes : 1);
	if(e != cudaSuccess) { ctx->err = std::string("dense SA cudaMalloc: ") + cudaGetErrorString(e); return -2; }
	if(ctx->info.off_size == 4) launch_build_dense_sa<uint32_t>(bt2g_dev_index<uint32_t>(ctx), rate, (uint32_t *)p, ctx->stream);
	else launch_build_dense_sa<uint64_t>(bt2g_dev_index<uint64_t>(ctx), rate, (uint64_t *)p, ctx->stream);
	e = cudaStreamSynchronize(ctx->stream);
	if(e == cudaSuccess) e = cudaGetLastError();
	if(e != cudaSuccess) { cudaFree(p); ctx->err = std::string("dense SA build: ") + cudaGetErrorString(e); return -2; }
	ctx->denseSa.ptr = p; ctx->denseSa.bytes = bytes; ctx->denseSa.owned = true; ctx->denseRate = rate;
	return 0;
}

int bt2g_frame_mate(bt2g_ctx *ctx, const bt2g_pe_policy *pol, const bt2g_mate_anchor *anchors, uint64_t n, bt2g_mate_frame *out) {
	if(!ctx) return -1;
	if(!pol || !anchors || !out || pol->pol < 1 || pol->pol > 4) { ctx->err = "bt2g_frame_mate: bad argument"; return -1; }
	if(n == 0) return 0;
	BT2G_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
	DBuf da, dout;
	BT2G_CUDA_TRY(ctx, da.alloc(n * sizeof(bt2g_mate_anchor))); BT2G_CUDA_TRY(ctx, dout.alloc(n * sizeof(bt2g_mate_frame)));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(da.p, anchors, da.bytes, cudaMemcpyHostToDevice, ctx->stream));
	launch_frame_mate(*pol, da.as<bt2g_mate_anchor>(), n, dout.as<bt2g_mate_frame>(), ctx->stream);
	BT2G_CUDA_TRY(ctx, cudaGetLastError());
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(out, dout.p, dout.bytes, cudaMemcpyDeviceToHost, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
	return 0;
}

int bt2g_pe_classify(bt2g_ctx *ctx, const bt2g_pe_policy *pol, const int64_t *pairs, uint64_t n, int32_t *out) {
	if(!ctx) return -1;
	if(!pol || !pairs || !out || pol->pol < 1 || pol->pol > 4) { ctx->err = "bt2g_pe_classify: bad argument"; return -1; }
	if(n == 0) return 0;
	BT2G_CUDA_TRY(ctx, cudaSetDevice(ctx->device));
	DBuf dp, dout;
	BT2G_CUDA_TRY(ctx, dp.alloc(n * 48)); BT2G_CUDA_TRY(ctx, dout.alloc(n * 4));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(dp.p, pairs, n * 48, cudaMemcpyHostToDevice, ctx->stream));
	launch_pe_classify(*pol, dp.as<int64_t>(), n, dout.as<int32_t>(), ctx->stream);
	BT2G_CUDA_TRY(ctx, cudaGetLastError());
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(out, dout.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
	return 0;
}

int bt2g_extend_exact(bt2g_ctx *ctx, const bt2g_reads *reads, const bt2g_seed_plan *plan, const uint64_t *ranges, uint8_t *out) {
	REQUIRE_LOADED(ctx);
	if(!reads || !plan || !ranges || !out || plan->max_seeds <= 0 || plan->seed_len <= 0) return -1;
	uint64_t n = reads->n_reads;
	if(n == 0) return 0;
	DBuf dseq, dqual, doff, dint, doffs, drng, dout;
	int rc = uploadReads(ctx, reads, dseq, dqual, doff, false);
	if(rc) return rc;
	const uint64_t nr = n * 2ull * plan->max_seeds;
	BT2G_CUDA_TRY(ctx, dint.alloc(n * 4)); BT2G_CUDA_TRY(ctx, doffs.alloc(n * 4));
	BT2G_CUDA_TRY(ctx, drng.alloc(nr * 32)); BT2G_CUDA_TRY(ctx, dout.alloc(nr * 2));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(dint.p, plan->interval, n * 4, cudaMemcpyHostToDevice, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(doffs.p, plan->offset, n * 4, cudaMemcpyHostToDevice, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(drng.p, ranges, nr * 32, cudaMemcpyHostToDevice, ctx->stream));
	DISPATCH(ctx, launch_extend<uint32_t>(bt2g_dev_index<uint32_t>(ctx), dseq.as<uint8_t>(), doff.as<uint64_t>(), n, plan->seed_len, plan->max_seeds, dint.as<int32_t>(), doffs.as<int32_t>(), drng.as<uint64_t>(), dout.as<uint8_t>(), ctx->stream),
	              launch_extend<uint64_t>(bt2g_dev_index<uint64_t>(ctx), dseq.as<uint8_t>(), doff.as<uint64_t>(), n, plan->seed_len, plan->max_seeds, dint.as<int32_t>(), doffs.as<int32_t>(), drng.as<uint64_t>(), dout.as<uint8_t>(), ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaGetLastError());
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(out, dout.p, nr * 2, cudaMemcpyDeviceToHost, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
	return 0;
}

// ---- K2 ------------------------------------------------------------------------------------
int bt2g_resolve(bt2g_ctx *ctx, const uint64_t *rows, const uint32_t *hitlen, uint64_t n, int rejectStraddle,
                 uint64_t *joined, uint64_t *tidx, uint64_t *textoff, uint64_t *tlen, uint8_t *flags) {
	REQUIRE_LOADED(ctx);
	if(!rows) return -1;
	if(n == 0) return 0;
	DBuf dr, dh, dj, dti, dto, dtl, dfl;
	BT2G_CUDA_TRY(ctx, dr.alloc(n * 8));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(dr.p, rows, n * 8, cudaMemcpyHostToDevice, ctx->stream));
	if(hitlen) { BT2G_CUDA_TRY(ctx, dh.alloc(n * 4)); BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(dh.p, hitlen, n * 4, cudaMemcpyHostToDevice, ctx->stream)); }
	if(joined) BT2G_CUDA_TRY(ctx, dj.alloc(n * 8));
	if(tidx) BT2G_CUDA_TRY(ctx, dti.alloc(n * 8));
	if(textoff) BT2G_CUDA_TRY(ctx, dto.alloc(n * 8));
	if(tlen) BT2G_CUDA_TRY(ctx, dtl.alloc(n * 8));
	if(flags) BT2G_CUDA_TRY(ctx, dfl.alloc(n));
	DBuf dnext;
	BT2G_CUDA_TRY(ctx, dnext.alloc(8));
	int sms = 148; cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
	DISPATCH(ctx, launch_resolve2<uint32_t>(bt2g_dev_index<uint32_t>(ctx), dr.as<uint64_t>(), dh.as<uint32_t>(), n, nullptr, rejectStraddle, dj.as<uint64_t>(), dti.as<uint64_t>(), dto.as<uint64_t>(), dtl.as<uint64_t>(), dfl.as<uint8_t>(), dnext.as<unsigned long long>(), sms, ctx->stream, nullptr),
	              launch_resolve2<uint64_t>(bt2g_dev_index<uint64_t>(ctx), dr.as<uint64_t>(), dh.as<uint32_t>(), n, nullptr, rejectStraddle, dj.as<uint64_t>(), dti.as<uint64_t>(), dto.as<uint64_t>(), dtl.as<uint64_t>(), dfl.as<uint8_t>(), dnext.as<unsigned long long>(), sms, ctx->stream, nullptr));
	BT2G_CUDA_TRY(ctx, cudaGetLastError());
	if(joined) BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(joined, dj.p, n * 8, cudaMemcpyDeviceToHost, ctx->stream));
	if(tidx) BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(tidx, dti.p, n * 8, cudaMemcpyDeviceToHost, ctx->stream));
	if(textoff) BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(textoff, dto.p, n * 8, cudaMemcpyDeviceToHost, ctx->stream));
	if(tlen) BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(tlen, dtl.p, n * 8, cudaMemcpyDeviceToHost, ctx->stream));
	if(flags) BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(flags, dfl.p, n, cudaMemcpyDeviceToHost, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
	return 0;
}

int bt2g_get_stretch(bt2g_ctx *ctx, const uint64_t *tidx, const int64_t *off, const int32_t *count, uint64_t n,
                     int32_t stride, uint8_t *out) {
	REQUIRE_LOADED(ctx);
	if(!ctx->info.has_ref) { ctx->err = "packed reference (.3/.4) not loaded"; return -1; }
	if(n == 0) return 0;
	DBuf dt, dof, dc, dout;
	BT2G_CUDA_TRY(ctx, dt.alloc(n * 8)); BT2G_CUDA_TRY(ctx, dof.alloc(n * 8)); BT2G_CUDA_TRY(ctx, dc.alloc(n * 4));
	BT2G_CUDA_TRY(ctx, dout.alloc(n * (uint64_t)stride));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(dt.p, tidx, n * 8, cudaMemcpyHostToDevice, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(dof.p, off, n * 8, cudaMemcpyHostToDevice, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(dc.p, count, n * 4, cudaMemcpyHostToDevice, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaMemsetAsync(dout.p, 4, n * (uint64_t)stride, ctx->stream));
	DISPATCH(ctx, launch_get_stretch<uint32_t>(bt2g_dev_index<uint32_t>(ctx), dt.as<uint64_t>(), dof.as<int64_t>(), dc.as<int32_t>(), n, stride, dout.as<uint8_t>(), ctx->stream),
	              launch_get_stretch<uint64_t>(bt2g_dev_index<uint64_t>(ctx), dt.as<uint64_t>(), dof.as<int64_t>(), dc.as<int32_t>(), n, stride, dout.as<uint8_t>(), ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaGetLastError());
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(out, dout.p, n * (uint64_t)stride, cudaMemcpyDeviceToHost, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
	return 0;
}

// ---- K3 ------------------------------------------------------------------------------------
// Scoring::initPens (scoring.h:103-132) for COST_MODEL_QUAL mismatches, constant N penalty
void bt2g_scoring_default(bt2g_scoring *sc, int local) {
	memset(sc, 0, sizeof(*sc));
	sc->match_bonus = local ? 2 : 0;
	sc->rdgap_const = 5; sc->rdgap_linear = 3; sc->rfgap_const = 5; sc->rfgap_linear = 3;
	sc->gapbar = 4;
	sc->local = local ? 1 : 0;
	for(int q = 0; q < 64; q++) {
		int ii = q < 40 ? q : 40;
		float frac = (float)ii / 40.0f;
		sc->mmpen[q] = (uint8_t)(2 + (int)(frac * (6 - 2)));
		sc->npen[q] = 1;
	}
	sc->nceil_const = 0.0; sc->nceil_linear = (double)0.15f;
}

int bt2g_set_scoring(bt2g_ctx *ctx, const bt2g_scoring *sc) {
	if(!ctx || !sc) return -1;
	if(sc->gapbar < 1) { ctx->err = "gapbar must be >= 1"; return -1; }
	ctx->scoring = *sc;
	return 0;
}

int bt2g_set_extend_mode(bt2g_ctx *ctx, int through_text) {
	if(!ctx) return -1;
	ctx->extendText = through_text ? 1 : 0;
	return 0;
}

int bt2g_set_dp_mode(bt2g_ctx *ctx, int cap) {
	if(!ctx || cap < 0 || cap > 3) return -1;
	ctx->dpModeCap = cap;
	return 0;
}

int bt2g_dp_extend(bt2g_ctx *ctx, const bt2g_reads *reads, const bt2g_dp_problem *probs, uint64_t n,
                   int32_t maxCands, int32_t maxAlns, int32_t maxOps,
                   bt2g_dp_summary *summ, bt2g_dp_cand *cands, bt2g_dp_aln *alns, uint8_t *ops) {
	REQUIRE_LOADED(ctx);
	if(!ctx->info.has_ref) { ctx->err = "packed reference (.3/.4) not loaded"; return -1; }
	if(!reads || !reads->qual || !probs || !summ || !cands || !alns || !ops) { ctx->err = "null argument"; return -1; }
	if(ctx->scoring.gapbar < 1) bt2g_scoring_default(&ctx->scoring, 0);
	if(n == 0) return 0;
	if(maxCands < 1 || maxAlns < 1 || maxOps < 1) return -1;
	// shape of the batch
	int maxCol = 1, maxLen = 1;
	int64_t minMinsc = 0;
	for(uint64_t i = 0; i < n; i++) {
		if(probs[i].minsc < minMinsc) minMinsc = probs[i].minsc;
		int64_t nc = probs[i].refr - probs[i].refl + 1;
		if(nc > maxCol) maxCol = (int)nc;
		if(probs[i].read_idx >= reads->n_reads) { ctx->err = "read_idx out of range"; return -1; }
		int len = (int)(reads->off[probs[i].read_idx + 1] - reads->off[probs[i].read_idx]);
		if(len > maxLen) maxLen = len;
	}
	if(maxLen > 512) { ctx->err = "reads longer than 512 are not supported by the DP kernel"; return -1; }
	maxCol += 1;                              // local mode keeps one extra reference character
	if(maxCol > 8192) { ctx->err = "DP window wider than 8192 columns"; return -1; }
	DBuf dseq, dqual, doff, dprob, dcodes, dlast, dsumm, dcand, daln, dops, draw;
	int rc = uploadReads(ctx, reads, dseq, dqual, doff, true);
	if(rc) return rc;
	DpLaunch L;
	L.n = n; L.nDev = nullptr; L.maxCol = maxCol;
	{
		int sms = 148; cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
		uint64_t want = (uint64_t)sms * 24;      // 24 resident warps per SM
		L.numSlots = ((n < want ? n : want) + 3) / 4 * 4;
	} L.maxCands = maxCands; L.maxAlns = maxAlns; L.maxOps = maxOps;
	L.packed = ctx->scoring.local ? 0 : dp_kernel_mode(ctx->scoring, minMinsc, maxLen, ctx->dpModeCap);
	L.codeStride = dp_code_stride(maxCol, maxLen, L.packed);
	BT2G_CUDA_TRY(ctx, dprob.alloc(n * sizeof(bt2g_dp_problem)));
	if(L.packed == 3) {
		L.chunk = dp_chunk_problems(L.codeStride, n);
		BT2G_CUDA_TRY(ctx, dcodes.alloc(L.chunk * L.codeStride));
	} else {
		BT2G_CUDA_TRY(ctx, dcodes.alloc(L.numSlots * L.codeStride * (L.packed ? 2 : 1)));
	}
	BT2G_CUDA_TRY(ctx, dlast.alloc(L.numSlots * (uint64_t)maxCol * 4));
	L.maxRaw = maxCands * 4 < 1024 ? 1024 : maxCands * 4;
	BT2G_CUDA_TRY(ctx, draw.alloc(L.numSlots * (uint64_t)L.maxRaw * 8));
	L.rawKeys = draw.as<uint64_t>();
	BT2G_CUDA_TRY(ctx, dsumm.alloc(n * sizeof(bt2g_dp_summary)));
	BT2G_CUDA_TRY(ctx, dcand.alloc(n * (uint64_t)maxCands * sizeof(bt2g_dp_cand)));
	BT2G_CUDA_TRY(ctx, daln.alloc(n * (uint64_t)maxAlns * sizeof(bt2g_dp_aln)));
	BT2G_CUDA_TRY(ctx, dops.alloc(n * (uint64_t)maxAlns * maxOps));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(dprob.p, probs, n * sizeof(bt2g_dp_problem), cudaMemcpyHostToDevice, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaMemsetAsync(dcand.p, 0, dcand.bytes, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaMemsetAsync(daln.p, 0, daln.bytes, ctx->stream));
	L.seq = dseq.as<uint8_t>(); L.qual = dqual.as<uint8_t>(); L.roff = doff.as<uint64_t>();
	L.probs = dprob.as<bt2g_dp_problem>(); L.codes = dcodes.as<uint8_t>(); L.lastH = dlast.as<int32_t>();
	L.summ = dsumm.as<bt2g_dp_summary>(); L.cands = dcand.as<bt2g_dp_cand>(); L.alns = daln.as<bt2g_dp_aln>(); L.ops = dops.as<uint8_t>();
	int lrc;
	if(ctx->scoring.local) {
		if(ctx->info.off_size == 4) lrc = launch_dp_local<uint32_t>(bt2g_dev_index<uint32_t>(ctx), ctx->scoring, L, maxLen, ctx->stream);
		else lrc = launch_dp_local<uint64_t>(bt2g_dev_index<uint64_t>(ctx), ctx->scoring, L, maxLen, ctx->stream);
	} else {
		if(ctx->info.off_size == 4) lrc = launch_dp_e2e<uint32_t>(bt2g_dev_index<uint32_t>(ctx), ctx->scoring, L, maxLen, ctx->stream);
		else lrc = launch_dp_e2e<uint64_t>(bt2g_dev_index<uint64_t>(ctx), ctx->scoring, L, maxLen, ctx->stream);
	}
	if(lrc) { ctx->err = "DP launch rejected"; return -1; }
	BT2G_CUDA_TRY(ctx, cudaGetLastError());
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(summ, dsumm.p, dsumm.bytes, cudaMemcpyDeviceToHost, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(cands, dcand.p, dcand.bytes, cudaMemcpyDeviceToHost, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(alns, daln.p, daln.bytes, cudaMemcpyDeviceToHost, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaMemcpyAsync(ops, dops.p, dops.bytes, cudaMemcpyDeviceToHost, ctx->stream));
	BT2G_CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
	return 0;
}

} // extern "C"
