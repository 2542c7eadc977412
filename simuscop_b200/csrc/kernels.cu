// kernels.cu -- sm_100a kernels of the read-generation hot path.
//
//   pack_kernel      ASCII haplotype strings -> 2-bit codes + non-ACGT mask (HBM layout)
//   census_kernel    Segment::yieldReads' failCount > 1000 rule for the bins that can fail
//   locate_kernel    first bin of every output tile of a batch
//   generate_kernel  the fused per-pair loop: fragment sampling (Segment.cpp:743-763),
//                    Profile::predict for both mates (Profile.cpp:1586-1701), reverse
//                    complement (Segment.cpp:819-821), FASTQ formatting (Segment.cpp:808-832)
//                    and ordered dense output (SeqWriter.cpp:49-54 order) in one launch.
//
// Mapping: one warp per pair, one lane per sequencing cycle (5 chunks of 32 lanes at RL 151);
// a CTA of 16 warps owns a tile of 32 consecutive pairs; records are formatted into shared
// memory staging and copied out with 16-byte stores at the exact byte offset obtained from a
// decoupled look-back scan over tiles, so the slab is byte-identical to the reference's file.
#include <cuda_runtime.h>
#include <cstdint>

#include "bam.cuh"
#include "device_types.h"
#include "gz.h"
#include "kernels.h"
#include "philox.cuh"

namespace ssc {

// ----------------------------------------------------------------------------------------
// draw -> value maps (ThreadPool::randomDouble / randomInteger, lib/threadpool/ThreadPool.cpp:203-212)
// ----------------------------------------------------------------------------------------
__device__ __forceinline__ double dev_draw_real(uint32_t u, double start, double end) {
	double frac = __dmul_rn((double)u, 2.3283064365386962890625e-10);  // u / 2^32, exact
	return __dadd_rn(start, __dmul_rn(__dsub_rn(end, start), frac));
}

// randomInteger(spos, epos+1): needs FP64 (spos + span*u/2^32 can round up), one per fragment attempt
__device__ __forceinline__ long long dev_draw_pos(uint32_t u, int spos, int epos) {
	double frac = __dmul_rn((double)u, 2.3283064365386962890625e-10);
	double v = __dadd_rn((double)spos, __dmul_rn((double)((long long)epos + 1 - spos), frac));
	return (long long)v;
}

#define SSC_ZF 2.2204e-16

__device__ __forceinline__ int dev_rand_indx_f64(const double* __restrict__ cdf, int ac, uint32_t u) {
	double r = dev_draw_real(u, SSC_ZF, 1.0);
	for (int k = 0; k < ac; k++)
		if (r <= cdf[k]) return k;
	return ac - 1;
}

// compressed CDF: sym[#{i : T[i] < u}], T ascending, last T = 0xFFFFFFFF
template <typename TP, typename SP>
__device__ __forceinline__ int compressed_lookup(TP T, SP sym, int n, uint32_t u) {
	int lo = 0, len = n - 1;  // the sentinel is never < u
	while (len > 0) {
		int half = len >> 1;
		if (T[lo + half] < u) { lo += half + 1; len -= half + 1; } else len = half;
	}
	return (int)sym[lo];
}

// ----------------------------------------------------------------------------------------
// pack_kernel: one thread per 32 bases.  The first and last word of an append may be shared
// with the neighbouring append (appends are stream-ordered), so edges are merged.
// ----------------------------------------------------------------------------------------
__global__ void pack_kernel(const uint8_t* __restrict__ ascii, uint64_t n, uint64_t firstBase,
                            uint32_t* __restrict__ hap2, uint32_t* __restrict__ hapN, const int8_t* __restrict__ lut) {
	uint64_t firstGroup = firstBase >> 5;
	uint64_t lastGroup = (firstBase + n - 1) >> 5;
	uint64_t group = firstGroup + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (group > lastGroup) return;
	uint64_t g0 = group << 5;
	uint32_t lo = 0, hi = 0, nm = 0, valid = 0;
#pragma unroll 8
	for (int i = 0; i < 32; i++) {
		uint64_t g = g0 + i;
		if (g >= firstBase && g < firstBase + n) {
			int code = lut[ascii[g - firstBase]];
			valid |= 1u << i;
			if (code > 3) { nm |= 1u << i; code = 0; }
			if (i < 16) lo |= (uint32_t)code << (2 * i); else hi |= (uint32_t)code << (2 * (i - 16));
		}
	}
	if (valid == 0xFFFFFFFFu) {
		hap2[2 * group] = lo; hap2[2 * group + 1] = hi; hapN[group] = nm;
	} else {
		uint32_t vlo = 0, vhi = 0;
		for (int i = 0; i < 16; i++) {
			if (valid & (1u << i)) vlo |= 3u << (2 * i);
			if (valid & (1u << (i + 16))) vhi |= 3u << (2 * i);
		}
		hap2[2 * group] = (hap2[2 * group] & ~vlo) | lo;
		hap2[2 * group + 1] = (hap2[2 * group + 1] & ~vhi) | hi;
		hapN[group] = (hapN[group] & ~valid) | nm;
	}
}

// ----------------------------------------------------------------------------------------
// poke_kernel / unpack_kernel: single-base overwrites of the packed store (SNP / SNV alleles on reference-built
// haplotypes, Segment.cpp:233-311) and the decoder back to ASCII (diagnostic)
// ----------------------------------------------------------------------------------------
__global__ void poke_kernel(uint32_t* __restrict__ hap2, uint32_t* __restrict__ hapN, const int64_t* __restrict__ pos,
                            const uint8_t* __restrict__ chars, int64_t n, const int8_t* __restrict__ lut) {
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const uint64_t g = (uint64_t)pos[i] + SSC_GPAD;
	int code = lut[chars[i]];
	const uint32_t nbit = 1u << (g & 31);
	if (code > 3) { atomicOr(&hapN[g >> 5], nbit); code = 0; } else atomicAnd(&hapN[g >> 5], ~nbit);
	const uint32_t sh = (uint32_t)(g & 15) * 2u;
	atomicAnd(&hap2[g >> 4], ~(3u << sh));
	atomicOr(&hap2[g >> 4], (uint32_t)code << sh);
}

__global__ void unpack_kernel(const uint32_t* __restrict__ hap2, const uint32_t* __restrict__ hapN, uint64_t firstBase, uint64_t n,
                              uint32_t baseChars, uint8_t* __restrict__ out) {
	const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const uint64_t g = firstBase + i;
	const uint32_t code = (hap2[g >> 4] >> ((g & 15) * 2)) & 3u;
	const bool isN = (hapN[g >> 5] >> (g & 31)) & 1u;
	out[i] = isN ? (uint8_t)'N' : (uint8_t)(baseChars >> (8 * code));
}

// ----------------------------------------------------------------------------------------
// gc_census_kernel: G/C and non-ACGT base counts of store intervals (one warp per interval),
// the device half of Segment::getWeightedLength -> calculateGCPercent (Segment.cpp:567-624,
// MyDefine.cpp:279-303).  A lane takes groups of 32 bases: two data words + one mask word.
// gcCodes: bit k set iff 2-bit code k is G or C in the profile's base order.
// ----------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t spread16(uint32_t x) {   // bit i of the low half -> bit 2i
	x &= 0xffffu;
	x = (x | (x << 8)) & 0x00FF00FFu;
	x = (x | (x << 4)) & 0x0F0F0F0Fu;
	x = (x | (x << 2)) & 0x33333333u;
	x = (x | (x << 1)) & 0x55555555u;
	return x;
}
__device__ __forceinline__ uint32_t gc_fields(uint32_t w, uint32_t gcCodes) {   // bit 2i set iff base i of the word is G or C
	const uint32_t lo = w & 0x55555555u, hi = (w >> 1) & 0x55555555u;
	uint32_t ind = 0;
	if (gcCodes & 1u) ind |= ~lo & ~hi;
	if (gcCodes & 2u) ind |= lo & ~hi;
	if (gcCodes & 4u) ind |= ~lo & hi;
	if (gcCodes & 8u) ind |= lo & hi;
	return ind & 0x55555555u;
}
__global__ void gc_census_kernel(const uint32_t* __restrict__ hap2, const uint32_t* __restrict__ hapN,
                                 const int64_t* __restrict__ starts, const int32_t* __restrict__ lens, int64_t n,
                                 uint32_t gcCodes, int32_t* __restrict__ gc, int32_t* __restrict__ nn) {
	const int lane = threadIdx.x & 31;
	const int64_t i = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
	if (i >= n) return;
	const int64_t a = starts[i] + SSC_GPAD, b = a + lens[i];
	int cgc = 0, cn = 0;
	for (int64_t g = (a >> 5) + lane; (g << 5) < b; g += 32) {
		const int64_t g0 = g << 5;
		const int lo = a > g0 ? (int)(a - g0) : 0, hi = b < g0 + 32 ? (int)(b - g0) : 32;
		uint32_t m = hi >= 32 ? 0xFFFFFFFFu : ((1u << hi) - 1u);
		m &= ~((1u << lo) - 1u);
		const uint32_t nm = hapN[g] & m;
		cn += __popc(nm);
		const uint32_t v = m & ~nm;                                   // valid ACGT bases (non-ACGT are stored as code 0)
		cgc += __popc(gc_fields(hap2[2 * g], gcCodes) & spread16(v)) + __popc(gc_fields(hap2[2 * g + 1], gcCodes) & spread16(v >> 16));
	}
#pragma unroll
	for (int d = 16; d > 0; d >>= 1) { cgc += __shfl_xor_sync(0xffffffffu, cgc, d); cn += __shfl_xor_sync(0xffffffffu, cn, d); }
	if (lane == 0) { gc[i] = cgc; nn[i] = cn; }
}

// ----------------------------------------------------------------------------------------
// one fragment attempt (Segment.cpp:743-762): start position, wanted length, clipped length
// ----------------------------------------------------------------------------------------
template <bool FP64>
__device__ __forceinline__ void frag_attempt(const DevTables& t, const uint32_t* isizeT, const uint16_t* isizeSym,
                                             uint64_t seed, uint64_t pair, uint32_t attempt,
                                             int64_t hap_base, int64_t contig_end, int spos, int epos,
                                             long long& pos, int& len, uint32_t& strandWord) {
	u32x4 b = draw_block(seed, pair, 0, STREAM_FRAG, 0, attempt);
	pos = dev_draw_pos(b.x, spos, epos);
	long long want;
	if (!t.paired) want = (long long)epos - spos + 1;
	else if (t.nIsize > 0) {
		if (FP64) want = t.minIS + dev_rand_indx_f64(t.f_isize, t.f_nIsize, b.y);
		else want = t.minIS + compressed_lookup(isizeT, isizeSym, t.nIsize, b.y);
	} else want = t.fixedInsert;
	long long avail = contig_end - (hap_base + pos);
	long long l = want < avail ? want : avail;
	if (l < 0) l = 0;
	len = (int)(l > 0x7fffffff ? 0x7fffffff : l);
	strandWord = b.z;
}

// census: one thread per risky bin, sequential like the reference's while(n > 0) loop.
template <bool FP64>
__global__ void census_kernel(DevTables t, const CensusBin* __restrict__ bins, int nBins, uint64_t seed,
                              uint16_t* __restrict__ riskyAttempt, int32_t* __restrict__ emitted) {
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= nBins) return;
	CensusBin b = bins[i];
	int fails = 0;
	int ord = 0;
	for (; ord < b.planned; ord++) {
		uint32_t a = 0;
		bool ok = false;
		while (true) {
			long long pos; int len; uint32_t sw;
			frag_attempt<FP64>(t, t.isizeT, t.isizeSym, seed, (uint64_t)(b.plan_base + ord), a,
			                   b.hap_base, b.contig_end, b.spos, b.epos, pos, len, sw);
			if (len >= t.RL) { ok = true; break; }
			fails++;
			if (fails > 1000) break;
			a++;
		}
		if (!ok) break;
		riskyAttempt[b.risky_base + ord] = (uint16_t)a;
	}
	emitted[i] = ord;
}

__global__ void locate_kernel(const int64_t* __restrict__ emitBase, int64_t nBins, int64_t emitLo, int tilePairs,
                              int nTiles, int32_t* __restrict__ tileStartBin) {
	int tIdx = blockIdx.x * blockDim.x + threadIdx.x;
	if (tIdx >= nTiles) return;
	int64_t e = emitLo + (int64_t)tIdx * tilePairs;
	// largest b with emitBase[b] <= e
	int64_t lo = 0, hi = nBins;  // emitBase[0] = 0 <= e < emitBase[nBins]
	while (hi - lo > 1) {
		int64_t mid = (lo + hi) >> 1;
		if (emitBase[mid] <= e) lo = mid; else hi = mid;
	}
	tileStartBin[tIdx] = (int32_t)lo;
}

// ----------------------------------------------------------------------------------------
// generate_kernel
// ----------------------------------------------------------------------------------------
static constexpr int HDR_MAX = 96;    // "@popu#chr#" + digits, enforced by the host (name_len <= 64)
static constexpr int EV_MAX = 32;     // indel events per read
#define ST_A (1ull << 62)
#define ST_P (2ull << 62)
#define ST_MASK (3ull << 62)

struct GenCfg {
	static constexpr int SRC_CAP = GEN_NCH * 32 + 96;                   // longest read the scratch holds
	static constexpr int REC_CAP = HDR_MAX + 2 * SRC_CAP + 8;
	static constexpr int STAGE_CAP = ((GEN_PPW * REC_CAP + 15) / 16) * 16 + 16;
};

struct SmemLayout {
	int sub, isizeT, isizeSym, insT, insSym, delT, delSym, src, ev, insb, stage, total;
};

__host__ __device__ inline SmemLayout smem_layout(int nSubTotal, int nIsize, int nIns, int nDel) {
	SmemLayout L;
	int o = 0;
	L.sub = o; o += nSubTotal * 16;
	L.isizeT = o; o += (nIsize * 4 + 15) / 16 * 16;
	L.isizeSym = o; o += (nIsize * 2 + 15) / 16 * 16;
	L.insT = o; o += (nIns * 4 + 15) / 16 * 16;
	L.insSym = o; o += (nIns * 2 + 15) / 16 * 16;
	L.delT = o; o += (nDel * 4 + 15) / 16 * 16;
	L.delSym = o; o += (nDel * 2 + 15) / 16 * 16;
	L.src = o; o += GEN_WARPS * GenCfg::SRC_CAP;
	L.ev = o; o += GEN_WARPS * EV_MAX * 4;
	L.insb = o; o += GEN_WARPS * 128;
	L.stage = o; o += GEN_WARPS * 2 * GenCfg::STAGE_CAP;
	L.total = o;
	return L;
}

__device__ __forceinline__ int ndigits(uint32_t v) {
	int n = 1;
	if (v >= 10u) n = 2;
	if (v >= 100u) n = 3;
	if (v >= 1000u) n = 4;
	if (v >= 10000u) n = 5;
	if (v >= 100000u) n = 6;
	if (v >= 1000000u) n = 7;
	if (v >= 10000000u) n = 8;
	if (v >= 100000000u) n = 9;
	if (v >= 1000000000u) n = 10;
	return n;
}

__device__ __forceinline__ uint32_t pow10u(int p) {
	uint32_t r = 1;
	for (int i = 0; i < p; i++) r *= 10u;
	return r;
}

// "@popu#chr#<posmod>#<fragCount>[/mate]\n"  (Segment.cpp:780, 809, 824); returns the length
__device__ __forceinline__ int write_header(uint8_t* dst, const char* __restrict__ name, int nameLen,
                                            uint32_t posmod, uint32_t fragCount, int mateTag, int lane) {
	int nd1 = ndigits(posmod), nd2 = ndigits(fragCount);
	int H = nameLen + nd1 + 1 + nd2 + (mateTag ? 2 : 0) + 1;
	for (int i = lane; i < H; i += 32) {
		uint8_t ch;
		if (i < nameLen) ch = (uint8_t)name[i];
		else {
			int k = i - nameLen;
			if (k < nd1) ch = (uint8_t)('0' + (posmod / pow10u(nd1 - 1 - k)) % 10u);
			else if (k == nd1) ch = '#';
			else {
				int k2 = k - nd1 - 1;
				if (k2 < nd2) ch = (uint8_t)('0' + (fragCount / pow10u(nd2 - 1 - k2)) % 10u);
				else {
					int k3 = k2 - nd2;
					if (mateTag) ch = (k3 == 0) ? '/' : (k3 == 1) ? (uint8_t)('0' + mateTag) : '\n';
					else ch = '\n';
				}
			}
		}
		dst[i] = ch;
	}
	return H;
}

// copy a warp's staged bytes (shared, 16-byte aligned start) to an arbitrary global byte offset
// with 16-byte stores; the shared side is re-aligned with funnel shifts.
__device__ __forceinline__ void copy_out(const uint8_t* sm, int len, uint8_t* g, int lane) {
	if (len <= 0) return;
	int head = (int)((16u - (uint32_t)((uintptr_t)g & 15u)) & 15u);
	if (head > len) head = len;
	if (lane < head) g[lane] = sm[lane];
	int nvec = (len - head) >> 4;
	const uint32_t* sm32 = (const uint32_t*)sm;
	int r = head & 3;
	int q0 = head >> 2;
	uint4* gv = (uint4*)(g + head);
	for (int v = lane; v < nvec; v += 32) {
		int q = q0 + 4 * v;
		uint32_t w0 = sm32[q], w1 = sm32[q + 1], w2 = sm32[q + 2], w3 = sm32[q + 3], w4 = sm32[q + 4];
		uint4 o;
		o.x = __funnelshift_r(w0, w1, 8 * r);
		o.y = __funnelshift_r(w1, w2, 8 * r);
		o.z = __funnelshift_r(w2, w3, 8 * r);
		o.w = __funnelshift_r(w3, w4, 8 * r);
		gv[v] = o;
	}
	int t0 = head + (nvec << 4);
	if (lane < len - t0) g[t0 + lane] = sm[t0 + lane];
}

// ILV (interleaved output, PE): mate 2's record goes right behind mate 1's in the warp's first stage buffer, whose neighbour is
// its second one (2 x STAGE_CAP hold both mates of GEN_PPW pairs), and the one slab P.out1 receives mate 1, mate 2 of every
// pair in turn; off2, the second length of the look-back and P.out2 stay unused.
// BLOB (gzip output): a tile is one ticket of GEN_TILE_PAIRS = FG_CHUNK pairs, written as the fast kernel writes its tickets:
// file f's records to out_f + tile * P.blobPitch, the packed lengths len1 << 31 | len2 to P.tileState[tile] (no flags, no
// look-back), for the deflate kernel and pass 2, which writes result->bytes1/2.  The FASTQ bytes go to result->rawBytes.
// BAM (with BLOB; PE with ILV): unaligned BAM records (bam.cuh) instead of FASTQ; rawBytes counts their bytes.
template <bool K3, bool FP64, bool ILV, bool BLOB, bool BAM>
__global__ void __launch_bounds__(GEN_THREADS, 1) generate_kernel(const GenParams P) {
	extern __shared__ __align__(16) uint8_t smem[];
	const DevTables& t = P.t;
	const int lane = threadIdx.x & 31;
	const int warp = threadIdx.x >> 5;
	const int subSmemRows = (K3 && !FP64) ? t.nSub * (t.useCdf2 ? 2 : 1) : 0;
	const SmemLayout L = smem_layout(subSmemRows, FP64 ? 0 : t.nIsize, FP64 ? 0 : t.nInsLen, FP64 ? 0 : t.nDelLen);

	uint4* s_sub = (uint4*)(smem + L.sub);
	uint32_t* s_isizeT = (uint32_t*)(smem + L.isizeT);
	uint16_t* s_isizeSym = (uint16_t*)(smem + L.isizeSym);
	uint32_t* s_insT = (uint32_t*)(smem + L.insT);
	uint16_t* s_insSym = (uint16_t*)(smem + L.insSym);
	uint32_t* s_delT = (uint32_t*)(smem + L.delT);
	uint16_t* s_delSym = (uint16_t*)(smem + L.delSym);
	uint8_t* s_src = smem + L.src + warp * GenCfg::SRC_CAP;
	uint32_t* s_ev = (uint32_t*)(smem + L.ev) + warp * EV_MAX;
	uint8_t* s_insb = smem + L.insb + warp * 128;
	uint8_t* s_stage1 = smem + L.stage + (warp * 2 + 0) * GenCfg::STAGE_CAP;
	uint8_t* s_stage2 = smem + L.stage + (warp * 2 + 1) * GenCfg::STAGE_CAP;

	__shared__ unsigned long long s_warpLen[GEN_WARPS];   // len1 << 32 | len2
	__shared__ unsigned long long s_warpOff[GEN_WARPS];
	__shared__ unsigned long long s_tileBase;
	__shared__ int s_tile;
	__shared__ unsigned long long s_stats[4];              // bases, reads, pairs, hapBytes

	// ---- stage the tables
	if (!FP64) {
		for (int i = threadIdx.x; i < subSmemRows; i += GEN_THREADS) s_sub[i] = t.sub[i];
		for (int i = threadIdx.x; i < t.nIsize; i += GEN_THREADS) { s_isizeT[i] = t.isizeT[i]; s_isizeSym[i] = t.isizeSym[i]; }
		for (int i = threadIdx.x; i < t.nInsLen; i += GEN_THREADS) { s_insT[i] = t.insLenT[i]; s_insSym[i] = t.insLenSym[i]; }
		for (int i = threadIdx.x; i < t.nDelLen; i += GEN_THREADS) { s_delT[i] = t.delLenT[i]; s_delSym[i] = t.delLenSym[i]; }
	}
	if (threadIdx.x < 4) s_stats[threadIdx.x] = 0;
	const uint4* subTab = (K3 && !FP64) ? s_sub : t.sub;
	const uint32_t* qualT = t.qualT;
	const uint8_t* qualSym = t.qualSym;

	const int RL = t.RL, B = t.B, K = t.K;
	const int nMates = t.paired ? 2 : 1;
	const int chunksRL = (RL + 31) >> 5;
	unsigned long long accBases = 0, accReads = 0, accPairs = 0, accHap = 0;
	unsigned long long accRaw = 0;   // BLOB: FASTQ bytes of the CTA's tiles (thread 0)

	while (true) {
		__syncthreads();   // staging of the previous tile fully copied out; tables visible
		if (threadIdx.x == 0) s_tile = (int)atomicAdd(P.ticket, 1u);
		__syncthreads();
		const int tile = s_tile;
		if (tile >= P.nTiles) break;
		const int64_t tileFirst = P.emitLo + (int64_t)tile * GEN_TILE_PAIRS;
		const int sb = P.tileStartBin[tile];
		int off1 = 0, off2 = 0;

		for (int ip = 0; ip < GEN_PPW; ip++) {
			const int64_t e = tileFirst + warp * GEN_PPW + ip;
			if (e >= P.emitHi) break;
			// ---- bin of this pair: largest b >= sb with emitBase[b] <= e (at most 32 bins ahead)
			int64_t probe = sb + lane + 1;
			int64_t eb = (probe <= P.nBins) ? P.emitBase[probe] : 0x7fffffffffffffffLL;
			int b = sb + __popc(__ballot_sync(0xffffffffu, eb <= e));
			const DevBin bin = P.bins[b];
			const int ord = (int)(e - bin.emit_base);
			const uint64_t pair = (uint64_t)(bin.plan_base + ord);
			const uint32_t fragCount = (uint32_t)(bin.frag_base + ord + 1);
			uint32_t attempt = 0;
			if (bin.risky_base >= 0) attempt = P.riskyAttempt[bin.risky_base + ord];
			long long pos; int flen; uint32_t strandWord;
			frag_attempt<FP64>(t, s_isizeT, s_isizeSym, P.seed, pair, attempt, bin.hap_base, bin.contig_end,
			                   bin.spos, bin.epos, pos, flen, strandWord);
			const int64_t fstart = bin.hap_base + pos;
			const uint32_t posmod = (uint32_t)pos % bin.segsize;
			const bool seReverse = (!t.paired) && ((strandWord >> 31) != 0);   // randomInteger(0,2) != 0
			accPairs += 1;
			accHap += (unsigned long long)((flen + 3) / 4 + (flen + 7) / 8);

			for (int mate = 0; mate < nMates; mate++) {
				const bool rev = (mate == 1) || seReverse;
				// template window of the read: forward [fstart, +RL), reverse [fstart+flen-RL, +RL) read backwards
				const int64_t g0 = rev ? (fstart + flen - RL) : fstart;
				const int64_t w0 = g0 >> 4, m0 = g0 >> 5;
				// lane l keeps data word w0+l and mask word m0+l (RL <= 320 -> at most 21 / 11 words)
				uint32_t dataW = 0, maskW = 0;
				if (lane <= (int)(((g0 + RL - 1) >> 4) - w0)) dataW = __ldg(P.hap2 + w0 + lane);
				if (lane <= (int)(((g0 + RL - 1) >> 5) - m0)) maskW = __ldg(P.hapN + m0 + lane);

				// ---- phase A: one Philox block per cycle; indel tests at reference position j
				uint32_t x2[GEN_NCH], x3[GEN_NCH], insMask[GEN_NCH], delMask[GEN_NCH];
				uint32_t tcode = 0;   // 3 bits per chunk
				uint32_t anyEv = 0;
#pragma unroll
				for (int c = 0; c < GEN_NCH; c++) {
					insMask[c] = 0; delMask[c] = 0; x2[c] = 0; x3[c] = 0;
					if (c < chunksRL) {
						const int j = c * 32 + lane;
						u32x4 blk = draw_block(P.seed, pair, mate, STREAM_CYCLE, 0, (uint32_t)j);
						x2[c] = blk.z; x3[c] = blk.w;
						bool ins, del;
						if (FP64) {
							double p = dev_draw_real(blk.x, 0.0, 1.0);
							ins = (j < RL) && (p <= t.insertRate);
							double p2 = dev_draw_real(blk.y, 0.0, 1.0);
							del = (j < RL) && !ins && (p2 < t.delThresh);
						} else {
							ins = (j < RL) && t.insEnable && (blk.x <= t.insT);
							del = (j < RL) && !ins && t.delEnable && (blk.y <= t.delT);
						}
						insMask[c] = __ballot_sync(0xffffffffu, ins);
						delMask[c] = __ballot_sync(0xffffffffu, del);
						anyEv |= insMask[c] | delMask[c];
						{
							// template base j
							int jj = j < RL ? j : RL - 1;
							int64_t g = rev ? (g0 + (RL - 1 - jj)) : (g0 + jj);
							uint32_t dw = __shfl_sync(0xffffffffu, dataW, (int)((g >> 4) - w0));
							uint32_t mw = __shfl_sync(0xffffffffu, maskW, (int)((g >> 5) - m0));
							uint32_t code = (dw >> ((uint32_t)(g & 15) * 2)) & 3u;
							if (rev) code = (t.compLut >> (2 * code)) & 3u;
							if ((mw >> (uint32_t)(g & 31)) & 1u) code = 4u;
							tcode |= code << (3 * c);
						}
					}
				}

				// ---- phase B: apply indel events (rare) and build the source sequence
				int m = RL;
				if (anyEv == 0) {
#pragma unroll
					for (int c = 0; c < GEN_NCH; c++) {
						const int j = c * 32 + lane;
						if (c < chunksRL && j < RL) s_src[j] = (uint8_t)((tcode >> (3 * c)) & 7u);
					}
				} else {
					int nEv = 0, insTotal = 0, indelLength = 0, skipUntil = 0;
					bool tooMany = false;
#pragma unroll
					for (int c = 0; c < GEN_NCH; c++) {
						uint32_t mask = insMask[c] | delMask[c];
						while (mask) {
							const int bit = __ffs(mask) - 1;
							mask &= mask - 1;
							const int j = c * 32 + bit;
							if (j < skipUntil) continue;
							u32x4 lb = draw_block(P.seed, pair, mate, STREAM_LEN, 0, (uint32_t)j);
							if ((insMask[c] >> bit) & 1u) {
								int Lk = FP64 ? dev_rand_indx_f64(t.f_ins, t.f_nIns, lb.x)
								              : compressed_lookup(s_insT, s_insSym, t.nInsLen, lb.x);
								if (Lk > 0) {
									if (nEv >= EV_MAX || insTotal + Lk > 128) { tooMany = true; break; }
									// inserted bases: randomInteger(0, N-1) = floor(3*u/2^32): A, C or T (Profile.cpp:1563-1566)
									for (int i = lane; i < Lk; i += 32) {
										u32x4 bb = draw_block(P.seed, pair, mate, STREAM_INSBASE, i >> 2, (uint32_t)j);
										uint32_t wsel = (i & 3) == 0 ? bb.x : (i & 3) == 1 ? bb.y : (i & 3) == 2 ? bb.z : bb.w;
										s_insb[insTotal + i] = (uint8_t)__umulhi((uint32_t)(t.N - 1), wsel);
									}
									if (lane == 0) s_ev[nEv] = (uint32_t)j | ((uint32_t)Lk << 12) | ((uint32_t)insTotal << 20) | (1u << 31);
									nEv++; insTotal += Lk; indelLength += Lk;
								}
							} else {
								int Lk = FP64 ? dev_rand_indx_f64(t.f_del, t.f_nDel, lb.y)
								              : compressed_lookup(s_delT, s_delSym, t.nDelLen, lb.y);
								if (Lk > RL - j) Lk = RL - j;
								if (Lk > 0) {
									if (nEv >= EV_MAX) { tooMany = true; break; }
									if (lane == 0) s_ev[nEv] = (uint32_t)j | ((uint32_t)Lk << 12);
									nEv++; indelLength -= Lk; skipUntil = j + Lk;
								}
							}
						}
					}
					if (RL + indelLength < 50) { nEv = 0; indelLength = 0; }   // Profile.cpp:1627-1634
					m = RL + indelLength;
					if (tooMany || m > GenCfg::SRC_CAP) {
						if (lane == 0) atomicOr(&P.result->errorFlags, tooMany ? 4u : 2u);
						nEv = 0; m = RL;
					}
					__syncwarp();
					// template bases to their output positions
#pragma unroll
					for (int c = 0; c < GEN_NCH; c++) {
						const int j = c * 32 + lane;
						if (c < chunksRL && j < RL) {
							int shift = 0; bool dropped = false;
							for (int k = 0; k < nEv; k++) {
								const uint32_t ev = s_ev[k];
								const int ej = (int)(ev & 0xfffu), el = (int)((ev >> 12) & 0xffu);
								if (ev >> 31) { if (ej < j) shift += el; }
								else { if (j >= ej && j < ej + el) dropped = true; else if (j >= ej + el) shift -= el; }
							}
							if (!dropped) s_src[j + shift] = (uint8_t)((tcode >> (3 * c)) & 7u);
						}
					}
					// inserted bases go right after their template base (Profile.cpp:1647-1656)
					int cum = 0;
					for (int k = 0; k < nEv; k++) {
						const uint32_t ev = s_ev[k];
						const int ej = (int)(ev & 0xfffu), el = (int)((ev >> 12) & 0xffu);
						if (ev >> 31) {
							const int io = (int)((ev >> 20) & 0x7ffu);
							for (int i = lane; i < el; i += 32) s_src[ej + cum + 1 + i] = s_insb[io + i];
							cum += el;
						} else cum -= el;
					}
				}
				__syncwarp();

				// ---- record header
				uint8_t* stage = (mate == 0 || ILV) ? s_stage1 + off1 : s_stage2 + off2;
				// BAM: the header without a mate suffix, one byte in front of the name's place, so that its '@' lands in the fixed
				// fields and its line feed on the name's NUL (both overwritten below)
				const int H = BAM ? BAM_FIXED - 1 + write_header(stage + (BAM_FIXED - 1), P.names + bin.name_off, bin.name_len, posmod, fragCount, 0, lane)
				                  : write_header(stage, P.names + bin.name_off, bin.name_len, posmod, fragCount,
				                           t.paired ? (mate + 1) : 0, lane);
				if (!BAM && lane == 0) { stage[H + m] = '\n'; stage[H + m + 1] = '+'; stage[H + m + 2] = '\n'; stage[H + 2 * m + 3] = '\n'; }

				// ---- phase C: substitution + quality at output position j
				const uint32_t inv = (m > 1) ? (0xffffffffu / (uint32_t)m + 1u) : 0xffffffffu;
				const int chunksM = (m + 31) >> 5;
				const uint4* subM = subTab + ((mate == 1 && t.useCdf2) ? t.nSub : 0);
				const double* fsub = (mate == 1 && t.useCdf2) ? t.f_sub2 : t.f_sub1;
				uint32_t bch = 0, bq = 0;   // BAM: the base and quality characters of emit, stored by the whole warp
				auto emit = [&](int j, uint32_t u2, uint32_t u3) {
					const uint32_t cur = s_src[j];
					int row = 0; uint32_t bad = cur & 4u;
					if (K3) {
						const uint32_t p1 = j >= 1 ? s_src[j - 1] : 0u;
						const uint32_t p2 = j >= 2 ? s_src[j - 2] : 0u;
						bad |= (p1 | p2) & 4u;
						row = j >= 2 ? (int)(20u + 16u * p2 + 4u * p1 + cur) : j == 1 ? (int)(4u + 4u * p1 + cur) : (int)cur;
					} else {
						int valid = j + 1 < K ? j + 1 : K;
						int offset = 0, pw = 4, v = 0;
						for (int q = 1; q < valid; q++) { offset += pw; pw *= 4; }
						for (int q = valid - 1; q >= 0; q--) { const uint32_t cc = s_src[j - q]; bad |= cc & 4u; v = v * 4 + (int)(cc & 3u); }
						row = offset + v;
					}
					const int binIdx = (int)__umulhi((uint32_t)(j * B), inv);
					int call;
					if (bad) call = (cur & 4u) ? -1 : (int)cur;
					else if (FP64) call = dev_rand_indx_f64(fsub + ((size_t)row * B + binIdx) * 4, 4, u2);
					else {
						const uint4 s = subM[row * B + binIdx];
						call = (int)s.w + (u2 > s.x) + (u2 > s.y) + (u2 > s.z);
					}
					uint8_t ch, q;
					if (call < 0) { ch = 'N'; q = (uint8_t)(t.minQ + __umulhi(20u, u3)); }   // randomInteger(33, 53)
					else {
						ch = (uint8_t)((t.baseChars >> (8 * call)) & 0xffu);
						const int qrow = ((int)cur * 4 + call) * B + binIdx;
						if (FP64) q = (uint8_t)(t.minQ + dev_rand_indx_f64(t.f_qual + (size_t)qrow * t.Q, t.Q, u3));
						else {
							const uint32_t* qt = qualT + qrow * t.qualPitch;
							int k = 0;
							for (int s = t.qualPitch >> 1; s > 0; s >>= 1) if (qt[k + s - 1] < u3) k += s;
							q = qualSym[qrow * t.qualPitch + k];
						}
					}
					if (BAM) { bch = ch; bq = q; }
					else {
						stage[H + j] = ch;
						stage[H + m + 3 + j] = q;
					}
				};
				if (BAM) {
					// the 4-bit codes of a chunk are packed by the whole warp, every lane inside the read or not
#pragma unroll
					for (int c = 0; c < GEN_NCH; c++) {
						const int j = c * 32 + lane;
						if (c < chunksM) {
							if (j < m) {
								if (c < chunksRL) emit(j, x2[c], x3[c]);
								else { u32x4 blk = draw_block(P.seed, pair, mate, STREAM_CYCLE, 0, (uint32_t)j); emit(j, blk.z, blk.w); }
							}
							bam_put_base(stage + H + (j >> 1), stage + H + ((m + 1) >> 1) + j, j < m, bch, bq, lane);
						}
					}
					for (int c = GEN_NCH; c < chunksM; c++) {
						const int j = c * 32 + lane;
						if (j < m) { u32x4 blk = draw_block(P.seed, pair, mate, STREAM_CYCLE, 0, (uint32_t)j); emit(j, blk.z, blk.w); }
						bam_put_base(stage + H + (j >> 1), stage + H + ((m + 1) >> 1) + j, j < m, bch, bq, lane);
					}
					__syncwarp();                                   // the header's '@' and line feed are in place
					const uint32_t lReadName = (uint32_t)(H - BAM_FIXED), tail = bam_tail_bytes(lReadName, (uint32_t)m, (uint32_t)P.rgLen);
					if (lane == 0) stage[H - 1] = 0;
					bam_fixed(stage, lReadName, t.paired ? (mate == 0 ? BAM_FLAG_PE1 : BAM_FLAG_PE2) : BAM_FLAG_SE, (uint32_t)m,
					          (uint32_t)P.rgLen, lane);
					bam_read_group(stage + BAM_FIXED + tail - P.rgLen - 4, P.rg, P.rgLen, lane);
					off1 += BAM_FIXED + (int)tail;
				} else {
#pragma unroll
					for (int c = 0; c < GEN_NCH; c++) {
						const int j = c * 32 + lane;
						if (c < chunksM && j < m) {
							if (c < chunksRL) emit(j, x2[c], x3[c]);
							else { u32x4 blk = draw_block(P.seed, pair, mate, STREAM_CYCLE, 0, (uint32_t)j); emit(j, blk.z, blk.w); }
						}
					}
					for (int c = GEN_NCH; c < chunksM; c++) {
						const int j = c * 32 + lane;
						if (j < m) { u32x4 blk = draw_block(P.seed, pair, mate, STREAM_CYCLE, 0, (uint32_t)j); emit(j, blk.z, blk.w); }
					}
					if (mate == 0 || ILV) off1 += H + 2 * m + 4; else off2 += H + 2 * m + 4;
				}
				accBases += (unsigned long long)m;
				accReads += 1;
				__syncwarp();
			}
		}

		// ---- tile scan + decoupled look-back over tiles
		if (lane == 0) s_warpLen[warp] = ((unsigned long long)(uint32_t)off1 << 32) | (uint32_t)off2;
		__syncthreads();
		if (warp == 0) {
			unsigned long long v = lane < GEN_WARPS ? s_warpLen[lane] : 0ull;
			unsigned long long incl = v;
#pragma unroll
			for (int d = 1; d < 32; d <<= 1) {
				unsigned long long o = __shfl_up_sync(0xffffffffu, incl, d);
				if (lane >= d) incl += o;
			}
			if (lane < GEN_WARPS) s_warpOff[lane] = incl - v;
			const unsigned long long tot = __shfl_sync(0xffffffffu, incl, 31);
			// packed tile value: len1 in bits 31..61, len2 in bits 0..30
			const unsigned long long packed = ((tot >> 32) << 31) | (tot & 0x7fffffffull);
			volatile unsigned long long* st = P.tileState;
			unsigned long long excl = 0;
			if (BLOB) {
				if (lane == 0) { st[tile] = packed; accRaw += (tot >> 32) + (tot & 0xffffffffull); }
			} else if (tile == 0) {
				if (lane == 0) st[0] = ST_P | packed;
			} else {
				if (lane == 0) st[tile] = ST_A | packed;
				int pred = tile - 1;
				while (true) {
					const int idx = pred - lane;
					unsigned long long sv;
					do {
						sv = idx >= 0 ? st[idx] : ST_P;      // virtual inclusive prefix 0 before tile 0
					} while (__any_sync(0xffffffffu, (sv & ST_MASK) == 0ull));
					const unsigned pm = __ballot_sync(0xffffffffu, (sv & ST_MASK) == ST_P);
					const int firstP = pm ? (__ffs(pm) - 1) : 32;
					unsigned long long contrib = (lane <= firstP) ? (sv & ~ST_MASK) : 0ull;
#pragma unroll
					for (int d = 16; d > 0; d >>= 1) contrib += __shfl_xor_sync(0xffffffffu, contrib, d);
					excl += contrib;
					if (pm) break;
					pred -= 32;
				}
				if (lane == 0) st[tile] = ST_P | (excl + packed);
			}
			if (!BLOB && lane == 0) {
				s_tileBase = excl;
				if (tile == P.nTiles - 1) {
					const unsigned long long fin = excl + packed;
					P.result->bytes1 = fin >> 31;
					P.result->bytes2 = fin & 0x7fffffffull;
				}
			}
		}
		__syncthreads();
		if (BLOB) {
			// the blob and the bytes of a stored block must fit the pitch: the deflate kernel writes a member that coding would
			// expand as one stored block, at the same pitch
			const unsigned long long wo = s_warpOff[warp];
			const unsigned long long o1 = wo >> 32, o2 = wo & 0xffffffffull;
			const unsigned long long lim = P.blobPitch - (uint32_t)GZ_BGZF_STORED_EXTRA;
			if (o1 + (unsigned)off1 > lim || o2 + (unsigned)off2 > lim) {
				if (lane == 0) atomicOr(&P.result->errorFlags, 1u);
			} else {
				const size_t blob = (size_t)tile * P.blobPitch;
				copy_out(s_stage1, off1, P.out1 + blob + o1, lane);
				if (t.paired && !ILV) copy_out(s_stage2, off2, P.out2 + blob + o2, lane);
			}
		} else {
			const unsigned long long tb = s_tileBase;
			const unsigned long long wo = s_warpOff[warp];
			const unsigned long long g1 = (tb >> 31) + (wo >> 32);
			const unsigned long long g2 = (tb & 0x7fffffffull) + (wo & 0xffffffffull);
			if (g1 + (unsigned)off1 > P.cap1 || g2 + (unsigned)off2 > P.cap2) {
				if (lane == 0) atomicOr(&P.result->errorFlags, 1u);
			} else {
				copy_out(s_stage1, off1, P.out1 + g1, lane);
				if (t.paired && !ILV) copy_out(s_stage2, off2, P.out2 + g2, lane);
			}
		}
	}

	// ---- statistics
	if (lane == 0) {
		atomicAdd(&s_stats[0], accBases); atomicAdd(&s_stats[1], accReads);
		atomicAdd(&s_stats[2], accPairs); atomicAdd(&s_stats[3], accHap);
	}
	__syncthreads();
	if (threadIdx.x == 0) {
		atomicAdd(&P.result->bases, s_stats[0]); atomicAdd(&P.result->reads, s_stats[1]);
		atomicAdd(&P.result->pairs, s_stats[2]); atomicAdd(&P.result->hapBytes, s_stats[3]);
		if (BLOB) atomicAdd(&P.result->rawBytes, accRaw);
	}
}

// ----------------------------------------------------------------------------------------
// host-side launchers
// ----------------------------------------------------------------------------------------
template <bool K3, bool FP64, bool ILV, bool BLOB, bool BAM>
static cudaError_t launch_variant(const GenParams& P, int grid, size_t smemBytes, cudaStream_t stream) {
	auto kern = generate_kernel<K3, FP64, ILV, BLOB, BAM>;
	cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemBytes);
	if (e != cudaSuccess) return e;
	kern<<<grid, GEN_THREADS, smemBytes, stream>>>(P);
	return cudaGetLastError();
}

GenVariant choose_variant(const DevTables& t, bool fp64, int smemLimit) {
	GenVariant v;
	v.fp64 = fp64;
	v.k3 = (t.K == 3) && !fp64;
	v.smemBytes = 0;
	v.ok = t.RL <= GEN_NCH * 32;
	auto size = [&](bool k3) {
		int nSub = k3 ? t.nSub * (t.useCdf2 ? 2 : 1) : 0;
		int a = fp64 ? 0 : t.nIsize, b = fp64 ? 0 : t.nInsLen, c = fp64 ? 0 : t.nDelLen;
		return smem_layout(nSub, a, b, c).total;
	};
	if (fp64) { v.smemBytes = size(false); return v; }
	if (v.k3 && size(true) <= smemLimit) { v.smemBytes = size(true); return v; }
	v.k3 = false;
	v.smemBytes = size(false);
	if ((int)v.smemBytes > smemLimit) v.ok = false;
	return v;
}

template <bool ILV, bool BLOB, bool BAM = false>
static cudaError_t launch_tables(const GenParams& P, const GenVariant& v, int grid, cudaStream_t stream) {
	if (v.fp64) return launch_variant<false, true, ILV, BLOB, BAM>(P, grid, v.smemBytes, stream);
	if (v.k3) return launch_variant<true, false, ILV, BLOB, BAM>(P, grid, v.smemBytes, stream);
	return launch_variant<false, false, ILV, BLOB, BAM>(P, grid, v.smemBytes, stream);
}

cudaError_t launch_generate(const GenParams& P, const GenVariant& v, int grid, cudaStream_t stream, bool interleaved, bool blobs, bool bam) {
	if (bam) return interleaved ? launch_tables<true, true, true>(P, v, grid, stream) : launch_tables<false, true, true>(P, v, grid, stream);
	if (blobs) return interleaved ? launch_tables<true, true>(P, v, grid, stream) : launch_tables<false, true>(P, v, grid, stream);
	return interleaved ? launch_tables<true, false>(P, v, grid, stream) : launch_tables<false, false>(P, v, grid, stream);
}

// ----------------------------------------------------------------------------------------
// unfold_kernel: the sequence lines of one FASTA record as they lie in the file (raw, line feeds included) -> the
// chromosome string the reference works on: line ends dropped, upper case (FastaReference::getSequence,
// lib/fastahack/Fasta.cpp:304-334, then Genome::getSubSequence's toupper).  The .fai entry gives the geometry: every
// line but the last holds lineBases bases in lineWidth bytes, so base i sits at raw[i + (i / lineBases) * (lineWidth -
// lineBases)].  One thread per 16 bases; *other counts the characters that are neither ACGT nor N (IUPAC codes: the host
// keeps such chromosomes on its own string path, see host_plan.cpp).
// ----------------------------------------------------------------------------------------
__global__ void unfold_kernel(const uint8_t* __restrict__ raw, uint64_t rawLen, uint32_t nBases, uint32_t lineBases, uint32_t pad,
                              uint8_t* __restrict__ out, unsigned long long* __restrict__ other) {
	const uint32_t i0 = (blockIdx.x * blockDim.x + threadIdx.x) * 16u;
	uint32_t bad = 0;
	if (i0 < nBases) {
		uint32_t line = i0 / lineBases, col = i0 - line * lineBases;
		uint64_t src = (uint64_t)i0 + (uint64_t)line * pad;
		uint32_t w[4] = {0u, 0u, 0u, 0u};
		const uint32_t n = min(16u, nBases - i0);
		for (uint32_t k = 0; k < n; k++) {
			uint32_t c = src < rawLen ? raw[src] : (uint32_t)'N';
			if (c - 'a' < 26u) c -= 32u;
			bad += !(c == 'A' || c == 'C' || c == 'G' || c == 'T' || c == 'N');
			w[k >> 2] |= c << (8 * (k & 3));
			src++;
			if (++col == lineBases) { col = 0; src += pad; }
		}
		if (n == 16u) *(uint4*)(out + i0) = make_uint4(w[0], w[1], w[2], w[3]);
		else for (uint32_t k = 0; k < n; k++) out[i0 + k] = (uint8_t)(w[k >> 2] >> (8 * (k & 3)));
	}
	bad = __reduce_add_sync(0xffffffffu, bad);
	if (bad && (threadIdx.x & 31) == 0) atomicAdd(other, (unsigned long long)bad);
}

cudaError_t launch_unfold(const uint8_t* raw, uint64_t rawLen, uint64_t nBases, uint32_t lineBases, uint32_t lineWidth, uint8_t* out,
                          unsigned long long* other, cudaStream_t stream) {
	if (nBases == 0) return cudaSuccess;
	const uint64_t threads = (nBases + 15) / 16;
	unfold_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, stream>>>(raw, rawLen, (uint32_t)nBases, lineBases, lineWidth - lineBases, out, other);
	return cudaGetLastError();
}

cudaError_t launch_pack(const uint8_t* ascii, uint64_t n, uint64_t firstBase, uint32_t* hap2, uint32_t* hapN,
                        const int8_t* lut, cudaStream_t stream) {
	if (n == 0) return cudaSuccess;
	uint64_t groups = ((firstBase + n - 1) >> 5) - (firstBase >> 5) + 1;
	int threads = 256;
	uint64_t blocks = (groups + threads - 1) / threads;
	pack_kernel<<<(unsigned)blocks, threads, 0, stream>>>(ascii, n, firstBase, hap2, hapN, lut);
	return cudaGetLastError();
}

cudaError_t launch_census(const DevTables& t, bool fp64, const CensusBin* bins, int nBins, uint64_t seed,
                          uint16_t* riskyAttempt, int32_t* emitted, cudaStream_t stream) {
	if (nBins == 0) return cudaSuccess;
	int threads = 64;
	int blocks = (nBins + threads - 1) / threads;
	if (fp64) census_kernel<true><<<blocks, threads, 0, stream>>>(t, bins, nBins, seed, riskyAttempt, emitted);
	else census_kernel<false><<<blocks, threads, 0, stream>>>(t, bins, nBins, seed, riskyAttempt, emitted);
	return cudaGetLastError();
}

cudaError_t launch_poke(uint32_t* hap2, uint32_t* hapN, const int64_t* pos, const uint8_t* chars, int64_t n, const int8_t* lut, cudaStream_t stream) {
	if (n <= 0) return cudaSuccess;
	poke_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(hap2, hapN, pos, chars, n, lut);
	return cudaGetLastError();
}

cudaError_t launch_unpack(const uint32_t* hap2, const uint32_t* hapN, uint64_t firstBase, uint64_t n, uint32_t baseChars, uint8_t* out, cudaStream_t stream) {
	if (n == 0) return cudaSuccess;
	unpack_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(hap2, hapN, firstBase, n, baseChars, out);
	return cudaGetLastError();
}

cudaError_t launch_gc_census(const uint32_t* hap2, const uint32_t* hapN, const int64_t* starts, const int32_t* lens, int64_t n,
                             uint32_t gcCodes, int32_t* gc, int32_t* nn, cudaStream_t stream) {
	if (n <= 0) return cudaSuccess;
	const int threads = 256;
	const int64_t blocks = (n + threads / 32 - 1) / (threads / 32);
	gc_census_kernel<<<(unsigned)blocks, threads, 0, stream>>>(hap2, hapN, starts, lens, n, gcCodes, gc, nn);
	return cudaGetLastError();
}

cudaError_t launch_locate(const int64_t* emitBase, int64_t nBins, int64_t emitLo, int tilePairs, int nTiles, int32_t* tileStartBin,
                          cudaStream_t stream) {
	if (nTiles == 0) return cudaSuccess;
	int threads = 256;
	int blocks = (nTiles + threads - 1) / threads;
	locate_kernel<<<blocks, threads, 0, stream>>>(emitBase, nBins, emitLo, tilePairs, nTiles, tileStartBin);
	return cudaGetLastError();
}

}  // namespace ssc
