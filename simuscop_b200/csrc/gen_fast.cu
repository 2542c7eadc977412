// gen_fast.cu -- the production generation kernel (N = 4, K = 3, RL <= 160, tables in shared memory).
//
// Same algorithm and bytes as generate_kernel (kernels.cu), engineered for instruction issue,
// which -- not HBM -- bounds this path (4 uniform draws per base = one Philox4x32-10 block per
// lane per cycle; the ALU and FMA-heavy pipes are the busiest units):
//   * one warp per pair, lane = sequencing cycle, both mates; FG_WORKERS independent warps per
//     CTA, one CTA per SM; a warp takes FG_CHUNK consecutive pairs per ticket (atomic counter), so
//     the bin record of a pair is almost always the one of the previous pair and no warp waits
//     for another;
//   * Philox rounds fully unrolled as IMAD.WIDE + LOP3 with the ten round keys read straight
//     from the kernel parameters (constant bank operands, computed once on the host); the first
//     two rounds are partly shared by the chunks of a read (same pair / mate / stream words);
//   * the k-mer context of cycle j is cut straight out of the 2-bit packed haplotype window
//     (two LDS + one funnel shift for three bases); a LUT turns it into the byte offset of the
//     substitution row, whose fourth word carries the offset of the quality row, whose entries
//     carry threshold, quality symbol and base character -- the common read never materialises
//     its bases and does no index arithmetic beyond three adds;
//   * cycle -> position-bin offsets are per-lane constants; record terminators ride on the idle
//     lanes of the last chunk;
//   * indel candidates and non-ACGT bases are only detected per lane (two compares per chunk, one
//     vote per read); such reads (about 17 % with the shipped rates) take a compact non-unrolled
//     path: the events become a sorted list of output segments, the post-indel read is spliced 16
//     bases per lane out of the packed window into a second packed array, and the per-base work is
//     the fast path's again (scan_events / splice_read / emit_packed); only reads next to a
//     non-ACGT base, or grown past the unrolled chunks, go position by position (emit_mapped);
//   * warps never wait for each other: the records of a ticket are written back to back into that
//     ticket's blob in an HBM scratch slab (pass 1).  Two small bandwidth-bound kernels then scan
//     the blob lengths and move every blob (about 10 KB per file) to its exact byte offset with
//     16-byte stores (pass 2), so the final slab is dense, ordered and byte-identical to the
//     reference's file.  (Moving the blobs from inside the generation kernel -- by the generating
//     warps with a lag, or by dedicated mover warps -- was measured slower: the moves are latency
//     bound and every warp they occupy is one less to hide the ALU latency of generation.)
#include <cuda_runtime.h>
#include <cstdint>

#include "bam.cuh"
#include "device_types.h"
#include "kernels.h"
#include "philox.cuh"

namespace ssc {

static constexpr int F_SRC_CAP = 256;           // longest read after indels
static constexpr int F_EV_MAX = 32;
static constexpr int F_INS_CAP = 128;
static constexpr int F_WIN_WORDS = 32;          // 16 data words + 9 mask words (+pad)
static constexpr int F_QROW = 68;               // bytes of a shared-memory quality row (QP == 8): 8 x {threshold, sym | char << 8} + one pad
                                                // word: an odd word pitch spreads the rows of a warp over all 32 banks
static constexpr int F_Q16_KEYS = 40;           // QP == 16: thresholds per quality row (16-bit keys)
static constexpr int F_Q16_ROW = 124;           // bytes of such a row: 40 keys + 40 symbols + pad (31 words: an odd word pitch)
__host__ __device__ inline int fast_sub_pitch(int B) { return B | 1; }   // entries per substitution row, odd for the same reason
static constexpr int F_LUT_N = 6 * 64;          // context LUT (16-bit entries: 64 entries = 32 banks, conflict free):
                                                // fwd, rev, fwd cycle 0, fwd cycle 1, rev cycle 0, rev cycle 1

struct FastLayout {
	int sub, qual, qualSym, isizeT, isizeSym, insT, insSym, delT, delSym, lut, dig, warp, total;
	int w_ev, w_insb, w_insp, w_out, w_win, perWarp;
};

__host__ __device__ inline FastLayout fast_layout(int subBytes, int qualBytes, int qualSymBytes, int nIsize, int nIns, int nDel) {
	FastLayout L;
	// per-warp scratch first, the LUT and the digit constants right behind it: their shared addresses are compile-time
	// constants (plus warp * perWarp), which matters because the register-starved kernel recomputes them wherever it needs them
	int w = 0;
	L.w_ev = w; w += F_EV_MAX * 8;
	L.w_insb = w; w += F_INS_CAP;
	L.w_insp = w; w += 48;                          // inserted bases, packed: one pad word in front, 8 + 1 words
	L.w_out = w; w += 80;                           // spliced (post-indel) read, packed like a window: one pad word in front, 16 + 1 words
	L.w_win = w; w += 2 * F_WIN_WORDS * 4;          // one window per mate, filled by cp.async
	L.perWarp = w;
	int o = 0;
	L.warp = o; o += FG_GEN * L.perWarp;
	L.lut = o; o += F_LUT_N * 2;
	L.dig = o; o += 32 * 16;                       // per-lane header digit constants
	L.sub = o; o += (subBytes + 15) / 16 * 16;
	L.qual = o; o += (qualBytes + 15) / 16 * 16;
	L.qualSym = o; o += (qualSymBytes + 15) / 16 * 16;
	L.isizeT = o; o += (nIsize * 4 + 15) / 16 * 16;
	L.isizeSym = o; o += (nIsize * 2 + 15) / 16 * 16;
	L.insT = o; o += (nIns * 4 + 15) / 16 * 16;
	L.insSym = o; o += (nIns * 2 + 15) / 16 * 16;
	L.delT = o; o += (nDel * 4 + 15) / 16 * 16;
	L.delSym = o; o += (nDel * 2 + 15) / 16 * 16;
	L.total = o;
	return L;
}

__host__ __device__ inline void fast_qual_bytes(const DevTables& t, int qp, int* qualBytes, int* qualSymBytes) {
	if (qp == 8) { *qualBytes = 16 * t.qualBins * F_QROW; *qualSymBytes = 0; }
	else if (qp == 16) { *qualBytes = 16 * t.B * F_Q16_ROW; *qualSymBytes = 0; }
	else if (qp == 2) { *qualBytes = 4 * t.B * (t.qualDiagPitch + 1) * 4; *qualSymBytes = 4 * t.B * (t.qualDiagPitch + 1); }   // odd word pitch
	else { *qualBytes = 0; *qualSymBytes = 0; }
}

// read-only table reads by shared-window address
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) { uint32_t v; asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr)); return v; }
__device__ __forceinline__ uint32_t lds_u8(uint32_t addr) { uint32_t v; asm("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(addr)); return v; }
__device__ __forceinline__ uint32_t lds_u16(uint32_t addr) { uint32_t v; asm("{\n\t.reg .u16 h;\n\tld.shared.u16 h, [%1];\n\tcvt.u32.u16 %0, h;\n\t}" : "=r"(v) : "r"(addr)); return v; }

__device__ __forceinline__ void cp_async4(uint32_t dstShared, const void* src) {
	asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dstShared), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// acc += inc if a > b (unsigned): one ISETP + one predicated IADD
__device__ __forceinline__ void add_gt(uint32_t& acc, uint32_t a, uint32_t b, uint32_t inc) {
	asm("{\n\t.reg .pred p;\n\tsetp.gt.u32 p, %1, %2;\n\t@p add.u32 %0, %0, %3;\n\t}" : "+r"(acc) : "r"(a), "r"(b), "r"(inc));
}
// acc += inc if a < b (unsigned)
__device__ __forceinline__ void add_lt(uint32_t& acc, uint32_t a, uint32_t b, uint32_t inc) {
	asm("{\n\t.reg .pred p;\n\tsetp.lt.u32 p, %1, %2;\n\t@p add.u32 %0, %0, %3;\n\t}" : "+r"(acc) : "r"(a), "r"(b), "r"(inc));
}
// The same with the add issued as a multiply-add (acc += inc * one, one == 1 from the kernel parameters, opaque to the
// compiler): the ALU pipe is the busiest unit of the hot loop, the FMA pipe has room.
__device__ __forceinline__ void fadd_gt(uint32_t& acc, uint32_t a, uint32_t b, uint32_t inc, uint32_t one) {
	asm("{\n\t.reg .pred p;\n\tsetp.gt.u32 p, %1, %2;\n\t@p mad.lo.u32 %0, %4, %3, %0;\n\t}" : "+r"(acc) : "r"(a), "r"(b), "r"(inc), "r"(one));
}
__device__ __forceinline__ void fadd_lt(uint32_t& acc, uint32_t a, uint32_t b, uint32_t inc, uint32_t one) {
	asm("{\n\t.reg .pred p;\n\tsetp.lt.u32 p, %1, %2;\n\t@p mad.lo.u32 %0, %4, %3, %0;\n\t}" : "+r"(acc) : "r"(a), "r"(b), "r"(inc), "r"(one));
}

__device__ __forceinline__ long long f_draw_pos(uint32_t u, int spos, int epos) {
	double frac = __dmul_rn((double)u, 2.3283064365386962890625e-10);
	double v = __dadd_rn((double)spos, __dmul_rn((double)((long long)epos + 1 - spos), frac));
	return (long long)v;
}

// binary search in a compressed CDF held in shared memory: sym[#{i : T[i] < u}] (per lane or warp-uniform u)
__device__ __forceinline__ int uni_lookup(const uint32_t* T, const uint16_t* sym, int n, uint32_t u) {
	int lo = 0, len = n - 1;
	while (len > 0) {
		int half = len >> 1;
		if (T[lo + half] < u) { lo += half + 1; len -= half + 1; } else len = half;
	}
	return (int)sym[lo];
}

__device__ __forceinline__ int f_ndigits(uint32_t v) {
	int n = 1;
	n += v >= 10u; n += v >= 100u; n += v >= 1000u; n += v >= 10000u; n += v >= 100000u;
	n += v >= 1000000u; n += v >= 10000000u; n += v >= 100000000u; n += v >= 1000000000u;
	return n;
}

// floor(v / 10^d) = umulhi(v, M) >> S for every v < 2^31 (checked exhaustively at the step boundaries)
__constant__ uint32_t c_pow10[10] = {1u, 10u, 100u, 1000u, 10000u, 100000u, 1000000u, 10000000u, 100000000u, 1000000000u};
__constant__ uint32_t c_divM[10] = {0u, 0x66666667u, 0x51eb851fu, 0x10624dd3u, 0x68db8badu, 0x14f8b589u, 0x431bde83u, 0x6b5fca6bu,
                                    0x55e63b89u, 0x44b82fa1u};
__constant__ uint32_t c_divS[10] = {0u, 2u, 5u, 6u, 12u, 13u, 18u, 22u, 25u, 28u};

struct QualTabs {
	const uint8_t* rows; int qbins;                   // QP == 8: shared, [ref*4+call][bin (qbins per block)] rows of F_QROW bytes
	const uint32_t* diagT; const uint8_t* diagSym;    // QP == 2: shared, ref == call rows
	const uint32_t* gT; const uint8_t* gSym;          // full table in global memory
	int pitch, diagPitch;
};

struct WarpCtx {
	int B, subPitch, minQ, RL, nInsLen, nDelLen, nBasesM1, mDelta;
	uint32_t baseChars, compLut;
	const uint4* sub;          // shared: table of the current mate
	QualTabs q;
	const uint32_t* insT; const uint16_t* insSym;
	const uint32_t* delT; const uint16_t* delSym;
	const uint32_t* win;       // shared window: data words [0..16), mask words [16..25)
	const uint8_t* lutB;       // shared: context LUT (16-bit entries, 6 variants of 64)
	uint32_t* ev; uint8_t* insb;
	uint32_t* insp; uint32_t* outw;   // packed inserted bases / spliced read (word 0 of each array, a pad word lies in front)
	const uint32_t* rk;        // Philox round keys
	uint32_t c0, c1;           // pair counter words
	uint32_t sub16S;           // QP == 16: shared address of the 8-byte substitution entries of the current mate
	const uint4* gsub;         // QP == 16: the exact substitution rows of the current mate in global memory (tie fallback)
	uint32_t qualBaseS;        // shared address folded into word 3 of the substitution rows
	uint32_t qstride;          // bytes between the quality rows (ref, call) and (ref, call + 1) of one bin
	int lane;
};

// Quality lookup.  Rows hold ascending inclusive thresholds padded with 0xFFFFFFFF; symbol index = #{i : T[i] < u}.
//   QP == 8: all 16*B rows in shared memory, 8 interleaved {threshold, symbol} entries, three search steps;
//   QP == 2: only the ref == call rows in shared memory (pitch = live symbols rounded up to 4, generic branch-free
//            lower bound); the rare substituted bases go to the full table in global memory (L2);
//   QP == 0: full table in global memory.
template <int QP>
__device__ __forceinline__ uint32_t qual_lookup(const QualTabs& q, uint32_t cur, uint32_t call, uint32_t binIdx, int B, uint32_t u3) {
	if (QP == 8) {
		const uint8_t* qa = q.rows + ((cur * 4u + call) * (uint32_t)q.qbins + binIdx) * (uint32_t)F_QROW;
		uint32_t k = 0;
		add_lt(k, *(const uint32_t*)(qa + 24), u3, 32u);
		add_lt(k, *(const uint32_t*)(qa + k + 8), u3, 16u);
		add_lt(k, *(const uint32_t*)(qa + k), u3, 8u);
		return qa[k + 4];
	}
	if (QP == 2 && cur == call) {
		const uint32_t base = (cur * (uint32_t)B + binIdx) * (uint32_t)(q.diagPitch + 1);   // rows padded to an odd pitch (banks)
		const uint32_t* qt = q.diagT + base;
		uint32_t k = 0;
		for (int len = q.diagPitch; len > 1;) {
			const int half = len >> 1;
			add_lt(k, qt[k + half - 1], u3, (uint32_t)half);
			len -= half;
		}
		return q.diagSym[base + k];
	}
	const uint32_t qrow = (cur * 4u + call) * (uint32_t)B + binIdx;
	const uint32_t* qt = q.gT + qrow * q.pitch;
	int k = 0;
	for (int s = q.pitch >> 1; s > 0; s >>= 1) if (qt[k + s - 1] < u3) k += s;
	return q.gSym[qrow * q.pitch + k];
}

// QP == 16: profiles whose quality rows have up to 40 live symbols (GAIIx, HiSeq2000, HiSeq2500).  Their 32-bit tables do not
// fit into shared memory, their HIGH HALVES do: substitution entries {k0, k1, k2, ref*4+base} and quality rows of 40 keys +
// 40 symbols, 16 bits per key.  For a draw u with high half uh, "u > T" is decided by "uh > key" unless uh == key (probability
// 2^-16 per compare); a lane that meets such a tie repeats the lookup on the exact 32-bit tables in global memory.  Same
// decision as the full compare for every u, by construction.  rowIdx: entry index of the substitution row (from the context
// LUT), passThrough: unknown k-mer context, the base passes through (Profile.cpp:1531-1533); cur: template base (0..3).
__device__ __forceinline__ void lookup16(const WarpCtx& w, uint32_t rowIdx, uint32_t binIdx, uint32_t u2, uint32_t u3, bool passThrough,
                                         uint32_t cur, uint32_t& ch, uint32_t& q) {
	uint32_t lo, hi;
	asm("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(lo), "=r"(hi) : "r"(w.sub16S + (rowIdx + binIdx) * 8u));
	const uint32_t uh2 = u2 >> 16, uh3 = u3 >> 16;
	const uint32_t k0 = lo & 0xffffu, k1 = lo >> 16, k2 = hi & 0xffffu;
	uint32_t rc = hi >> 16;                                         // (ref, base) row: ref * 4 + base
	add_gt(rc, uh2, k0, 1u); add_gt(rc, uh2, k1, 1u); add_gt(rc, uh2, k2, 1u);
	bool tie = (uh2 == k0) | (uh2 == k1) | (uh2 == k2);
	if (passThrough) { rc = cur * 5u; tie = false; }
	const uint32_t qa = w.qualBaseS + (rc * (uint32_t)w.B + binIdx) * (uint32_t)F_Q16_ROW;
	uint32_t kp = qa;                                               // address of the first key >= uh3: lower bound over 40 keys,
	add_lt(kp, lds_u16(kp + 38), uh3, 40u);                         // steps of 20, 10, 5, 2, 1, 1 keys (a running address: one
	add_lt(kp, lds_u16(kp + 18), uh3, 20u);                         // add less per step than row address + offset)
	add_lt(kp, lds_u16(kp + 8), uh3, 10u);
	add_lt(kp, lds_u16(kp + 2), uh3, 4u);
	add_lt(kp, lds_u16(kp), uh3, 2u);
	add_lt(kp, lds_u16(kp), uh3, 2u);
	tie |= lds_u16(kp) == uh3;                                      // (offset <= 78: the last key of a row is read at most)
	q = lds_u8(((qa + kp) >> 1) + 2u * F_Q16_KEYS);                 // symbol (kp - qa) / 2 of the row; qa + kp is even
	uint32_t call = rc & 3u;
	if (tie) {
		// exact repeat on the 32-bit tables (global memory, L2)
		const uint32_t row = rowIdx / (uint32_t)w.subPitch;
		const uint4 sr = w.gsub[row * (uint32_t)w.B + binIdx];
		call = passThrough ? cur : sr.w + (u2 > sr.x) + (u2 > sr.y) + (u2 > sr.z);
		const uint32_t ref = passThrough ? cur : (row & 3u);
		const uint32_t qrow = (ref * 4u + call) * (uint32_t)w.B + binIdx;
		const uint32_t* qt = w.q.gT + qrow * w.q.pitch;
		int kk = 0;
		for (int st = w.q.pitch >> 1; st > 0; st >>= 1) if (qt[kk + st - 1] < u3) kk += st;
		q = w.q.gSym[qrow * w.q.pitch + kk];
	}
	ch = __byte_perm(w.baseChars, 0, 0x4440u | call);
}

// template base code (0..3, 4 = non-ACGT) of read position j, from the shared window
__device__ __forceinline__ uint32_t window_code(const WarpCtx& w, int relBase /* base index relative to window word 0 */,
                                                bool rev) {
	const uint32_t d = w.win[relBase >> 4];
	uint32_t code = (d >> ((relBase & 15) * 2)) & 3u;
	if (rev) code = (w.compLut >> (2 * code)) & 3u;
	const int relM = relBase + w.mDelta;
	const uint32_t mk = w.win[16 + (relM >> 5)];
	if ((mk >> (relM & 31)) & 1u) code = 4u;
	return code;
}

// cooperative lower bound in a compressed CDF held in shared memory (warp-uniform u, all lanes converged):
// sym[#{i < n-1 : T[i] < u}] -- the same index uni_lookup finds, one ballot per 32 thresholds
__device__ __forceinline__ int coop_lookup(const uint32_t* T, const uint16_t* sym, int n, uint32_t u, int lane) {
	int cnt = 0;
	for (int b = 0; b < n - 1; b += 32) {
		const int i = b + lane;
		cnt += __popc(__ballot_sync(0xffffffffu, i < n - 1 && T[i] < u));
	}
	return (int)sym[cnt];
}

// Slow path of Profile::predict (a read with an indel candidate or a non-ACGT base): compact, not unrolled.
// Step 1, scan_events: the indel events of the read (Profile.cpp:1610-1634) as a sorted list of output-coordinate
//   segments {first output position behind the event's template base, inserted bases, template shift behind it}.
// Step 2a, splice_read + emit_packed (no non-ACGT base near the read, post-indel length within the NCH chunks): the
//   post-indel source sequence (Profile.cpp:1636-1658) is assembled 16 bases per lane from the packed window with funnel
//   shifts, in store orientation, and the per-base work is the fast path's (context cut out of packed words).
// Step 2b, emit_mapped (everything else): every lane maps its output position to a template base of the window (or an
//   inserted base) and gets the two context bases from its neighbours by shuffle.
struct IndelPlan {
	uint2 e0;          // first event (the others are in w.ev[1..])
	int nEv, m, insTotal;
};

// evbits: per lane, bit 2c = insertion test hit at cycle 32c+lane, bit 2c+1 = deletion test hit.
__device__ __forceinline__ IndelPlan scan_events(const WarpCtx& w, uint32_t evbits, int mate, unsigned int* errorFlags) {
	const int RL = w.RL, lane = w.lane;
	const uint32_t c2len = ((uint32_t)mate << 28) | ((uint32_t)STREAM_LEN << 24);
	const uint32_t c2ins = ((uint32_t)mate << 28) | ((uint32_t)STREAM_INSBASE << 24);
	// event k: x = first output position behind the event's template base | inserted bases << 9 | their offset in insb << 17,
	//          y = output position - template position of everything behind the event (running indelLength)
	uint2* evs = (uint2*)w.ev;
	uint2 e0 = make_uint2(0u, 0u);
	int nEv = 0, insTotal = 0, cum = 0, skipUntil = 0;
	bool tooMany = false;
	// chunks with a candidate in any lane (REDUX.OR over the warp): bit 2c
	const uint32_t anyBits = __reduce_or_sync(0xffffffffu, evbits);
	uint32_t chunkBits = (anyBits | (anyBits >> 1)) & 0x55555555u;
	while (chunkBits) {
		const int c = (__ffs(chunkBits) - 1) >> 1;
		chunkBits &= chunkBits - 1;
		const uint32_t insMask = __ballot_sync(0xffffffffu, (evbits >> (2 * c)) & 1u);
		const uint32_t delMask = __ballot_sync(0xffffffffu, (evbits >> (2 * c + 1)) & 1u);
		uint32_t mask = insMask | delMask;
		while (mask) {
			const int bit = __ffs(mask) - 1;
			mask &= mask - 1;
			const int j = c * 32 + bit;
			if (j < skipUntil) continue;
			const u32x4 lb = philox_rk(w.c0, w.c1, c2len, (uint32_t)j, w.rk);
			if ((insMask >> bit) & 1u) {
				const int Lk = coop_lookup(w.insT, w.insSym, w.nInsLen, lb.x, lane);     // Profile::getInsertLen
				if (Lk > 0) {
					if (nEv >= F_EV_MAX || insTotal + Lk > F_INS_CAP) { tooMany = true; break; }
					for (int i = lane; i < Lk; i += 32) {                                  // Profile.cpp:1563-1566
						const u32x4 bb = philox_rk(w.c0, w.c1, c2ins | (uint32_t)(i >> 2), (uint32_t)j, w.rk);
						const uint32_t ws = (i & 3) == 0 ? bb.x : (i & 3) == 1 ? bb.y : (i & 3) == 2 ? bb.z : bb.w;
						w.insb[insTotal + i] = (uint8_t)__umulhi((uint32_t)w.nBasesM1, ws);
					}
					// the inserted bases follow template base j (Profile.cpp:1650-1656)
					const uint2 e = make_uint2((uint32_t)(j + cum + 1) | ((uint32_t)Lk << 9) | ((uint32_t)insTotal << 17), (uint32_t)(cum + Lk));
					if (nEv == 0) e0 = e; else if (lane == 0) evs[nEv] = e;
					nEv++; insTotal += Lk; cum += Lk;
				}
			} else {
				int Lk = coop_lookup(w.delT, w.delSym, w.nDelLen, lb.y, lane);           // Profile::getDelLen
				if (Lk > RL - j) Lk = RL - j;                                             // Profile.cpp:1613
				if (Lk > 0) {
					if (nEv >= F_EV_MAX) { tooMany = true; break; }
					const uint2 e = make_uint2((uint32_t)(j + cum), (uint32_t)(cum - Lk));
					if (nEv == 0) e0 = e; else if (lane == 0) evs[nEv] = e;
					nEv++; cum -= Lk; skipUntil = j + Lk;
				}
			}
		}
	}
	if (RL + cum < 50) { nEv = 0; cum = 0; }                                             // Profile.cpp:1627-1634
	int m = RL + cum;
	if (tooMany || m > F_SRC_CAP) {
		if (lane == 0) atomicOr(errorFlags, tooMany ? 4u : 2u);
		nEv = 0; m = RL;
	}
	__syncwarp();
	IndelPlan pl;
	pl.e0 = e0; pl.nEv = nEv; pl.m = m; pl.insTotal = nEv ? insTotal : 0;
	return pl;
}

// Step 2a.  A packed array holds base i in bits 2*(i & 15) of word i >> 4.  gather16: the 16 bases src[q .. q+16) of such an
// array, restricted to the positions [lo, hi) of the word (0 <= lo < hi <= 16); q + lo >= 0 (q itself may be negative: the
// arrays have a pad word in front).
__device__ __forceinline__ uint32_t gather16(const uint32_t* src, int q, int lo, int hi) {
	const int wi = q >> 4;
	const uint32_t f = __funnelshift_r(src[wi], src[wi + 1], (uint32_t)(q & 15) * 2u);
	return f & (0xffffffffu >> (32 - 2 * hi)) & (0xffffffffu << (2 * lo));
}

// The post-indel read in store orientation (forward reads: output order; reverse reads: reversed, template and inserted
// bases as the store holds them, i.e. complemented), base y at packed index dOff + y of w.outw -- exactly what the
// window holds for an indel-free read of length m, so that the fast path's context extraction applies unchanged.
// Lane L < 16 assembles word L from the template runs between the events (slices of the window) and the inserted runs.
__device__ __forceinline__ void splice_read(const WarpCtx& w, const IndelPlan& pl, bool rev, int dOff) {
	const int RL = w.RL, lane = w.lane, m = pl.m, insTotal = pl.insTotal;
	const uint2* evs = (const uint2*)w.ev;
	// inserted bases, packed in store orientation
	if (lane < 9) w.insp[lane] = 0u;
	__syncwarp();
	for (int i = lane; i < insTotal; i += 32) {
		uint32_t code = w.insb[rev ? insTotal - 1 - i : i];
		if (rev) code = (w.compLut >> (2 * code)) & 3u;
		atomicOr(&w.insp[i >> 4], code << ((i & 15) * 2));
	}
	__syncwarp();
	const int y0 = 16 * lane - dOff;                   // store-order index of the first base of this lane's word
	uint32_t word = 0;
	int prevO = 0, prevShift = 0;
#pragma unroll 1
	for (int k = 0; k <= pl.nEv; k++) {
		int start = m, nIns = 0, insOff = 0, shiftAfter = 0;
		if (k < pl.nEv) {
			const uint2 e = k == 0 ? pl.e0 : evs[k];
			start = (int)(e.x & 0x1ffu); nIns = (int)((e.x >> 9) & 0xffu); insOff = (int)(e.x >> 17); shiftAfter = (int)e.y;
		}
		// template run: output [prevO, start) <- template [prevO - prevShift, start - prevShift)
		{
			const int n = start - prevO, t1 = prevO - prevShift;
			const int dst = rev ? m - start : prevO;
			const int src = rev ? RL - (t1 + n) : t1;
			const int lo = max(dst, y0) - y0, hi = min(dst + n, y0 + 16) - y0;
			if (lo < hi) word |= gather16(w.win, dOff + src + y0 - dst, lo, hi);
		}
		if (nIns > 0) {
			const int dst = rev ? m - (start + nIns) : start;
			const int src = rev ? insTotal - (insOff + nIns) : insOff;
			const int lo = max(dst, y0) - y0, hi = min(dst + nIns, y0 + 16) - y0;
			if (lo < hi) word |= gather16(w.insp, src + y0 - dst, lo, hi);
		}
		prevO = start + nIns; prevShift = shiftAfter;
	}
	if (lane < 16) w.outw[lane] = word;
	__syncwarp();
}

// Output modes of generate_slots_kernel (see there)
enum { OUT_FASTQ = 0, OUT_ARRAYS = 1, OUT_INTERLEAVED = 2, OUT_BAM = 3 };

// One base of a chunk: the character to pB, the quality to pQ (lanes inside the read); BAM: see bam_put_base, pB is the
// chunk's byte of 4-bit codes for this lane pair, and every lane of the warp must call it.
template <int OUT>
__device__ __forceinline__ void put_base(uint8_t* pB, uint8_t* pQ, bool in, uint32_t ch, uint32_t q, int lane) {
	if (OUT == OUT_BAM) bam_put_base(pB, pQ, in, ch, q, lane);
	else if (in) { *pB = (uint8_t)ch; *pQ = (uint8_t)q; }
}

// Per-base work of a read of m <= 32 * NCH bases whose source sequence is packed at index dOff (store orientation) of
// win: the fast path's phase C with the position bins of the post-indel length (Profile.cpp:1671), rolled.
// OUT_ARRAYS: the qualities lie `pitch` bytes behind the bases (array output) instead of m + 3 (FASTQ record); OUT_BAM: the
// bases are 4-bit codes, (m + 1) / 2 bytes, the qualities behind them.
template <int NCH, int QP, int OUT>
__device__ __forceinline__ void emit_packed(const WarpCtx& w, const uint32_t* win, int dOff, bool rev, int m, uint32_t lut0, uint32_t lutN,
                                            uint8_t* stage, int H, uint32_t pitch, const uint32_t (&x2)[NCH], const uint32_t (&x3)[NCH]) {
	constexpr bool ARRAYS = OUT == OUT_ARRAYS, BAM = OUT == OUT_BAM;
	const int lane = w.lane;
	const uint32_t inv = (m > 1) ? (0xffffffffu / (uint32_t)m + 1u) : 0xffffffffu;
	const int chunksM = (m + 31) >> 5;
	uint8_t* pB = stage + H + (BAM ? lane >> 1 : lane);   // this lane's base of the current chunk; its quality follows m + 3 bytes later
	uint8_t* pQ = ARRAYS ? pB + pitch : BAM ? stage + H + ((m + 1) >> 1) + lane : pB + m + 3;
	uint32_t a2[NCH], a3[NCH];
#pragma unroll
	for (int k = 0; k < NCH; k++) { a2[k] = x2[k]; a3[k] = x3[k]; }
#pragma unroll 1
	for (int c = 0; c < chunksM; c++) {
		const int j = c * 32 + lane;
		const uint32_t u2 = a2[0], u3 = a3[0];
#pragma unroll
		for (int k = 0; k + 1 < NCH; k++) { a2[k] = a2[k + 1]; a3[k] = a3[k + 1]; }
		const int jc = j < m ? j : m - 1;                // lanes past the read end: any valid index
		// forward: the three bases of cycles (j-2, j-1, j) start at index dOff + j - 2; reverse: cycles (j, j-1, j-2) at dOff + m-1 - j
		const int rel = rev ? dOff + m - 1 - jc : dOff + jc - 2;
		const uint32_t v6 = __funnelshift_r(win[rel >> 4], win[(rel >> 4) + 1], (uint32_t)(rel & 15) * 2u) & 63u;
		const uint32_t rowIdx = *(const uint16_t*)(w.lutB + (c == 0 ? lut0 : lutN) + v6 * 2u);
		const uint32_t binIdx = __umulhi((uint32_t)(jc * w.B), inv);
		uint32_t ch, q;
		if (QP == 16) {
			lookup16(w, rowIdx, binIdx, u2, u3, false, 0u, ch, q);
			put_base<OUT>(pB, pQ, j < m, ch, q, lane);
			pB += BAM ? 16 : 32; pQ += 32;
			continue;
		}
		const uint4 sr = w.sub[rowIdx + binIdx];
		uint32_t acc = sr.w;
		add_gt(acc, u2, sr.x, w.qstride); add_gt(acc, u2, sr.y, w.qstride); add_gt(acc, u2, sr.z, w.qstride);
		if (QP == 8) {
			uint32_t qa = binIdx * (uint32_t)F_QROW + acc;
			add_lt(qa, lds_u32(qa + 24), u3, 32u);
			add_lt(qa, lds_u32(qa + 8), u3, 16u);
			add_lt(qa, lds_u32(qa), u3, 8u);
			q = lds_u16(qa + 4);                                                // symbol | base character << 8
			ch = q >> 8;
		} else {
			const uint32_t r16 = acc / w.qstride;                              // qualBaseS == 0, qstride == F_QROW here
			q = qual_lookup<QP>(w.q, r16 >> 2, r16 & 3u, binIdx, w.B, u3);
			ch = __byte_perm(w.baseChars, 0, 0x4440u | (r16 & 3u));
		}
		put_base<OUT>(pB, pQ, j < m, ch, q, lane);
		pB += BAM ? 16 : 32; pQ += 32;
	}
}

// Step 2b.  x2/x3: the substitution / quality draws of output positions 32c+lane, c < NCH (registers of the caller).
// Writes bases/quals into stage[H ..] (qualities as in emit_packed).  OUT_BAM: every lane runs the per-base work, lanes past
// the read end on the position bin of base m - 1, so that the warp packs the 4-bit codes together.
template <int NCH, int QP, int OUT>
__device__ __forceinline__ void emit_mapped(const WarpCtx& w, const IndelPlan& pl, int mate, bool rev, int relFirst,
                                            uint8_t* stage, int H, uint32_t pitch, const uint32_t (&x2)[NCH], const uint32_t (&x3)[NCH]) {
	constexpr bool ARRAYS = OUT == OUT_ARRAYS, BAM = OUT == OUT_BAM;
	const int RL = w.RL, lane = w.lane, m = pl.m, nEv = pl.nEv;
	const uint2 e0 = pl.e0;
	const uint2* evs = (const uint2*)w.ev;
	const uint32_t c2cyc = ((uint32_t)mate << 28) | ((uint32_t)STREAM_CYCLE << 24);
	const uint32_t inv = (m > 1) ? (0xffffffffu / (uint32_t)m + 1u) : 0xffffffffu;
	const int chunksM = (m + 31) >> 5;
	uint32_t prev = 0;                               // codes of the previous chunk ('X' pads in front of the read: code 0, no flag)
	// the first event (almost always the only one) stays in registers: every lane computed it
	const int e0start = nEv > 0 ? (int)(e0.x & 0x1ffu) : 0x7fffffff;
	const int e0ins = (int)((e0.x >> 9) & 0xffu), e0off = (int)(e0.x >> 17), e0shift = (int)e0.y;
	uint8_t* const stB = stage + H + lane;          // bases of this lane; the qualities follow m + 3 bytes later
	// the draws of the first NCH chunks are the caller's registers: taken from the front of a copy that is shifted down
	// by one chunk per iteration (kept rolled: the hot loop has to stay inside the instruction cache)
	uint32_t a2[NCH], a3[NCH];
#pragma unroll
	for (int k = 0; k < NCH; k++) { a2[k] = x2[k]; a3[k] = x3[k]; }
#pragma unroll 1
	for (int c = 0; c < chunksM; c++) {
		const int j = c * 32 + lane;
		uint32_t u2 = a2[0], u3 = a3[0];
#pragma unroll
		for (int k = 0; k + 1 < NCH; k++) { a2[k] = a2[k + 1]; a3[k] = a3[k + 1]; }
		if (c >= NCH && j < m) {
			const u32x4 blk = philox_rk(w.c0, w.c1, c2cyc, (uint32_t)j, w.rk);
			u2 = blk.z; u3 = blk.w;
		}
		// source base of output position j: the last event segment that starts at or before j decides
		int shift = 0, insIdx = -1;
		{
			const int d = j - e0start;
			if (d >= 0) { shift = e0shift; insIdx = d < e0ins ? e0off + d : -1; }
		}
#pragma unroll 1
		for (int k = 1; k < nEv; k++) {
			const uint2 e = evs[k];
			const int d = j - (int)(e.x & 0x1ffu);
			if (d >= 0) {
				shift = (int)e.y;
				insIdx = d < (int)((e.x >> 9) & 0xffu) ? (int)(e.x >> 17) + d : -1;
			}
		}
		int tpos = j - shift;                            // lanes past the read end / on inserted bases: any valid window index
		tpos = tpos < 0 ? 0 : (tpos > RL - 1 ? RL - 1 : tpos);
		uint32_t code = window_code(w, rev ? relFirst - tpos : relFirst + tpos, rev);   // 0..3, 4 = non-ACGT
		if (insIdx >= 0) code = w.insb[insIdx];
		// the two bases in front (Profile.cpp:1660-1666): lanes 0 and 1 take them from the previous chunk
		const uint32_t both = code | (prev << 4);
		const uint32_t r1 = __shfl_sync(0xffffffffu, both, (lane + 31) & 31), r2 = __shfl_sync(0xffffffffu, both, (lane + 30) & 31);
		const uint32_t p1 = lane >= 1 ? (r1 & 7u) : (r1 >> 4), p2 = lane >= 2 ? (r2 & 7u) : (r2 >> 4);
		prev = code;
		if (BAM || j < m) {
			const uint32_t cur = code & 3u;
			const uint32_t v6 = (p2 & 3u) | ((p1 & 3u) << 2) | (cur << 4);
			const uint32_t n3 = (p2 >> 2) | ((p1 >> 2) << 1) | ((code >> 2) << 2);          // bit 2 = the base itself
			const uint32_t var = j >= 2 ? 0u : (j == 0 ? 2u : 3u);                          // 'X' padded contexts
			const uint32_t rowIdx = *(const uint16_t*)(w.lutB + var * 128u + v6 * 2u);
			const uint32_t binIdx = __umulhi((uint32_t)((BAM && j >= m ? m - 1 : j) * w.B), inv);
			uint32_t ch, q;
			if (QP == 16) {
				if (n3 & 4u) { ch = 'N'; q = (uint32_t)w.minQ + __umulhi(20u, u3); }   // randomInteger(33, 53), Profile.cpp:1583
				else lookup16(w, rowIdx, binIdx, u2, u3, n3 != 0u, cur, ch, q);
				if (BAM) bam_put_base(stage + H + 16 * c + (lane >> 1), stage + H + ((m + 1) >> 1) + j, j < m, ch, q, lane);
				else {
					stB[c * 32] = (uint8_t)ch;
					if (ARRAYS) stB[pitch + c * 32] = (uint8_t)q;
					else stB[m + 3 + c * 32] = (uint8_t)q;
				}
				continue;
			}
			const uint4 sr = w.sub[rowIdx + binIdx];
			uint32_t acc = sr.w;
			add_gt(acc, u2, sr.x, w.qstride); add_gt(acc, u2, sr.y, w.qstride); add_gt(acc, u2, sr.z, w.qstride);
			if (n3) acc = w.qualBaseS + cur * (5u * w.qstride);                    // unknown context: the base passes through
			if (n3 & 4u) { ch = 'N'; q = (uint32_t)w.minQ + __umulhi(20u, u3); }   // randomInteger(33, 53), Profile.cpp:1583
			else if (QP == 8) {
				uint32_t qa = binIdx * (uint32_t)F_QROW + acc;
				add_lt(qa, lds_u32(qa + 24), u3, 32u);
				add_lt(qa, lds_u32(qa + 8), u3, 16u);
				add_lt(qa, lds_u32(qa), u3, 8u);
				q = lds_u16(qa + 4);                                                // symbol | base character << 8
				ch = q >> 8;
			} else {
				const uint32_t r16 = acc / w.qstride;                              // qualBaseS == 0, qstride == F_QROW here
				q = qual_lookup<QP>(w.q, r16 >> 2, r16 & 3u, binIdx, w.B, u3);
				ch = __byte_perm(w.baseChars, 0, 0x4440u | (r16 & 3u));
			}
			if (BAM) bam_put_base(stage + H + 16 * c + (lane >> 1), stage + H + ((m + 1) >> 1) + j, j < m, ch, q, lane);
			else {
				stB[c * 32] = (uint8_t)ch;
				if (ARRAYS) stB[pitch + c * 32] = (uint8_t)q;
				else stB[m + 3 + c * 32] = (uint8_t)q;
			}
		}
	}
}

// ---------------------------------------------------------------------------------------------
// blob -> dense slab (pass 2)
// ---------------------------------------------------------------------------------------------
// copy len bytes from a 16-byte aligned global source to an arbitrarily aligned global destination with 16-byte stores.
// Vector v of the destination (16-byte aligned) takes source bytes [head + 16 v, head + 16 v + 16): five 4-byte loads and
// four funnel shifts (32 registers, 8 CTAs per SM: 5.15 TB/s of DRAM traffic; a form with two 16-byte loads per vector needs
// more registers than that).  Streaming accesses (ld.global.cs / st.global.cs): the blob is read once and the slab is not
// read again on the device.  The source may be read up to 4 bytes past len (blob pitch).
__device__ __forceinline__ void copy_realign(const uint8_t* __restrict__ src, int len, uint8_t* __restrict__ dst, int lane) {
	int head = (int)((16u - (uint32_t)((uintptr_t)dst & 15u)) & 15u);
	if (head > len) head = len;
	if (lane < head) dst[lane] = __ldcs(src + lane);
	const int nvec = (len - head) >> 4;
	const uint32_t* s32 = (const uint32_t*)src;
	const int r8 = (head & 3) * 8;
	const int q0 = head >> 2;
	uint4* dv = (uint4*)(dst + head);
#pragma unroll 4
	for (int v = lane; v < nvec; v += 32) {
		const int q = q0 + 4 * v;
		const uint32_t w0 = __ldcs(s32 + q), w1 = __ldcs(s32 + q + 1), w2 = __ldcs(s32 + q + 2), w3 = __ldcs(s32 + q + 3), w4 = __ldcs(s32 + q + 4);
		uint4 o;
		o.x = __funnelshift_r(w0, w1, r8);
		o.y = __funnelshift_r(w1, w2, r8);
		o.z = __funnelshift_r(w2, w3, r8);
		o.w = __funnelshift_r(w3, w4, r8);
		__stcs(dv + v, o);
	}
	const int t0 = head + (nvec << 4);
	if (lane < len - t0) dst[t0 + lane] = __ldcs(src + t0 + lane);
}

// pass 2a: exclusive prefix of the packed blob lengths (len1 << 31 | len2; a slab holds < 2^31 bytes), one CTA,
// rounds of SC_THREADS * 8 lengths (each thread 64 contiguous bytes), warp-shuffle scans
static constexpr int SC_THREADS = 1024;
__global__ void __launch_bounds__(SC_THREADS) scan_blobs_kernel(const GenParams P) {
	__shared__ unsigned long long s_warp[SC_THREADS / 32];
	__shared__ unsigned long long s_carry;
	const int n = P.nTiles;
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	if (threadIdx.x == 0) s_carry = 0;
	__syncthreads();
	for (int base = 0; base < n; base += SC_THREADS * 8) {
		const int i0 = base + threadIdx.x * 8;
		unsigned long long v[8];
#pragma unroll
		for (int k = 0; k < 8; k++) v[k] = (i0 + k < n) ? P.tileState[i0 + k] : 0ull;
		unsigned long long sum = 0;
#pragma unroll
		for (int k = 0; k < 8; k++) sum += v[k];
		unsigned long long incl = sum;
#pragma unroll
		for (int d = 1; d < 32; d <<= 1) {
			const unsigned long long o = __shfl_up_sync(0xffffffffu, incl, d);
			if (lane >= d) incl += o;
		}
		if (lane == 31) s_warp[warp] = incl;
		__syncthreads();
		if (warp == 0) {
			unsigned long long w = s_warp[lane];
#pragma unroll
			for (int d = 1; d < 32; d <<= 1) {
				const unsigned long long o = __shfl_up_sync(0xffffffffu, w, d);
				if (lane >= d) w += o;
			}
			s_warp[lane] = w;                     // inclusive prefix of the warp totals
		}
		__syncthreads();
		unsigned long long run = s_carry + (warp ? s_warp[warp - 1] : 0ull) + incl - sum;
#pragma unroll
		for (int k = 0; k < 8; k++) { if (i0 + k < n) P.blobPrefix[i0 + k] = run; run += v[k]; }
		__syncthreads();
		if (threadIdx.x == SC_THREADS - 1) s_carry = run;
		__syncthreads();
	}
	if (threadIdx.x == 0) {
		const unsigned long long fin = s_carry;
		P.result->bytes1 = fin >> 31;
		P.result->bytes2 = fin & 0x7fffffffull;
		if ((fin >> 31) > P.cap1 || (fin & 0x7fffffffull) > P.cap2) atomicOr(&P.result->errorFlags, 1u);
	}
}

// pass 2b: blob j of a batch -> its place in the dense slabs (one warp)
__device__ __forceinline__ void move_blob(const uint8_t* __restrict__ blobs1, const uint8_t* __restrict__ blobs2, uint32_t blobPitch,
                                          const unsigned long long* __restrict__ tileState, const unsigned long long* __restrict__ prefix,
                                          uint8_t* __restrict__ dense1, uint8_t* __restrict__ dense2, unsigned long long cap1,
                                          unsigned long long cap2, int j, int lane) {
	const unsigned long long excl = __ldcg(prefix + j), mine = __ldcg(tileState + j);
	const unsigned long long d1 = excl >> 31, d2 = excl & 0x7fffffffull;
	const int l1 = (int)(mine >> 31), l2 = (int)(mine & 0x7fffffffull);
	if (d1 + (unsigned)l1 > cap1 || d2 + (unsigned)l2 > cap2) return;   // flagged by the scan
	const size_t blob = (size_t)j * blobPitch;
	copy_realign(blobs1 + blob, l1, dense1 + d1, lane);
	if (l2) copy_realign(blobs2 + blob, l2, dense2 + d2, lane);
}

// stand-alone form: the last batch of a call, every batch when the concurrent mover is off, and the gzip members
static constexpr int CP_THREADS = 256;
__global__ void __launch_bounds__(CP_THREADS, 8) move_blobs_kernel(const GenParams P) {
	const int lane = threadIdx.x & 31;
	const int nWarps = gridDim.x * (CP_THREADS / 32);
	for (int j = blockIdx.x * (CP_THREADS / 32) + (threadIdx.x >> 5); j < P.nTiles; j += nWarps)
		move_blob(P.out1, P.out2, P.blobPitch, P.tileState, P.blobPrefix, P.dense1, P.dense2, P.cap1, P.cap2, j, lane);
}

// ---------------------------------------------------------------------------------------------
// pass 2b on a few SMs, under the generation kernel of the next batch (round 2).
// The stand-alone move kernel reaches its 5 TB/s with ~9 500 warps in flight (each warp is bound by the latency of its own
// loads), i.e. it needs the whole GPU -- which the generation kernel needs too.  This form needs 8 of the 148 SMs: every
// warp pulls a blob in 4 KB pieces into its own shared-memory ring with bulk asynchronous copies (cp.async.bulk, the TMA
// engine: no registers, no warp stalled on a load), waits on the ring's mbarriers, and stores the pieces 16 bytes per lane
// at their final, arbitrarily aligned place (two LDS.128 + four funnel shifts per store).  A warp keeps up to 12 KB in flight
// instead of 2.5 KB, so 128 warps move a batch in less time than the other 140 SMs need to generate the next one.
// ---------------------------------------------------------------------------------------------
static constexpr int MV_WARPS = 16;
static constexpr int MV_THREADS = MV_WARPS * 32;
static constexpr int MV_STAGES = 3;
static constexpr int MV_PIECE = 4096;
static constexpr int MV_STAGE_BYTES = MV_PIECE + 32;         // the vector loop reads one 16-byte chunk past the piece
static constexpr int MV_WARP_BYTES = MV_STAGES * MV_STAGE_BYTES + 32;   // + the ring's mbarriers

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count)); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
	asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
	asm volatile("{\n\t.reg .pred p;\n\tMV_WAIT:\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t@!p bra MV_WAIT;\n\t}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_load(uint32_t dstShared, const void* src, uint32_t bytes, uint32_t bar) {
	asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dstShared), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

// one piece (n <= 4096 bytes, in the warp's stage at shared address st) to dst (any alignment)
template <int Q0>
__device__ __forceinline__ void store_piece_vectors(uint32_t st, uint4* __restrict__ dv, int nvec, int r8, int lane) {
#pragma unroll 2
	for (int v = lane; v < nvec; v += 32) {
		uint32_t w[8];
		asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]) : "r"(st + 16u * v));
		asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7]) : "r"(st + 16u * v + 16u));
		uint4 o;
		o.x = __funnelshift_r(w[Q0], w[Q0 + 1], r8);
		o.y = __funnelshift_r(w[Q0 + 1], w[Q0 + 2], r8);
		o.z = __funnelshift_r(w[Q0 + 2], w[Q0 + 3], r8);
		o.w = __funnelshift_r(w[Q0 + 3], w[Q0 + 4], r8);
		__stcs(dv + v, o);
	}
}

__device__ __forceinline__ void store_piece(uint32_t st, const uint8_t* stGeneric, int n, uint8_t* __restrict__ dst, int lane) {
	int head = (int)((16u - (uint32_t)((uintptr_t)dst & 15u)) & 15u);
	if (head > n) head = n;
	if (lane < head) dst[lane] = stGeneric[lane];
	const int nvec = (n - head) >> 4;
	const int r8 = (head & 3) * 8;
	uint4* dv = (uint4*)(dst + head);
	switch (head >> 2) {
	case 0: store_piece_vectors<0>(st, dv, nvec, r8, lane); break;
	case 1: store_piece_vectors<1>(st, dv, nvec, r8, lane); break;
	case 2: store_piece_vectors<2>(st, dv, nvec, r8, lane); break;
	default: store_piece_vectors<3>(st, dv, nvec, r8, lane); break;
	}
	const int t0 = head + (nvec << 4);
	if (lane < n - t0) dst[t0 + lane] = stGeneric[t0 + lane];
}

// (A continuous ring of pieces across blobs -- the next load issued as soon as a stage is stored -- was measured too: no
// faster, 4.10 vs 3.97 ms per step on 8 SMs; an SM moves 45-50 GB/s each way either way.)
__global__ void __launch_bounds__(MV_THREADS, 1) move_blobs_tma_kernel(const GenParams P) {
	extern __shared__ __align__(128) uint8_t mv_smem[];
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	uint8_t* ring = mv_smem + warp * MV_WARP_BYTES;
	const uint32_t ringS = (uint32_t)__cvta_generic_to_shared(ring);
	const uint32_t barS = ringS + MV_STAGES * MV_STAGE_BYTES;
	if (lane == 0) {
		for (int i = 0; i < MV_STAGES; i++) mbar_init(barS + 8u * i, 1u);
		asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
	}
	__syncwarp();
	uint32_t phase = 0;                               // one parity bit per stage
	const int nWarps = gridDim.x * MV_WARPS;
	for (int j = blockIdx.x * MV_WARPS + warp; j < P.nTiles; j += nWarps) {
		const unsigned long long excl = __ldcg(P.blobPrefix + j), mine = __ldcg(P.tileState + j);
		const unsigned long long d[2] = {excl >> 31, excl & 0x7fffffffull};
		const int len[2] = {(int)(mine >> 31), (int)(mine & 0x7fffffffull)};
		if (d[0] + (unsigned)len[0] > P.cap1 || d[1] + (unsigned)len[1] > P.cap2) continue;   // flagged by the scan
#pragma unroll 1
		for (int f = 0; f < 2; f++) {
			const uint8_t* src = (f ? P.out2 : P.out1) + (size_t)j * P.blobPitch;
			uint8_t* dst = (f ? P.dense2 : P.dense1) + d[f];
			const int nPieces = (len[f] + MV_PIECE - 1) / MV_PIECE;
#pragma unroll 1
			for (int p0 = 0; p0 < nPieces; p0 += MV_STAGES) {
				const int np = min(MV_STAGES, nPieces - p0);
				if (lane == 0) {
					// the stages were read with ordinary loads a moment ago: order those before the asynchronous writes
					asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
					for (int i = 0; i < np; i++) {
						const int off = (p0 + i) * MV_PIECE;
						const uint32_t bytes = (uint32_t)((min(MV_PIECE, len[f] - off) + 15) & ~15);
						mbar_expect_tx(barS + 8u * i, bytes);
						bulk_load(ringS + (uint32_t)(i * MV_STAGE_BYTES), src + off, bytes, barS + 8u * i);
					}
				}
				for (int i = 0; i < np; i++) {
					mbar_wait(barS + 8u * i, (phase >> i) & 1u);
					const int off = (p0 + i) * MV_PIECE;
					store_piece(ringS + (uint32_t)(i * MV_STAGE_BYTES), ring + i * MV_STAGE_BYTES, min(MV_PIECE, len[f] - off), dst + off, lane);
					phase ^= 1u << i;
				}
				__syncwarp();
			}
		}
	}
}

// Array output: zeroes bytes [m, pitch) of a read's base row (row0) and of its quality row (pitch bytes behind).  row0 and
// pitch are multiples of 16: bytes up to the next 16-byte boundary one lane each, the rest with 16-byte stores.
__device__ __forceinline__ void clear_rows(uint8_t* row0, int m, uint32_t pitch, int lane) {
	const int a = (m + 15) & ~15;
	const int i = m + (lane & 15);
	if (i < a) row0[(lane >> 4) * pitch + i] = 0;
	const int nv = ((int)pitch - a) >> 4;
	for (int v = lane; v < 2 * nv; v += 32) {
		const int r = v >= nv ? 1 : 0;
		*(uint4*)(row0 + r * pitch + a + 16 * (v - r * nv)) = make_uint4(0u, 0u, 0u, 0u);
	}
}

// ---------------------------------------------------------------------------------------------
// pass 1: generation into per-ticket blobs (FASTQ records), or, OUT_ARRAYS, into fixed slots of caller-owned arrays: the bases
// and the qualities of a read at [pair][mate][0 / 1][pitch] without record text, the read-name fields of a pair in arrays of
// their own.  OUT_FASTQ: one blob per ticket and file (PE: file 2's blob P.file2Off bytes behind file 1's); OUT_INTERLEAVED
// (PE only): one blob per ticket holding mate 1, mate 2 of every pair in turn, at pitch 2 x FG_CHUNK x FG_SLOT over both halves
// of the scratch.  Mate 2's header is written at the cursor behind mate 1's record, which is known once mate 1's indel scan
// has fixed its length.  OUT_BAM: the same blobs (PE: the interleaved layout) hold unaligned BAM records (bam.cuh): the name
// comes from the header code without '@', mate suffix and line feed, and the 36 fixed bytes and the read group tag are
// written once the read's length is known.
// ---------------------------------------------------------------------------------------------
template <int NCH, int QP, int OUT>
__global__ void __launch_bounds__(FG_THREADS, 1) generate_slots_kernel(const __grid_constant__ GenParams P) {
	constexpr bool ARRAYS = OUT == OUT_ARRAYS;
	constexpr bool ILV = OUT == OUT_INTERLEAVED;
	constexpr bool BAM = OUT == OUT_BAM;
	extern __shared__ __align__(16) uint8_t smem[];
	const DevTables& t = P.t;
	const int lane = threadIdx.x & 31;
	const int warp = threadIdx.x >> 5;
	const int nSubTotal = t.nSub * (t.useCdf2 ? 2 : 1);
	int qualBytes, qualSymBytes;
	fast_qual_bytes(t, QP, &qualBytes, &qualSymBytes);
	const int subPitch = fast_sub_pitch(t.B);
	const int nRowsTotal = nSubTotal / t.B;
	const FastLayout L = fast_layout(nRowsTotal * subPitch * (QP == 16 ? 8 : 16), qualBytes, qualSymBytes, t.nIsize, t.nInsLen, t.nDelLen);

	uint4* s_sub = (uint4*)(smem + L.sub);
	uint8_t* s_qual = smem + L.qual;
	uint8_t* s_qualSym = smem + L.qualSym;
	uint32_t* s_isizeT = (uint32_t*)(smem + L.isizeT);
	uint16_t* s_isizeSym = (uint16_t*)(smem + L.isizeSym);
	uint32_t* s_insT = (uint32_t*)(smem + L.insT);
	uint16_t* s_insSym = (uint16_t*)(smem + L.insSym);
	uint32_t* s_delT = (uint32_t*)(smem + L.delT);
	uint16_t* s_delSym = (uint16_t*)(smem + L.delSym);
	uint16_t* s_lut = (uint16_t*)(smem + L.lut);
	uint4* s_dig = (uint4*)(smem + L.dig);

	const int RL = t.RL, B = t.B;
	// shared-window address of the quality rows, folded into the substitution rows (QP == 8)
	const uint32_t qualBaseS = (QP == 8 || QP == 16) ? (uint32_t)__cvta_generic_to_shared(s_qual) : 0u;
	const uint32_t qstride = P.qstride;            // QP == 8: qualBins * F_QROW, else F_QROW
	// ---- stage the tables
	// substitution rows: word 3 becomes the byte offset of the quality row (ref, base) inside a bin block;
	// the three compare-adds then step it to (ref, call).  ref = last base of the context = row & 3.
#pragma unroll 1
	for (int i = threadIdx.x; i < nSubTotal; i += FG_THREADS) {
		uint4 v = t.sub[i];
		const int rowAll = i / B, bin = i - rowAll * B;
		const int row = rowAll % t.nRows;
		if (QP == 16) {
			// high halves of the three thresholds + the (ref, base) row
			((uint2*)s_sub)[rowAll * subPitch + bin] = make_uint2((v.x >> 16) | (v.y & 0xffff0000u), (v.z >> 16) | (((uint32_t)(row & 3) * 4u + v.w) << 16));
		} else {
			v.w = qualBaseS + ((uint32_t)(row & 3) * 4u + v.w) * qstride;
			s_sub[rowAll * subPitch + bin] = v;
		}
	}
	if (QP == 16) {
		// [ref*4+call][bin] rows of 40 keys (high halves of the thresholds; rows are padded with 0xFFFFFFFF) + 40 symbols
#pragma unroll 1
		for (int i = threadIdx.x; i < t.nQualRows * F_Q16_KEYS; i += FG_THREADS) {
			const int r = i / F_Q16_KEYS, k = i - r * F_Q16_KEYS;
			const int src = r * t.qualPitch + (k < t.qualPitch ? k : t.qualPitch - 1);
			uint8_t* row = s_qual + r * F_Q16_ROW;
			((uint16_t*)row)[k] = k < t.qualPitch ? (uint16_t)(t.qualT[src] >> 16) : (uint16_t)0xffffu;
			row[2 * F_Q16_KEYS + k] = t.qualSym[src];
		}
	} else if (QP == 8) {
		// [ref*4+call][bin][8] x {threshold, sym | char << 8}: the rows one warp instruction touches (about eleven bins x
		// four ref == call rows) spread over the banks; t.qualBins >= B pads the (ref, call) blocks for that
#pragma unroll 1
		for (int i = threadIdx.x; i < t.nQualRows * 8; i += FG_THREADS) {
			const int r = i >> 3, k = i & 7;
			const int rc = r / B, bin = r - rc * B;
			uint32_t* dst = (uint32_t*)(s_qual + (rc * t.qualBins + bin) * F_QROW + k * 8);
			dst[0] = t.qualT[i];
			dst[1] = (uint32_t)t.qualSym[i] | (((t.baseChars >> (8 * (rc & 3))) & 0xffu) << 8);
		}
	} else if (QP == 2) {
#pragma unroll 1
		for (int i = threadIdx.x; i < 4 * B * t.qualDiagPitch; i += FG_THREADS) {
			const int r = i / t.qualDiagPitch, k = i - r * t.qualDiagPitch;
			((uint32_t*)s_qual)[r * (t.qualDiagPitch + 1) + k] = t.qualDiagT[i];
			s_qualSym[r * (t.qualDiagPitch + 1) + k] = t.qualDiagSym[i];
		}
	}
#pragma unroll 1
	for (int i = threadIdx.x; i < t.nIsize; i += FG_THREADS) { s_isizeT[i] = t.isizeT[i]; s_isizeSym[i] = t.isizeSym[i]; }
#pragma unroll 1
	for (int i = threadIdx.x; i < t.nInsLen; i += FG_THREADS) { s_insT[i] = t.insLenT[i]; s_insSym[i] = t.insLenSym[i]; }
#pragma unroll 1
	for (int i = threadIdx.x; i < t.nDelLen; i += FG_THREADS) { s_delT[i] = t.delLenT[i]; s_delSym[i] = t.delLenSym[i]; }
#pragma unroll 1
	for (int i = threadIdx.x; i < F_LUT_N; i += FG_THREADS) {
		// context LUT: index = variant << 6 | b0 | b1 << 2 | b2 << 4 (three consecutive store bases), value = entry
		// index of the substitution row.  forward: (b0,b1,b2) = cycles (j-2, j-1, j); reverse: raw bases of cycles
		// (j, j-1, j-2).  Cycles 0 and 1 have the 'X' padded contexts (Profile.cpp:1661-1666, rows 0..19).
		const int v = i & 63, var = i >> 6;
		const bool rev = var == 1 || var >= 4;
		const uint32_t b0 = v & 3, b1 = (v >> 2) & 3, b2 = (v >> 4) & 3;
		uint32_t cur, p1, p2;
		if (!rev) { p2 = b0; p1 = b1; cur = b2; }
		else { cur = (t.compLut >> (2 * b0)) & 3u; p1 = (t.compLut >> (2 * b1)) & 3u; p2 = (t.compLut >> (2 * b2)) & 3u; }
		const int cyc = var < 2 ? 2 : ((var - 2) & 1);
		const uint32_t row = cyc == 0 ? cur : (cyc == 1 ? 4u + 4u * p1 + cur : 20u + 16u * p2 + 4u * p1 + cur);
		s_lut[i] = (uint16_t)(row * (uint32_t)subPitch);
	}
	if (threadIdx.x < 32) {
		// header digits: lanes 0..9 digit d of the position, lanes 10..19 digit d of the fragment counter
		const int d = lane < 10 ? lane : (lane < 20 ? lane - 10 : 0);
		s_dig[lane] = make_uint4(lane < 20 ? c_pow10[d] : 0xFFFFFFFFu /* digit d exists iff value >= 10^d */, c_divM[d], c_divS[d], d == 0);
	}
	__syncthreads();

	const int nMates = t.paired ? 2 : 1;
	uint8_t* wbase = smem + L.warp + warp * L.perWarp;
	WarpCtx w;
	w.B = t.B; w.subPitch = subPitch; w.minQ = t.minQ; w.RL = t.RL; w.nInsLen = t.nInsLen; w.nDelLen = t.nDelLen;
	w.nBasesM1 = t.N - 1; w.mDelta = 0; w.baseChars = t.baseChars; w.compLut = t.compLut;
	w.q.rows = s_qual; w.q.qbins = t.qualBins; w.q.diagT = (const uint32_t*)s_qual; w.q.diagSym = s_qualSym;
	w.q.gT = t.qualT; w.q.gSym = t.qualSym; w.q.pitch = t.qualPitch; w.q.diagPitch = t.qualDiagPitch;
	w.insT = s_insT; w.insSym = s_insSym; w.delT = s_delT; w.delSym = s_delSym;
	w.win = (const uint32_t*)(wbase + L.w_win);
	const uint32_t* s_win0 = (const uint32_t*)(wbase + L.w_win);
	// destination of this lane's window word (cp.async), shared-window address
	const uint32_t winS = (uint32_t)__cvta_generic_to_shared(wbase + L.w_win) + 4u * lane;
	w.ev = (uint32_t*)(wbase + L.w_ev); w.insb = wbase + L.w_insb;
	w.insp = (uint32_t*)(wbase + L.w_insp) + 1; w.outw = (uint32_t*)(wbase + L.w_out) + 1;
	w.rk = P.rk;
	w.qualBaseS = qualBaseS; w.qstride = qstride;
	w.lane = lane;

	// ---- per-lane constants
	// bin of output position j = j*B/RL (Profile.cpp:1671) for an indel-free read, as the byte offset of that bin's
	// substitution row entry; lanes past the read end (last chunk only) are clamped so that every table index stays valid
	uint32_t binOf[NCH];
#pragma unroll
	for (int c = 0; c < NCH; c++) {
		int j = c * 32 + lane;
		if (j > RL - 1) j = RL - 1;
		binOf[c] = (uint32_t)((j * B) / RL);
	}
	// insertion / deletion candidate tests as "u < limit" (0 = disabled); a limit of 2^32 forces the slow path
	// (P.insLim / P.delLim / P.alwaysSlow, computed by the host, are constant-bank operands: no registers)
	const bool foldTail = ((RL + 31) >> 5) == NCH && (RL & 31) >= 1 && (RL & 31) <= 29;
	const int jLast = (NCH - 1) * 32 + lane;
	const uint32_t lutFwd0 = (lane == 0 ? 2u : (lane == 1 ? 3u : 0u)) * 128u;
	const uint32_t lutRev0 = (lane == 0 ? 4u : (lane == 1 ? 5u : 1u)) * 128u;
	const uint8_t* lutB = (const uint8_t*)s_lut;
	w.lutB = lutB;
	const uint32_t baseChars = t.baseChars;
	const uint32_t one = P.one;

	// window prefetch: lanes 0..15 fetch data words (16 bases each), lanes 16..24 mask words (32 bases each)
	const uint32_t* winPtr = lane < 16 ? P.hap2 + lane : P.hapN + (lane - 16);
	const int winHalf = lane < 16 ? 0 : 1;            // a mask word covers 32 bases, a data word 16

	while (true) {
		// ---- a ticket = FG_CHUNK consecutive pairs
		int chunk = 0;
		if (lane == 0) chunk = (int)atomicAdd(P.ticket, 1u);
		chunk = __shfl_sync(0xffffffffu, chunk, 0);
		if (chunk >= P.nTiles) break;
		// slot = pair index inside the batch (a batch has < 2^31 / FG_SLOT pairs)
		const uint32_t slot0 = (uint32_t)chunk * FG_CHUNK;
		const uint32_t nSlots = (uint32_t)(P.emitHi - P.emitLo);
		const int count = (int)(slot0 + FG_CHUNK < nSlots ? FG_CHUNK : nSlots - slot0);
		uint32_t acc = 0;                                // bases | haplotype bytes << 16 of this ticket
		// next free byte of this ticket's two blobs, relative to P.out1 (file 2's blobs lie P.file2Off bytes behind file 1's in the
		// same allocation; scratch < 2^32 bytes).
		// posA belongs to the file of the current mate: the two cursors change places after every mate of a pair (interleaved
		// output: posA is the one cursor of the ticket's blob, posB is not used).
		const uint32_t blobBase = (uint32_t)chunk * P.blobPitch;
		uint32_t posA = blobBase, posB = blobBase + P.file2Off;

		// ---- ticket prologue, lane-parallel: lane L prepares pair slot0 + L (bin, pair ID, fragment draw, header digit counts);
		// the pair loop below fetches these by shuffle instead of every lane repeating the same scalar work for every pair
		uint32_t k_pairLo, k_pairHi, k_winA, k_winB, k_g, k_posmod, k_frag, k_name;
		{
			const uint32_t mySlot = slot0 + (uint32_t)(lane < count ? lane : count - 1);
			const int b0 = P.tileStartBin[chunk];
			// bin of my pair: bins hold >= 1 pair, so it is one of b0 .. b0+31; lane i looks at the first pair of bin b0+1+i
			const int64_t probe = (int64_t)b0 + 1 + lane;
			const int64_t startRel64 = probe <= P.nBins ? P.emitBase[probe] - P.emitLo : 0x7fffffffLL;
			const uint32_t startRel = startRel64 > 0x7fffffffLL ? 0x7fffffffu : (uint32_t)startRel64;
			int cnt = 0;                                 // number of those bins that start at or before my pair (starts ascend)
#pragma unroll
			for (int step = 16; step > 0; step >>= 1) {
				const int tprobe = cnt + step - 1;
				const uint32_t sv = __shfl_sync(0xffffffffu, startRel, tprobe & 31);
				if (tprobe <= 30 && sv <= mySlot) cnt += step;
			}
			const DevBin bin = P.bins[b0 + cnt];
			const int ord = (int)((int64_t)mySlot - (bin.emit_base - P.emitLo));
			const uint64_t pair = (uint64_t)(bin.plan_base + ord);
			const uint32_t fragCount = (uint32_t)(bin.frag_base + ord + 1);
			uint32_t attempt = 0;
			if (bin.risky_base >= 0) attempt = P.riskyAttempt[bin.risky_base + ord];
			// fragment (Segment.cpp:743-751)
			const u32x4 fb = philox_rk((uint32_t)pair, (uint32_t)(pair >> 32), (uint32_t)STREAM_FRAG << 24, attempt, P.rk);
			const long long pos = f_draw_pos(fb.x, bin.spos, bin.epos);
			long long want;
			if (!t.paired) want = (long long)bin.epos - bin.spos + 1;
			else if (t.nIsize > 0) want = t.minIS + uni_lookup(s_isizeT, s_isizeSym, t.nIsize, fb.y);
			else want = t.fixedInsert;
			const int64_t fstart = bin.hap_base + pos;
			const long long avail = bin.contig_end - fstart;
			const int flen = (int)(want < avail ? want : avail);
			uint32_t posmod = (uint32_t)pos;                                             // pos % segsize: only copies past the first need the division
			if (posmod >= bin.segsize) posmod %= bin.segsize;
			const bool seReverse = (!t.paired) && ((fb.z >> 31) != 0);                   // randomInteger(0, 2) != 0
			uint32_t hapB = lane < count ? min((uint32_t)((flen + 3) / 4 + (flen + 7) / 8), 2047u) : 0u;   // haplotype bytes (statistics)
#pragma unroll
			for (int d = 16; d > 0; d >>= 1) hapB += __shfl_xor_sync(0xffffffffu, hapB, d);
			acc = hapB << 16;
			k_pairLo = (uint32_t)pair; k_pairHi = (uint32_t)(pair >> 32);
			// window origins of the two mates (first template base in the store): data word index of base g0 - 32, and the low
			// five bits of g0 (the mask word index is half the data word index)
			const int64_t g0b = fstart + flen - RL;
			const int64_t g0a = seReverse ? g0b : fstart;
			k_winA = (uint32_t)((uint64_t)(g0a - 32) >> 4); k_winB = (uint32_t)((uint64_t)(g0b - 32) >> 4);
			k_g = ((uint32_t)g0a & 31u) | (((uint32_t)g0b & 31u) << 8) | (seReverse ? 0x80000000u : 0u);
			k_posmod = posmod; k_frag = fragCount;
			// name_off (17 bits) | name_len << 17 (7 bits) | digits of posmod << 24 | digits of fragCount << 28
			k_name = (uint32_t)bin.name_off | ((uint32_t)bin.name_len << 17) | ((uint32_t)f_ndigits(posmod) << 24) | ((uint32_t)f_ndigits(fragCount) << 28);
			if (ARRAYS && lane < count) {
				// the read-name fields of pair slot0 + L, one coalesced store per array
				const uint32_t row = slot0 + (uint32_t)lane;
				P.rdPairId[row] = (int64_t)pair; P.rdSegment[row] = bin.segment;
				P.rdPos[row] = (int32_t)posmod; P.rdFrag[row] = (int32_t)fragCount;
			}
		}

#pragma unroll 1
		for (int p = 0; p < count; p++) {
			w.c0 = __shfl_sync(0xffffffffu, k_pairLo, p); w.c1 = __shfl_sync(0xffffffffu, k_pairHi, p);
			const uint32_t kg = __shfl_sync(0xffffffffu, k_g, p);
			const uint32_t posmod = __shfl_sync(0xffffffffu, k_posmod, p), fragCount = __shfl_sync(0xffffffffu, k_frag, p);
			const uint32_t nameNd = __shfl_sync(0xffffffffu, k_name, p);
			const bool seReverse = (kg >> 31) != 0;

			// ---- prefetch the packed windows of both mates (data words lanes 0..15, mask words lanes 16..24)
			// (global -> shared without passing through registers; waited for after phase A of the first mate)
			const uint32_t g0lo = kg & 0x1f1fu;              // low five bits of the two window origins
			{
				const uint32_t wA = __shfl_sync(0xffffffffu, k_winA, p), wB = __shfl_sync(0xffffffffu, k_winB, p);
				if (lane < 25) {
					cp_async4(winS, winPtr + (wA >> winHalf));
					cp_async4(winS + F_WIN_WORDS * 4, winPtr + (wB >> winHalf));
				}
				cp_async_commit();
			}

			// ---- header digits: lanes 0..9 digit d of posmod, lanes 10..19 digit d of fragCount
			const uint32_t dsrc = lane < 10 ? posmod : fragCount;
			const uint4 dc = s_dig[lane];                                            // {10^d (unused here), M, S, d == 0}
			const int nd1 = (int)((nameNd >> 24) & 15u), nd2 = (int)(nameNd >> 28);
			uint32_t qd = __umulhi(dsrc, dc.y) >> dc.z;
			if (dc.w) qd = dsrc;
			const uint32_t dg = qd - 10u * (__umulhi(qd, 0xCCCCCCCDu) >> 3) + '0';
			const int nameLen = (int)((nameNd >> 17) & 127u), nameOff = (int)(nameNd & 0x1ffffu);
			// BAM: the name (header characters 1 .. nameEnd, the last one a NUL) starts at byte 36 of the record
			const int nameEnd = nameLen + nd1 + 1 + nd2;
			const int H = ARRAYS ? 0 : BAM ? BAM_FIXED + nameEnd : nameLen + nd1 + 1 + nd2 + (t.paired ? 2 : 0) + 1;   // array output: no header
			const int hWords = ((BAM ? nameEnd + 1 : H) + 31) >> 5;
			const uint32_t slash = BAM ? 0u : t.paired ? (uint32_t)'/' : (uint32_t)'\n';
			const int mateAt = t.paired ? H - 2 : -1;
			uint32_t hdr = 0;                                                        // interleaved: this lane's header characters, byte r
#pragma unroll
			for (int r = 0; r < 3; r++) {
				if (ARRAYS || r >= hWords) break;
				// character i of the header: name | digits of pos % segsize (most significant first) | '#' | digits of the
				// fragment counter | "/1\n" or "\n" -- selected without branches; the digits come from lanes 0..19 by shuffle
				const int i = lane + 32 * r;
				const int k = i - nameLen, k2 = k - nd1 - 1;
				const bool d1 = (unsigned)k < (unsigned)nd1, d2 = (unsigned)k2 < (unsigned)nd2;
				const int srcLane = d1 ? nd1 - 1 - k : 9 + nd2 - k2;
				const uint32_t dv = __shfl_sync(0xffffffffu, dg, srcLane & 31);
				uint32_t ch = k == nd1 ? (uint32_t)'#' : (k2 == nd2 ? slash : (uint32_t)'\n');
				ch = (d1 || d2) ? dv : ch;
				if (r < 2 && k < 0) ch = (uint8_t)P.names[nameOff + i];          // names are at most 64 bytes
				// straight into both records of the pair (the cursors of file 1 / file 2 are posA / posB here); only the mate
				// digit in front of the final '\n' differs
				if (BAM) {
					if (i >= 1 && i <= nameEnd) P.out1[posA + (BAM_FIXED - 1) + i] = (uint8_t)ch;
				} else if (i < H) {
					const bool mateDigit = i == mateAt;
					P.out1[posA + i] = (uint8_t)(mateDigit ? (uint32_t)'1' : ch);
					if (t.paired && !ILV) P.out1[posB + i] = (uint8_t)(mateDigit ? (uint32_t)'2' : ch);
				}
				if (ILV || BAM) hdr |= (ch & 0xffu) << (8 * r);                        // mate 2's header (name), written behind mate 1's record
			}

#pragma unroll 1
			for (int mate = 0; mate < nMates; mate++) {
				const bool rev = (mate == 1) || seReverse;
				const uint32_t g5 = (mate == 0 ? g0lo : (g0lo >> 8)) & 31u;   // window = bases [g0 - 32 rounded down to 32, ...)
				const int dOff = (int)(g5 & 15u) + 32;         // index of base g0 relative to data word 0
				const int mOff = (int)g5 + 32;                 // same, relative to mask word 0 (32 bases per word)
				const uint32_t* s_win = s_win0 + (mate == 0 ? 0 : F_WIN_WORDS);
				w.win = s_win;
				w.mDelta = mOff - dOff;
				const uint32_t c2cyc = ((uint32_t)mate << 28) | ((uint32_t)STREAM_CYCLE << 24);
				// array output: the read's slot, (pair * M + mate) * 2 * pitch bytes into the batch (< 2^32, clamped by the host)
				const uint32_t readIdx = (slot0 + (uint32_t)p) * (uint32_t)nMates + (uint32_t)mate;
				uint8_t* stage = ARRAYS ? P.out1 + readIdx * 2u * P.pitch : P.out1 + posA;
				const uint4* subM = s_sub + ((mate == 1 && t.useCdf2) ? t.nRows * subPitch : 0);
				w.sub = subM;
				if (QP == 16) {
					w.sub16S = (uint32_t)__cvta_generic_to_shared(s_sub) + ((mate == 1 && t.useCdf2) ? (uint32_t)(t.nRows * subPitch) * 8u : 0u);
					w.gsub = t.sub + ((mate == 1 && t.useCdf2) ? t.nSub : 0);
				}

				// ---- phase A: one Philox block per cycle (chunks interleaved); indel candidates at reference position j
				uint32_t x0[NCH], x1[NCH], x2[NCH], x3[NCH];
				bool cand = false;
				philox_chunks<NCH>(w.c0, w.c1, c2cyc, (uint32_t)lane, P.rk, x0, x1, x2, x3);
#pragma unroll
				for (int c = 0; c < NCH; c++) {
					const bool hit = (x0[c] < P.insLim) | (x1[c] < P.delLim);
					cand |= (c == NCH - 1) ? (hit && jLast < RL) : hit;
				}
				if (mate == 0) { cp_async_wait_all(); __syncwarp(); }
				// any non-ACGT base in the 288-base window also goes the slow way
				const bool slow = __any_sync(0xffffffffu, cand || (lane >= 16 && lane < 25 && s_win[lane] != 0u)) || P.alwaysSlow;

				int m = RL;
				if (!slow) {
					// ---- phase C, fast path (branch free): context straight from the packed window.
					// forward: window of cycle j starts at base g0 + j - 2; reverse: at base g0 + RL-1 - j
					const int rel0 = rev ? (dOff + RL - 1 - lane) : (dOff + lane - 2);
					const uint32_t dsh = (uint32_t)(rel0 & 15) * 2u;
					const uint32_t* dptr = w.win + (rel0 >> 4);
					const int dstep = rev ? -2 : 2;
					const uint8_t* lut0 = lutB + (rev ? lutRev0 : lutFwd0);
					const uint8_t* lutN = lutB + (rev ? 128 : 0);
					const uint8_t* subMB = (const uint8_t*)subM;
					uint8_t* st1 = stage + H + lane;
					uint8_t* st2 = ARRAYS ? st1 + P.pitch : st1 + RL + 3;
					uint8_t* sq1 = stage + H + (lane >> 1);                               // BAM: bases, 16 bytes per chunk
					uint8_t* sq2 = stage + H + ((RL + 1) >> 1) + lane;                     // BAM: qualities
#pragma unroll
					for (int c = 0; c < NCH; c++) {
						const uint32_t v6 = __funnelshift_r(dptr[c * dstep], dptr[c * dstep + 1], dsh) & 63u;
						const uint32_t rowIdx = *(const uint16_t*)((c == 0 ? lut0 : lutN) + v6 * 2u);
						uint32_t ch, q;
						uint4 sr = make_uint4(0u, 0u, 0u, 0u);
						uint32_t acc = 0;
						if (QP == 16) lookup16(w, rowIdx, binOf[c], x2[c], x3[c], false, 0u, ch, q);
						else {
							sr = *(const uint4*)(subMB + (rowIdx + binOf[c]) * 16u);
							acc = sr.w;
							fadd_gt(acc, x2[c], sr.x, P.qstride, one);
							fadd_gt(acc, x2[c], sr.y, P.qstride, one);
							fadd_gt(acc, x2[c], sr.z, P.qstride, one);
						}
						if (QP == 16) {
						} else if (QP == 8) {
							uint32_t qa = binOf[c] * (uint32_t)F_QROW + acc;         // shared address of row (ref, call, bin)
							fadd_lt(qa, lds_u32(qa + 24), x3[c], 32u, one);
							fadd_lt(qa, lds_u32(qa + 8), x3[c], 16u, one);
							fadd_lt(qa, lds_u32(qa), x3[c], 8u, one);
							q = lds_u16(qa + 4);                                     // symbol | base character << 8
							ch = q >> 8;
						} else {
							const uint32_t r16 = acc / (uint32_t)F_QROW;             // qualBaseS == 0 here
							const uint32_t call = r16 & 3u;
							q = qual_lookup<QP>(w.q, r16 >> 2, call, binOf[c], B, x3[c]);
							ch = __byte_perm(baseChars, 0, 0x4440u | call);
						}
						if (BAM) {
							put_base<OUT>(sq1 + c * 16, sq2 + c * 32, c < NCH - 1 || jLast < RL, ch, q, lane);
						} else if (c < NCH - 1) {
							st1[c * 32] = (uint8_t)ch;
							st2[c * 32] = (uint8_t)q;
						} else if (ARRAYS) {
							if (jLast >= RL) { ch = 0u; q = 0u; }                  // lanes past the read end zero their bytes
							st1[c * 32] = (uint8_t)ch;
							st2[c * 32] = (uint8_t)q;
						} else if (foldTail) {
							// "\n+\n" after the bases and the final '\n' ride on the idle lanes of the last chunk
							if (jLast >= RL) { ch = (jLast == RL + 1) ? '+' : '\n'; q = '\n'; }
							if (jLast < RL + 3) st1[c * 32] = (uint8_t)ch;
							if (jLast < RL + 1) st2[c * 32] = (uint8_t)q;
						} else if (jLast < RL) {
							st1[c * 32] = (uint8_t)ch;
							st2[c * 32] = (uint8_t)q;
						}
					}
					if (ARRAYS) clear_rows(stage, 32 * NCH, P.pitch, lane);
					else if (!BAM && !foldTail && lane == 0) { stage[H + m] = '\n'; stage[H + m + 1] = '+'; stage[H + m + 2] = '\n'; stage[H + 2 * m + 3] = '\n'; }
				} else {
					uint32_t evbits = 0;
#pragma unroll
					for (int c = 0; c < NCH; c++) {
						const bool valid = c < NCH - 1 || jLast < RL;
						const bool ins = valid && t.insEnable && x0[c] <= t.insT;        // p <= insertRate, Profile.cpp:1560-1561
						const bool del = valid && t.delEnable && x1[c] <= t.delT;        // p2 < delRate/(1-insertRate), :1569-1570
						if (ins) evbits |= 1u << (2 * c);
						else if (del) evbits |= 2u << (2 * c);
					}
					IndelPlan pl = scan_events(w, evbits, mate, &P.result->errorFlags);
					if (ARRAYS && pl.m > RL + 96) {
						// longer than a slot holds (pitch >= RL + 96): flagged as a read that outgrew the scratch, nothing written past the slot
						if (lane == 0) atomicOr(&P.result->errorFlags, 2u);
						pl.nEv = 0; pl.m = RL; pl.insTotal = 0;
					}
					m = pl.m;
					// a non-ACGT base in the window, or a read that outgrew the NCH chunks of draws: position-by-position path
					const bool hasN = __any_sync(0xffffffffu, lane >= 16 && lane < 25 && s_win[lane] != 0u);
					if (hasN || m > 32 * NCH || P.noSplice) {
						const int relFirst = rev ? (dOff + RL - 1) : dOff;
						emit_mapped<NCH, QP, OUT>(w, pl, mate, rev, relFirst, stage, H, P.pitch, x2, x3);
					} else {
						if (pl.nEv) splice_read(w, pl, rev, dOff);
						emit_packed<NCH, QP, OUT>(w, pl.nEv ? w.outw : s_win, dOff, rev, m, rev ? lutRev0 : lutFwd0, rev ? 128u : 0u, stage, H,
						                             P.pitch, x2, x3);
					}
					if (ARRAYS) clear_rows(stage, m, P.pitch, lane);
					else if (!BAM && lane == 0) { stage[H + m] = '\n'; stage[H + m + 1] = '+'; stage[H + m + 2] = '\n'; stage[H + 2 * m + 3] = '\n'; }
				}
				if (ARRAYS && lane == 0) P.rdLength[readIdx] = (int16_t)m;
				if (BAM) {
					const uint32_t tail = bam_tail_bytes((uint32_t)nameEnd, (uint32_t)m, (uint32_t)P.rgLen);
					bam_fixed(stage, (uint32_t)nameEnd, t.paired ? (mate == 0 ? BAM_FLAG_PE1 : BAM_FLAG_PE2) : BAM_FLAG_SE, (uint32_t)m,
					          (uint32_t)P.rgLen, lane);
					bam_read_group(stage + BAM_FIXED + tail - P.rgLen - 4, P.rg, P.rgLen, lane);
					posA += (uint32_t)BAM_FIXED + tail;
					if (mate == 0 && nMates == 2) {
#pragma unroll
						for (int r = 0; r < 3; r++) {                                        // mate 2's name is mate 1's
							const int i = lane + 32 * r;
							if (i >= 1 && i <= nameEnd) P.out1[posA + (BAM_FIXED - 1) + i] = (uint8_t)((hdr >> (8 * r)) & 0xffu);
						}
					}
				} else {
					posA += (uint32_t)(H + 2 * m + 4);
					if (ILV) {
						if (mate == 0) {
#pragma unroll
							for (int r = 0; r < 3; r++) {
								const int i = lane + 32 * r;
								if (i < H) P.out1[posA + i] = (uint8_t)(i == mateAt ? (uint32_t)'2' : (hdr >> (8 * r)) & 0xffu);
							}
						}
					} else if (nMates == 2) { const uint32_t tswap = posA; posA = posB; posB = tswap; }
				}
				acc += (uint32_t)m;                                                    // bases of the ticket (<= 2^14)
				__syncwarp();
			}
		}
		{
			const uint32_t ticket = (uint32_t)chunk;
			const uint32_t len1 = posA - blobBase, len2 = (nMates == 2 && !ILV && !BAM) ? posB - blobBase - P.file2Off : 0u;
			if (lane == 0) {
				if (!ARRAYS) P.tileState[ticket] = ((unsigned long long)len1 << 31) | len2;   // blob lengths, scanned by pass 2
				const uint32_t nPairs = (uint32_t)count;
				atomicAdd(&P.result->bases, (unsigned long long)(acc & 0xffffu)); atomicAdd(&P.result->hapBytes, (unsigned long long)(acc >> 16));
				atomicAdd(&P.result->pairs, (unsigned long long)nPairs); atomicAdd(&P.result->reads, (unsigned long long)(nPairs * nMates));
				if (!ARRAYS) atomicAdd(&P.result->rawBytes, (unsigned long long)len1 + len2);
			}
		}
	}

}

// Bins per (ref, call) block of the shared-memory quality image.  The three probes of a quality search are one word per
// lane at row (ref, call, bin); the 32 lanes of a warp instruction cover about RL/32 consecutive bins and mostly the four
// ref == call rows.  The candidate in [B, B + 8) with the fewest bank conflicts on a deterministic sample of such access
// patterns wins (bin-major rows, the first layout, cost 4.7 wavefronts per probe; this one about 2).
int fast_choose_qbins(int B, int RL) {
	int best = B; long bestScore = -1;
	for (int qb = B; qb < B + 8; qb++) {
		long score = 0;
		uint32_t lcg = 12345u;
		for (int trial = 0; trial < 64; trial++) {
			for (int c = 0; c * 32 < RL; c++) {
				int nAddr[32] = {0}; int addr[32][32];
				for (int lane = 0; lane < 32; lane++) {
					int j = c * 32 + lane; if (j > RL - 1) j = RL - 1;
					lcg = lcg * 1664525u + 1013904223u;
					const int ref = (int)(lcg >> 30);
					const int word = ((ref * 5) * qb + (j * B) / RL) * (F_QROW / 4) + 6;
					int* a = addr[word & 31]; int& n = nAddr[word & 31];
					bool seen = false;
					for (int i = 0; i < n; i++) seen |= a[i] == word;
					if (!seen) a[n++] = word;
				}
				int worst = 0;
				for (int b = 0; b < 32; b++) worst = nAddr[b] > worst ? nAddr[b] : worst;
				score += worst;
			}
		}
		if (bestScore < 0 || score < bestScore) { bestScore = score; best = qb; }
	}
	return best;
}

bool fast_supported(const DevTables& t, int smemLimit, int* qmode, size_t* smemBytes) {
	if (t.N != 4 || t.K != 3 || t.RL > 160 || t.RL < 33 || t.nIsize > 1024 || t.B > 160) return false;
	const int nSubTotal = t.nSub * (t.useCdf2 ? 2 : 1);
	// 8: all quality rows (<= 8 live symbols) in shared memory, 32-bit; 16: all rows (<= 40 live symbols) with 16-bit keys;
	// 2: only the ref == call rows; 0: quality table in global memory
	const int modes[4] = {8, 16, 2, 0};
	for (int k = 0; k < 4; k++) {
		if (t.fastQmode >= 0 && modes[k] != t.fastQmode) continue;
		if (modes[k] == 8 && t.qualPitch != 8) continue;
		if (modes[k] == 16 && t.maxQualRow > F_Q16_KEYS) continue;
		int qb, qs;
		fast_qual_bytes(t, modes[k], &qb, &qs);
		const int total = fast_layout(nSubTotal / t.B * fast_sub_pitch(t.B) * (modes[k] == 16 ? 8 : 16), qb, qs, t.nIsize, t.nInsLen, t.nDelLen).total;
		if (total <= smemLimit) { *qmode = modes[k]; *smemBytes = (size_t)total; return true; }
	}
	return false;
}

template <int NCH, int QP, int OUT>
static cudaError_t launch_fast_variant(const GenParams& P, size_t smemBytes, int grid, cudaStream_t stream) {
	auto kern = generate_slots_kernel<NCH, QP, OUT>;
	cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemBytes);
	if (e != cudaSuccess) return e;
	kern<<<grid, FG_THREADS, smemBytes, stream>>>(P);
	return cudaGetLastError();
}

// chunks of 32 cycles of the fast kernel instance for read length RL (33..160): exact, only the last chunk has idle lanes
int fast_nch(int RL) { return RL <= 64 ? 2 : (RL + 31) / 32; }

template <int OUT>
static cudaError_t launch_fast_instance(const GenParams& P, int qmode, size_t smemBytes, int grid, cudaStream_t stream) {
	const int nch = fast_nch(P.t.RL);
	if (qmode == 8) {
		if (nch == 2) return launch_fast_variant<2, 8, OUT>(P, smemBytes, grid, stream);
		if (nch == 3) return launch_fast_variant<3, 8, OUT>(P, smemBytes, grid, stream);
		if (nch == 4) return launch_fast_variant<4, 8, OUT>(P, smemBytes, grid, stream);
		return launch_fast_variant<5, 8, OUT>(P, smemBytes, grid, stream);
	} else if (qmode == 16) {
		if (nch == 2) return launch_fast_variant<2, 16, OUT>(P, smemBytes, grid, stream);
		if (nch == 3) return launch_fast_variant<3, 16, OUT>(P, smemBytes, grid, stream);
		if (nch == 4) return launch_fast_variant<4, 16, OUT>(P, smemBytes, grid, stream);
		return launch_fast_variant<5, 16, OUT>(P, smemBytes, grid, stream);
	} else if (qmode == 2) {
		if (nch == 2) return launch_fast_variant<2, 2, OUT>(P, smemBytes, grid, stream);
		if (nch == 3) return launch_fast_variant<3, 2, OUT>(P, smemBytes, grid, stream);
		if (nch == 4) return launch_fast_variant<4, 2, OUT>(P, smemBytes, grid, stream);
		return launch_fast_variant<5, 2, OUT>(P, smemBytes, grid, stream);
	}
	if (nch == 2) return launch_fast_variant<2, 0, OUT>(P, smemBytes, grid, stream);
	if (nch == 3) return launch_fast_variant<3, 0, OUT>(P, smemBytes, grid, stream);
	if (nch == 4) return launch_fast_variant<4, 0, OUT>(P, smemBytes, grid, stream);
	return launch_fast_variant<5, 0, OUT>(P, smemBytes, grid, stream);
}

// P.out1/out2 = blob scratch, P.dense1/dense2 = final slabs, P.nTiles = tickets of FG_CHUNK pairs.  Launches pass 1.
// interleaved (PE): one blob per ticket, P.blobPitch = 2 x FG_CHUNK x FG_SLOT.  bam: BAM records, PE in the interleaved layout.
cudaError_t launch_generate_fast(const GenParams& P, int qmode, size_t smemBytes, int grid, cudaStream_t stream, bool interleaved, bool bam) {
	if (bam) return launch_fast_instance<OUT_BAM>(P, qmode, smemBytes, grid, stream);
	return interleaved ? launch_fast_instance<OUT_INTERLEAVED>(P, qmode, smemBytes, grid, stream)
	                   : launch_fast_instance<OUT_FASTQ>(P, qmode, smemBytes, grid, stream);
}

// Array output: P.out1 = reads of the batch's first pair ([pair][mate][2][P.pitch], 16-byte aligned, pairs * M * 2 * pitch < 2^32),
// P.rdLength / rdPairId / rdSegment / rdPos / rdFrag at the same first pair, P.nTiles = tickets of FG_CHUNK pairs.
cudaError_t launch_generate_reads(const GenParams& P, int qmode, size_t smemBytes, int grid, cudaStream_t stream) {
	return launch_fast_instance<OUT_ARRAYS>(P, qmode, smemBytes, grid, stream);
}

// pass 2a alone: blob lengths P.tileState -> offsets P.blobPrefix, totals in P.result->bytes1/2
cudaError_t launch_scan_blobs(const GenParams& P, cudaStream_t stream) {
	scan_blobs_kernel<<<1, SC_THREADS, 0, stream>>>(P);
	return cudaGetLastError();
}

// pass 2b alone: blobs P.out1/out2 -> dense slabs P.dense1/dense2 at the offsets of the scan
cudaError_t launch_move_blobs(const GenParams& P, int smCount, cudaStream_t stream) {
	int cgrid = smCount * 8;
	if (cgrid * (CP_THREADS / 32) > P.nTiles) cgrid = (P.nTiles + CP_THREADS / 32 - 1) / (CP_THREADS / 32);
	if (cgrid < 1) cgrid = 1;
	move_blobs_kernel<<<cgrid, CP_THREADS, 0, stream>>>(P);
	return cudaGetLastError();
}

// pass 2b on `ctas` SMs (see move_blobs_tma_kernel): meant to run on a second stream under the next batch's generation kernel
cudaError_t launch_move_blobs_tma(const GenParams& P, int ctas, cudaStream_t stream) {
	const int smem = MV_WARPS * MV_WARP_BYTES;
	cudaError_t e = cudaFuncSetAttribute(move_blobs_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
	if (e != cudaSuccess) return e;
	move_blobs_tma_kernel<<<ctas, MV_THREADS, smem, stream>>>(P);
	return cudaGetLastError();
}

// pass 2: blobs P.out1/out2 with packed lengths P.tileState -> dense slabs P.dense1/dense2, totals in P.result->bytes1/2
cudaError_t launch_pass2(const GenParams& P, int smCount, cudaStream_t stream) {
	cudaError_t e = launch_scan_blobs(P, stream);
	if (e != cudaSuccess) return e;
	return launch_move_blobs(P, smCount, stream);
}

}  // namespace ssc
