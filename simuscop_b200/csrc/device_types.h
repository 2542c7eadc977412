// device_types.h -- structures shared between the host runtime (api.cu) and the kernels.
#pragma once
#include <cstdint>

namespace ssc {

// Compacted device bin (only bins that emit at least one pair), 64 bytes.
struct DevBin {
	int64_t hap_base;     // store index of segSequences[hap][0]
	int64_t contig_end;   // clip limit of the (population, chromosome, haplotype) contig
	int64_t plan_base;    // first planned pair ID of the bin (Philox key)
	int64_t emit_base;    // first emitted-pair index of the bin (output order)
	int32_t spos, epos;
	uint32_t segsize;
	int32_t frag_base;    // emitted pairs in earlier bins of the same segment (fragCount - 1 of ordinal 0)
	int32_t name_off, name_len;
	int32_t risky_base;   // index into riskyAttempt of ordinal 0, or -1 when attempt 0 always succeeds
	int32_t segment;      // index into the ssc_segment array of the plan (array output: the read-name prefix)
};
static_assert(sizeof(DevBin) == 64, "DevBin must be 64 bytes");

// Bin as seen by the census kernel (every bin flagged risky by the host).
struct CensusBin {
	int64_t hap_base, contig_end, plan_base;
	int32_t spos, epos;
	int32_t planned;      // planned pairs
	int32_t risky_base;
};

struct DevTables {
	int N, K, B, Q, minQ, RL, paired, useCdf2, fixedInsert, minIS, nRows;
	uint32_t insT, delT;
	int insEnable, delEnable;
	int nIsize, nInsLen, nDelLen;            // compressed lengths
	const uint32_t* isizeT; const uint16_t* isizeSym;
	const uint32_t* insLenT; const uint16_t* insLenSym;
	const uint32_t* delLenT; const uint16_t* delLenSym;
	const uint4* sub; int nSub;              // rows*B per read table; table of read 2 follows when useCdf2
	const uint32_t* qualT; const uint8_t* qualSym; int qualPitch; int nQualRows;
	int maxQualRow;                          // live symbols of the longest quality row
	int fastQmode;                           // tests: -1 = automatic, else the only quality-table mode fast_supported may choose
	int qualBins;                            // fast kernel: bins per (ref, call) block of the shared quality image (>= B, see fast_choose_qbins)
	const uint32_t* qualDiagT; const uint8_t* qualDiagSym; int qualDiagPitch;   // ref == call rows, [N*B][pitch]
	uint32_t compLut;
	uint32_t baseChars;                      // 4 ASCII characters, code i in byte i
	// FP64 ground-truth tables (the reference's own arrays)
	const double* f_isize; const double* f_ins; const double* f_del;
	const double* f_sub1; const double* f_sub2; const double* f_qual;
	int f_nIsize, f_nIns, f_nDel;
	double insertRate, delThresh;
};

struct BatchResult {
	unsigned long long bytes1, bytes2;
	unsigned long long bases, reads, pairs, hapBytes;
	unsigned int errorFlags;   // bit0: slab overflow, bit1: read outgrew scratch, bit2: too many indel events
	unsigned int pad;
	unsigned long long rawBytes;   // FASTQ bytes generated: fast kernel, generic kernel in gzip mode (bytes1/bytes2 are compressed sizes in gzip mode)
};

struct GenParams {
	DevTables t;
	const uint32_t* hap2;      // 2-bit codes, 16 bases per word
	const uint32_t* hapN;      // non-ACGT mask, 32 bases per word
	const DevBin* bins;
	const int64_t* emitBase;   // nBins+1 entries
	int64_t nBins;
	const uint16_t* riskyAttempt;
	const char* names;
	uint64_t seed;
	uint32_t rk[20];            // Philox round keys: rk[2r] = seed_lo + r*0x9E3779B9, rk[2r+1] = seed_hi + r*0xBB67AE85
	uint32_t insLim, delLim;    // fast kernel: candidate tests as u < limit (0 = disabled)
	int alwaysSlow;             // a rate of 1 (limit 2^32) sends every read down the slow path
	int noSplice;               // tests: reads with indel events always take the position-by-position path (emit_mapped)
	uint32_t one;               // 1, opaque to the compiler (see fadd_gt in gen_fast.cu)
	uint32_t qstride;           // fast kernel: bytes from quality row (ref, call) to (ref, call + 1): qualBins * 68 with all rows in shared memory, else 68
	int64_t emitLo, emitHi;    // emitted-pair index range of this batch
	const int32_t* tileStartBin;
	int nTiles;
	unsigned long long* tileState;
	unsigned long long* blobPrefix;   // fast kernel: exclusive prefix of the blob lengths (pass 2)
	unsigned int* ticket;       // work counter of the generation kernel (tiles / tickets of FG_CHUNK pairs), zeroed per launch
	uint8_t* out1; uint8_t* out2;       // generic kernel: final slabs (gzip mode: blob scratch); fast kernel: blob scratch (pass 1: out2 == out1 + file2Off)
	uint32_t blobPitch;                 // ticket blobs: bytes from the blob of ticket j to the blob of ticket j + 1 (pass 1 output, pass 2 / deflate input)
	uint32_t file2Off;                  // fast kernel, pass 1: file 2's blobs start this many bytes behind file 1's (one allocation, 32-bit cursors)
	uint8_t* dense1; uint8_t* dense2;   // ticket blobs: final slabs (pass 2)
	unsigned long long cap1, cap2;
	BatchResult* result;
	// array output (generate_slots_kernel<NCH, QP, true>): out1 = reads of the batch's first pair, [pair][mate][2][pitch];
	// the per-pair arrays start at the batch's first pair too
	int16_t* rdLength;          // [pair][mate]
	int64_t* rdPairId;
	int32_t* rdSegment; int32_t* rdPos; int32_t* rdFrag;
	uint32_t pitch;
	// BAM output: the read group id every record carries as RG:Z (device memory, rgLen bytes, 0 = no tag)
	const char* rg;
	int rgLen;
};

}  // namespace ssc
