// bam.cuh -- the pieces of an unaligned BAM record (SAM specification v1, section 4.2) that both generation kernels write.
//
// A record: block_size, 32 bytes of fixed fields (refID, pos, next_refID, next_pos -1; mapq 0; bin 4680 = reg2bin(-1, 0);
// n_cigar_op 0; tlen 0), the read name and its NUL, the bases as 4-bit codes (first base in the high nibble, a zero pad nibble
// behind an odd-length read), the qualities as phred values, then RG:Z:<id> when a read group is set.
#pragma once
#include <cstdint>

namespace ssc {

static constexpr int BAM_FIXED = 36;            // block_size + the fixed fields: the read name starts here
static constexpr uint32_t BAM_FLAG_PE1 = 77;    // paired, unmapped, mate unmapped, first in template
static constexpr uint32_t BAM_FLAG_PE2 = 141;   // paired, unmapped, mate unmapped, last in template
static constexpr uint32_t BAM_FLAG_SE = 4;      // unmapped

// 4-bit code of a base character: bits 1..3 of the ASCII code tell A, C, G, T and N apart (A 1, C 2, G 4, T 8, N 15)
__device__ __forceinline__ uint32_t bam_nibble(uint32_t ch) { return (0xF0004821u >> (((ch >> 1) & 7u) * 4u)) & 15u; }

// Bytes behind the fixed fields: name + NUL, bases, qualities, RG tag
__host__ __device__ __forceinline__ uint32_t bam_tail_bytes(uint32_t lReadName, uint32_t m, uint32_t rgLen) {
	return lReadName + ((m + 1u) >> 1) + m + (rgLen ? rgLen + 4u : 0u);
}

// The fixed part, bytes 0..35 of the record at rec: lane i writes byte i, lanes 0..3 also the four bytes of tlen.  Warp-wide.
__device__ __forceinline__ void bam_fixed(uint8_t* rec, uint32_t lReadName, uint32_t flag, uint32_t m, uint32_t rgLen, int lane) {
	const int wi = lane >> 2;
	uint32_t w = 0xffffffffu;                                                   // refID, pos, next_refID, next_pos
	if (wi == 0) w = (uint32_t)(BAM_FIXED - 4) + bam_tail_bytes(lReadName, m, rgLen);   // block_size
	if (wi == 3) w = lReadName | (4680u << 16);                                 // l_read_name, mapq, bin
	if (wi == 4) w = flag << 16;                                                // n_cigar_op, flag
	if (wi == 5) w = m;                                                         // l_seq
	rec[lane] = (uint8_t)(w >> (8 * (lane & 3)));
	if (lane < 4) rec[32 + lane] = 0;
}

// RG:Z:<id> NUL at dst (nothing when rgLen == 0).  Warp-wide.
__device__ __forceinline__ void bam_read_group(uint8_t* dst, const char* rg, int rgLen, int lane) {
	if (rgLen == 0) return;
	for (int i = lane; i < rgLen + 4; i += 32)
		dst[i] = i == 0 ? 'R' : i == 1 ? 'G' : i == 2 ? 'Z' : (i < rgLen + 3 ? (uint8_t)rg[i - 3] : 0);
}

// One base of a chunk of 32: the nibbles of lanes 2i and 2i + 1 become byte i at seq (one store per even lane), the quality
// character q goes to qual as phred.  in: the lane's base lies inside the read (else its nibble is 0 and nothing is stored).
// All 32 lanes must call it together.
__device__ __forceinline__ void bam_put_base(uint8_t* seq, uint8_t* qual, bool in, uint32_t ch, uint32_t q, int lane) {
	const uint32_t nib = in ? bam_nibble(ch) : 0u;
	const uint32_t lo = __shfl_down_sync(0xffffffffu, nib, 1);
	if (in && !(lane & 1)) *seq = (uint8_t)((nib << 4) | lo);
	if (in) *qual = (uint8_t)(q - 33u);
}

}  // namespace ssc
