// gz.h -- on-GPU gzip of the FASTQ blobs (see gz.cu).
#pragma once
#include <cuda_runtime.h>
#include <cstddef>
#include <cstdint>

namespace ssc {

static constexpr int GZ_PREFIX_WORDS = 96;   // gzip member header + dynamic block header, as a bit stream
// a stored member: 10-byte gzip header, one stored block (0x01, LEN, NLEN: 5 bytes), the raw bytes, CRC-32 and ISIZE.  A member
// whose coded form would be longer than the raw bytes plus this is written stored, so no member exceeds it.
static constexpr int GZ_STORED_EXTRA = 23;
// BGZF (the "bgzf" option, SAM specification 4.1): the member header grows by the 8-byte FEXTRA field with the BC subfield
// that holds the block size, so a stored block is the raw bytes plus 31.  A block may be at most 65 536 bytes.
static constexpr int GZ_BGZF_EXTRA_FIELD = 8;
static constexpr int GZ_BGZF_STORED_EXTRA = GZ_STORED_EXTRA + GZ_BGZF_EXTRA_FIELD;
static constexpr int GZ_BGZF_MAX_BLOCK = 65536;

// Built on the host from a byte histogram of the plan's own output, read by the encoder kernel.
struct GzTables {
	uint32_t lut[257];          // Huffman code (bit-reversed) | length << 16 per byte value; [256] = end of block
	uint32_t crcT[4][256];      // CRC-32 slice-by-4
	uint32_t crcS[4][256];      // remainder advanced by 128 zero bytes, by byte of the remainder
	uint32_t xp[256];           // x^(8n) mod P
	uint32_t prefix[GZ_PREFIX_WORDS];
	uint32_t prefixBits;
	uint32_t headerBytes;       // the gzip header at the start of the prefix: 10, or 18 for a BGZF block (BSIZE 0 in the prefix)
};

// "" on success.  bgzf: the member header of the prefix is a BGZF block header (FLG.FEXTRA, XLEN 6, 'B' 'C', SLEN 2, BSIZE 0);
// the DEFLATE bits behind it are the same, 64 bits later.
const char* gz_build_tables(const uint64_t hist[256], GzTables* out, bool bgzf = false);
uint32_t gz_crc32_host(const uint8_t* p, size_t n);
size_t gz_member_host(const GzTables* t, const uint8_t* src, uint32_t len, uint8_t* dst, size_t cap);

cudaError_t launch_deflate_blobs(const uint8_t* raw1, const uint8_t* raw2, const unsigned long long* rawLens, int nTiles, uint32_t rawPitch,
                                 uint8_t* gz1, uint8_t* gz2, unsigned long long* gzLens, uint32_t gzPitch, const GzTables* tab,
                                 int smCount, cudaStream_t stream);

}  // namespace ssc
