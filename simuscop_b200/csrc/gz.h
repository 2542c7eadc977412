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

// Built on the host from a byte histogram of the plan's own output, read by the encoder kernel.
struct GzTables {
	uint32_t lut[257];          // Huffman code (bit-reversed) | length << 16 per byte value; [256] = end of block
	uint32_t crcT[4][256];      // CRC-32 slice-by-4
	uint32_t crcS[4][256];      // remainder advanced by 128 zero bytes, by byte of the remainder
	uint32_t xp[256];           // x^(8n) mod P
	uint32_t prefix[GZ_PREFIX_WORDS];
	uint32_t prefixBits;
};

const char* gz_build_tables(const uint64_t hist[256], GzTables* out);   // "" on success
uint32_t gz_crc32_host(const uint8_t* p, size_t n);
size_t gz_member_host(const GzTables* t, const uint8_t* src, uint32_t len, uint8_t* dst, size_t cap);

cudaError_t launch_deflate_blobs(const uint8_t* raw1, const uint8_t* raw2, const unsigned long long* rawLens, int nTiles, uint32_t rawPitch,
                                 uint8_t* gz1, uint8_t* gz2, unsigned long long* gzLens, uint32_t gzPitch, const GzTables* tab,
                                 int smCount, cudaStream_t stream);

}  // namespace ssc
