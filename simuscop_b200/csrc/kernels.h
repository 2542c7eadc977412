// kernels.h -- launch interface between the host runtime (api.cu) and kernels.cu.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

#include "device_types.h"

#define GEN_WARPS 16
#define GEN_THREADS (GEN_WARPS * 32)
#define GEN_PPW 2                                 /* pairs per warp per tile */
#define GEN_TILE_PAIRS (GEN_WARPS * GEN_PPW)
#define GEN_NCH 10                                /* chunks of 32 cycles the generic kernel holds in registers (RL <= 320) */

#ifndef FG_WORKERS
#define FG_WORKERS 32                             /* warps per CTA of the fast kernel */
#endif
#define FG_GEN FG_WORKERS
#define FG_THREADS (FG_WORKERS * 32)
#ifndef FG_CHUNK
#define FG_CHUNK 32                               /* consecutive pairs a warp of the fast kernel takes per ticket */
#endif
#define FG_SLOT 640                               /* bytes of HBM scratch per record (>= 96 + 2*256 + 4) */
#define SSC_GPAD 64                               /* zero bases in front of the haplotype store */
/* largest haplotype store: the fast kernel's 32-bit window word index (g - 32) >> 4 of device base g = SSC_GPAD + store
   index must not wrap for any base, i.e. SSC_GPAD + total_bases - 1 - 32 < 2^36 */
#define SSC_MAX_STORE_BASES ((1ull << 36) + 32 - SSC_GPAD)

namespace ssc {

struct GenVariant {
	bool k3;        // K == 3 fast context indexing with the substitution tables in shared memory
	bool fp64;      // FP64 linear-search ground truth
	size_t smemBytes;
	bool ok;
};

GenVariant choose_variant(const DevTables& t, bool fp64, int smemLimit);
// interleaved: PE, one slab; blobs: gzip output, one ticket blob per tile and file (P.out1/out2 blob scratch, P.blobPitch, P.tileState);
// bam: BAM records in such blobs (blobs must be set; PE: interleaved)
cudaError_t launch_generate(const GenParams& P, const GenVariant& v, int grid, cudaStream_t stream, bool interleaved, bool blobs, bool bam);
bool fast_supported(const DevTables& t, int smemLimit, int* qmode, size_t* smemBytes);   // qmode: 8 / 16 / 2 / 0, see gen_fast.cu
int fast_choose_qbins(int B, int RL);
int fast_nch(int RL);
cudaError_t launch_generate_fast(const GenParams& P, int qmode, size_t smemBytes, int grid, cudaStream_t stream, bool interleaved, bool bam);
cudaError_t launch_generate_reads(const GenParams& P, int qmode, size_t smemBytes, int grid, cudaStream_t stream);
cudaError_t launch_scan_blobs(const GenParams& P, cudaStream_t stream);
cudaError_t launch_move_blobs(const GenParams& P, int smCount, cudaStream_t stream);
cudaError_t launch_move_blobs_tma(const GenParams& P, int ctas, cudaStream_t stream);
cudaError_t launch_issue_floor(int mode, int RL, int64_t nPairs, uint64_t seed, int grid, uint32_t* scratch, uint8_t* blobs,
                               uint32_t blobPitch, uint32_t file2Off, cudaStream_t stream);   // floor.cu
cudaError_t launch_pass2(const GenParams& P, int smCount, cudaStream_t stream);
cudaError_t launch_pack(const uint8_t* ascii, uint64_t n, uint64_t firstBase, uint32_t* hap2, uint32_t* hapN,
                        const int8_t* lut, cudaStream_t stream);
cudaError_t launch_unfold(const uint8_t* raw, uint64_t rawLen, uint64_t nBases, uint32_t lineBases, uint32_t lineWidth, uint8_t* out,
                          unsigned long long* other, cudaStream_t stream);
cudaError_t launch_census(const DevTables& t, bool fp64, const CensusBin* bins, int nBins, uint64_t seed,
                          uint16_t* riskyAttempt, int32_t* emitted, cudaStream_t stream);
cudaError_t launch_poke(uint32_t* hap2, uint32_t* hapN, const int64_t* pos, const uint8_t* chars, int64_t n, const int8_t* lut, cudaStream_t stream);
cudaError_t launch_unpack(const uint32_t* hap2, const uint32_t* hapN, uint64_t firstBase, uint64_t n, uint32_t baseChars, uint8_t* out, cudaStream_t stream);
cudaError_t launch_gc_census(const uint32_t* hap2, const uint32_t* hapN, const int64_t* starts, const int32_t* lens, int64_t n,
                             uint32_t gcCodes, int32_t* gc, int32_t* nn, cudaStream_t stream);
cudaError_t launch_locate(const int64_t* emitBase, int64_t nBins, int64_t emitLo, int tilePairs, int nTiles, int32_t* tileStartBin,
                          cudaStream_t stream);

}  // namespace ssc
