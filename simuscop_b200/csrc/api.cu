// api.cu -- C ABI of include/simuscop.h: device memory, plan upload, census, batched
// generation with pinned double-buffered device->host streaming.  No CPU fallback: every
// entry point needs a CUDA device and fails loudly otherwise.
#include <cuda_runtime.h>
#include <unistd.h>

#include <algorithm>
#include <cerrno>
#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <functional>
#include <string>
#include <thread>
#include <vector>

#include "../../include/simuscop.h"
#include "bam.cuh"
#include "device_types.h"
#include "kernels.h"
#include "tables.h"
#include "gz.h"

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
	char buf[1024];
	va_list ap;
	va_start(ap, fmt);
	vsnprintf(buf, sizeof(buf), fmt, ap);
	va_end(ap);
	g_err = buf;
	return code;
}

#define CK(call)                                                                                   \
	do {                                                                                           \
		cudaError_t e__ = (call);                                                                  \
		if (e__ != cudaSuccess)                                                                    \
			return fail(SSC_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
	} while (0)

// n elements of T in device memory, or in pinned host memory (Pinned); freed when the buffer is re-allocated or destroyed
template <class T, bool Pinned> struct Buffer {
	T* p = nullptr;
	size_t n = 0;
	Buffer() = default;
	Buffer(Buffer&& o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
	Buffer& operator=(Buffer&& o) noexcept { std::swap(p, o.p); std::swap(n, o.n); return *this; }
	~Buffer() { release(); }
	cudaError_t alloc(size_t count) {
		release();
		if (count == 0) return cudaSuccess;
		const cudaError_t e = Pinned ? cudaMallocHost((void**)&p, count * sizeof(T)) : cudaMalloc((void**)&p, count * sizeof(T));
		if (e == cudaSuccess) n = count;
		return e;
	}
	cudaError_t upload(const std::vector<T>& v, cudaStream_t s) {
		cudaError_t e = alloc(v.size());
		if (e != cudaSuccess || v.empty()) return e;
		return cudaMemcpyAsync(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, s);
	}
	void release() {
		if (p) { if (Pinned) cudaFreeHost(p); else cudaFree(p); }
		p = nullptr; n = 0;
	}
};
template <class T> using DevBuf = Buffer<T, false>;
template <class T> using HostBuf = Buffer<T, true>;

// A stream or event that is destroyed with its owner; it converts to the raw handle for the runtime calls
template <class H, cudaError_t (*Destroy)(H)> struct Owned {
	H h = nullptr;
	Owned() = default;
	Owned(Owned&& o) noexcept : h(o.h) { o.h = nullptr; }
	Owned& operator=(Owned&& o) noexcept { std::swap(h, o.h); return *this; }
	~Owned() { if (h) Destroy(h); }
	operator H() const { return h; }
};
using Stream = Owned<cudaStream_t, cudaStreamDestroy>;
using Event = Owned<cudaEvent_t, cudaEventDestroy>;

cudaError_t create(Stream& s) { return cudaStreamCreateWithFlags(&s.h, cudaStreamNonBlocking); }
cudaError_t create(Event& e, unsigned flags = cudaEventDisableTiming) { return cudaEventCreateWithFlags(&e.h, flags); }

// Everything a batch in flight owns.  The handle has two sets: batch k+1 is generated into one while the blobs of batch k are
// moved and its slabs copied out of the other.
struct BufferSet {
	DevBuf<uint8_t> d_out[2];                   // [file] dense slabs
	HostBuf<uint8_t> h_out[2];                  // their host copies (ssc_generate)
	DevBuf<uint8_t> d_slots;                    // ticket blob scratch: the fast kernel's pass 1, the generic kernel's gzip mode
	size_t file2Off = 0;                        // file 2's blobs start this many bytes into d_slots (0: one file)
	DevBuf<unsigned long long> d_blobPrefix;
	DevBuf<int32_t> d_tileStart;
	DevBuf<unsigned long long> d_tileState;
	DevBuf<unsigned int> d_ticket;
	DevBuf<ssc::BatchResult> d_result;
	HostBuf<ssc::BatchResult> h_result;
	Event evDense;                              // the dense slabs are complete in the compute stream
	Event evScanned;                            // the batch's last kernel (fast kernel, plain output: the scan) done
	Event evResult;                             // the BatchResult is in h_result
	Event evMoved;                              // the mover has moved the blobs
	Event evCopy, evCopy2;                      // the device->host copies of file 1 / file 2 are done
};

}  // namespace

struct ssc_handle {
	int device = 0;
	int smCount = 0;
	int smemLimit = 0;
	Stream compute, copy, copy2;                  // copy/copy2: device->host of file 1 / file 2 (two copy engines)
	Event evStart, evStop;

	// options
	int64_t batchPairs = 1 << 20;
	bool fp64 = false;
	bool forceGeneric = false;
	bool noSplice = false;        // tests: see GenParams::noSplice
	int maxCtas = 0;              // > 0: cap the grid of the generation kernel (tests: many tickets per warp on small inputs)
	int moverCtas = 0;            // "concurrent_move": pass 2b of batch k runs on that many SMs (bulk-copy mover, second stream) under the
	                              // generation kernel of batch k+1, which leaves them free; 0 or [1, smCount), 0 = a stand-alone move
	                              // after every batch.  Default: init_handle
	Stream mover;                 // pass 2 of the fast kernel's plain output: the scans and the concurrent moves
	Event evPre;                  // a point of the compute stream the mover stream waits for (recorded anew for every wait)
	// the device->host copy of a batch's BatchResult: on a stream of its own, because the copy engines may be busy with the
	// FASTQ slabs of ssc_generate for milliseconds, and no kernel must queue behind it
	Stream results;
	int fastQmode = -1;           // "fast_qmode": -1 automatic, else the only quality-table mode the fast kernel may use (tests)
	bool gzip = false;            // slabs hold gzip members (one per ticket blob) instead of plain FASTQ
	bool bgzf = false;            // "bgzf": with gzip, every member is a BGZF block (no effect without gzip)
	bool interleave = false;      // "interleave": a PE plan's mates go to one stream, mate 1 and mate 2 of each pair in turn
	bool bam = false;             // "bam": BGZF blocks of unaligned BAM records (PE: both mates in one stream), whatever gzip / bgzf / interleave say
	int rgLen = 0;                // ssc_set_read_group: bytes of the id in d_rg (0: no RG tag)
	DevBuf<char> d_rg;
	size_t gzBlobBytes = 0;       // allocation of d_gzBlobs[0] (interleaved: both mates per ticket)
	bool haveGz = false;          // Huffman / CRC tables of the current plan are on the device
	bool gzBam = false;           // ... fitted to BAM records (refitted when the output format changes)
	DevBuf<ssc::GzTables> d_gzTab;      // [0] gzip members, [1] BGZF blocks: one Huffman table, two member headers
	DevBuf<uint8_t> d_gzBlobs[2];
	DevBuf<unsigned long long> d_gzLens;

	// profile
	bool haveProfile = false;
	ssc::DeviceTablesHost th;
	ssc::DevTables dt;
	DevBuf<uint32_t> d_isizeT, d_insT, d_delT, d_qualT, d_qualDiagT;
	DevBuf<uint8_t> d_qualDiagSym;
	DevBuf<uint16_t> d_isizeSym, d_insSym, d_delSym;
	DevBuf<uint8_t> d_qualSym;
	DevBuf<uint4> d_sub;
	DevBuf<double> d_fIsize, d_fIns, d_fDel, d_fSub1, d_fSub2, d_fQual;
	DevBuf<int8_t> d_lut;

	// genome
	DevBuf<uint32_t> d_hap2, d_hapN;
	uint64_t genomeCap = 0, genomeSize = 0;
	DevBuf<uint8_t> d_ref;                        // ASCII chromosome for ssc_genome_append_ref
	DevBuf<uint8_t> d_raw;                        // raw FASTA lines of the chromosome (ssc_reference_upload_fasta), grow-only
	DevBuf<unsigned long long> d_other;
	// ssc_reference_prefetch_fasta: the next record is read and unfolded into a second set of buffers by a background thread
	// on its own stream while the caller works with the current reference; ssc_reference_adopt_prefetched swaps the sets
	DevBuf<uint8_t> d_ref2, d_raw2;
	DevBuf<unsigned long long> d_other2;
	Stream upload;
	Event evRefFree;
	std::thread prefetchThread;
	bool prefetching = false;
	int prefetchRc = 0;
	std::string prefetchErr;
	uint64_t prefetchBases = 0, prefetchRaw = 0, prefetchOther = 0;
	uint64_t refSize = 0;
	HostBuf<uint8_t> h_stage[2];                  // pinned upload staging
	DevBuf<uint8_t> d_stage[2];
	Event evStage[2];
	static constexpr int FA_READERS = 2;          // ssc_reference_upload_fasta: reader threads, one pinned buffer each (four readers
	                                              // of 16 MB chunks were slower on the 16-vCPU boxes: 0.69 vs 0.28-0.31 s for the 3 Gb FASTA)
	HostBuf<uint8_t> h_fa[2 * FA_READERS];        // [0, FA_READERS): foreground, the rest: prefetch
	Event evFa[2 * FA_READERS];
	size_t faBytes = 32u << 20;
	size_t stageBytes = 32u << 20;

	// plan
	bool havePlan = false;
	uint64_t seed = 0;
	std::vector<int64_t> planBaseAll, emitBaseAll;   // per original bin (+1 sentinel)
	std::vector<int64_t> devEmitBase;                // per device bin (+1 sentinel): host copy of d_emitBase
	DevBuf<ssc::DevBin> d_bins;
	DevBuf<int64_t> d_emitBase;
	DevBuf<uint16_t> d_risky;
	DevBuf<char> d_names;
	std::vector<char> names;                         // host copy of the name blob and of the segments' name ranges (ssc_segment_name)
	std::vector<int32_t> segNameOff, segNameLen;
	int64_t nDevBins = 0, plannedPairs = 0, emittedPairs = 0;
	int maxRecBytes = 0;                             // worst-case FASTQ record of the plan
	int maxName = 0;                                 // longest segment name of the plan, '@' included
	int64_t badQnameSeg = -1;                        // first segment whose name is not a valid BAM read name (-1: none)
	int badQnameByte = 0;

	// batch resources
	int64_t slabPairs = 0;
	uint64_t slabCap = 0;
	int slabFiles = 0;                             // output streams the slabs were allocated for (out_files)
	uint32_t blobBytes = 0;                        // blob scratch per ticket and file the sets were allocated for (ticket_bytes)
	BufferSet set[2];
	struct { bool valid = false; int buf = 0; ssc::GenParams P; } pending;   // generated (scan queued), blobs not yet moved
	DevBuf<int64_t> d_cenStarts;                  // ssc_gc_census scratch (grow-only)
	DevBuf<int32_t> d_cenLens, d_cenGc, d_cenNn;
	// ssc_generate_reads: the bookkeeping of its batches only (no slab, blob scratch or pinned host memory: the caller owns the output);
	// the batches run back to back on the compute stream and add to one BatchResult
	DevBuf<int32_t> d_rdTileStart;
	DevBuf<unsigned int> d_rdTicket;
	DevBuf<ssc::BatchResult> d_rdResult;
	Event evCaller;                                  // the caller's stream at the call: the compute stream waits for it

	// kernel timing of ssc_generate_device: events kev[2 i] and kev[2 i + 1] bracket the i-th timed piece of work of the call,
	// whose time goes to *kevSum[i] when the call ends (see time_begin)
	std::vector<Event> kev;
	std::vector<double*> kevSum;
	int kevUsed = 0;
	bool timeKernels = false;

	ssc_stats stats;
};

namespace {

bool use_fast(const ssc_handle* h, int* qmode, size_t* smemBytes) {
	if (h->fp64 || h->forceGeneric) return false;
	return ssc::fast_supported(h->dt, h->smemLimit, qmode, smemBytes);
}

// PE plan with the "interleave" or the "bam" option: one output stream holding both mates (no effect on SE plans)
bool interleaved(const ssc_handle* h) { return (h->interleave || h->bam) && h->dt.paired; }

// output streams of ssc_generate / ssc_generate_device: 2 for two-file PE, 1 for SE and interleaved PE
int out_files(const ssc_handle* h) { return h->dt.paired && !interleaved(h) ? 2 : 1; }

// the slabs hold compressed members (gzip, or BAM, which always goes through the gzip arm) / BGZF blocks
bool gz_mode(const ssc_handle* h) { return h->gzip || h->bam; }
bool bgzf_mode(const ssc_handle* h) { return h->bam || (h->gzip && h->bgzf); }

// Worst-case record bytes of the plan in the running format.  FASTQ: header + 2 x (RL + 96) + 4.  BAM: 36 fixed bytes, the name
// without '@' and its two fields and NUL (name + 21), the 4-bit codes and qualities of RL + 96 bases, RG:Z:<id> NUL.
int rec_bytes(const ssc_handle* h) {
	if (!h->bam) return h->maxRecBytes;
	const uint32_t m = (uint32_t)h->dt.RL + 96u;
	return ssc::BAM_FIXED + (int)ssc::bam_tail_bytes((uint32_t)h->maxName + 21u, m, (uint32_t)h->rgLen);
}

// Bytes of blob scratch per ticket and file: the pitch of one file's ticket blobs and of their gzip members (interleaved: one
// blob of both mates at twice this).  The fast kernel's tickets take FG_SLOT bytes per record.  The generic kernel writes
// ticket blobs only in gzip mode; its records are longer (up to 924 bytes at RL 320 with 64-byte names), so the pitch is its
// tile of the plan's worst-case records plus a stored BGZF block, rounded to 16 bytes.
uint32_t ticket_bytes(const ssc_handle* h) {
	int qm = 0; size_t sb = 0;
	if (!gz_mode(h) || use_fast(h, &qm, &sb)) return FG_CHUNK * FG_SLOT;
	return (uint32_t)(((uint64_t)GEN_TILE_PAIRS * (uint64_t)rec_bytes(h) + ssc::GZ_BGZF_STORED_EXTRA + 15) / 16 * 16);
}

int ensure_batch_resources(ssc_handle* h, bool needHost) {
	int64_t pairs = std::min<int64_t>(h->batchPairs, std::max<int64_t>(h->emittedPairs, 1));
	pairs = ((pairs + GEN_TILE_PAIRS - 1) / GEN_TILE_PAIRS) * GEN_TILE_PAIRS;   // multiple of both tile sizes
	// gzip mode: a member is at most its blob plus the bytes of a stored block (gz.cu: 23, a BGZF block 31), and there is one
	// member per ticket.  Interleaved output: a slab holds both mates of a pair.  The scan packs a slab length into 31 bits, so
	// the slab bound stays below 2^31 in every mode: the clamp budgets the stored-block bytes as ceil(extra / 32) = 1 per pair.
	const uint64_t recBytes = (uint64_t)rec_bytes(h) * (interleaved(h) ? 2u : 1u);
	const uint64_t gzExtra = gz_mode(h) ? (uint64_t)(bgzf_mode(h) ? ssc::GZ_BGZF_STORED_EXTRA : ssc::GZ_STORED_EXTRA) : 0;
	const uint64_t perPair = recBytes + (gzExtra + FG_CHUNK - 1) / FG_CHUNK;
	auto slab_cap = [&](int64_t n) { return (uint64_t)n * recBytes + 4096 + (uint64_t)(n / FG_CHUNK) * gzExtra; };
	uint64_t cap = slab_cap(pairs);
	if (cap >= (1ull << 31)) {
		pairs = (int64_t)(((1ull << 31) - 8192) / perPair);
		pairs = (pairs / GEN_TILE_PAIRS) * GEN_TILE_PAIRS;
		if (pairs <= 0) return fail(SSC_ERR_INVALID, "record size too large");
		cap = slab_cap(pairs);
	}
	int nFiles = h->dt.paired ? 2 : 1;             // halves of the blob scratch (interleaved: one blob of both mates across both)
	const int slabFiles = out_files(h);
	// where tickets go through blobs (the fast kernel, gzip mode), a ticket's blob of worst-case records (interleaved: both mates),
	// and in gzip mode its stored member, fit the blob pitch, which is a multiple of 16; a stored member fits one BGZF block.  The
	// fast kernel's fixed slots hold any plan it takes (RL <= 160).
	const uint32_t blobBytes = ticket_bytes(h);
	int qm = 0; size_t sb = 0;
	if (gz_mode(h) || use_fast(h, &qm, &sb)) {
		const uint64_t mates = interleaved(h) ? 2 : 1, pitch = blobBytes * mates;
		const uint64_t maxBlob = (uint64_t)GEN_TILE_PAIRS * (uint64_t)rec_bytes(h) * mates;
		if (pitch % 16 || maxBlob + gzExtra > pitch || (gz_mode(h) && maxBlob + gzExtra > (uint64_t)ssc::GZ_BGZF_MAX_BLOCK))
			return fail(SSC_ERR_INVALID, "a ticket of %d records of up to %d bytes does not fit its blob pitch of %llu bytes", GEN_TILE_PAIRS,
			            rec_bytes(h) * (int)mates, (unsigned long long)pitch);
	}
	{
		// the fast kernel addresses its blob scratch (FG_SLOT bytes per record, both mates) with 32-bit offsets
		const int64_t maxFast = (int64_t)(((1ull << 32) - (1ull << 20)) / ((uint64_t)FG_SLOT * (uint64_t)nFiles));
		if (pairs > maxFast) {
			pairs = (maxFast / GEN_TILE_PAIRS) * GEN_TILE_PAIRS;
			cap = slab_cap(pairs);
		}
	}
	if (pairs != h->slabPairs || cap != h->slabCap || slabFiles != h->slabFiles || blobBytes != h->blobBytes) {
		h->slabPairs = 0; h->slabCap = 0; h->slabFiles = 0; h->blobBytes = 0;   // committed below, once every allocation has succeeded
		h->pending.valid = false;
		h->d_gzBlobs[0].release(); h->d_gzBlobs[1].release();   // sized by the slabs: allocated below when gzip is on
		h->gzBlobBytes = 0;
		int nTiles = (int)(pairs / 16) + 2;   // enough for every kernel's tile size
		for (BufferSet& S : h->set) {
			// file 2's blobs behind file 1's: the kernel addresses both from one base pointer with 32-bit cursors
			const size_t fileBytes = (size_t)(pairs / GEN_TILE_PAIRS) * blobBytes + 256;
			CK(S.d_slots.alloc(fileBytes * nFiles));
			S.file2Off = nFiles == 2 ? fileBytes : 0;
			CK(S.d_blobPrefix.alloc(nTiles));
			for (int f = 0; f < 2; f++) {
				S.h_out[f].release();                   // allocated below when the call copies to the host
				CK(S.d_out[f].alloc(f < slabFiles ? cap : 0));
			}
			CK(S.d_tileStart.alloc(nTiles));
			CK(S.d_tileState.alloc(nTiles));
			CK(S.d_ticket.alloc(1));
		}
		h->slabPairs = pairs; h->slabCap = cap; h->slabFiles = slabFiles; h->blobBytes = blobBytes;
	}
	// gzip members: one per ticket blob, at the blob's pitch (interleaved: twice the per-file pitch, one file)
	const size_t gzBytes = (size_t)(h->slabPairs / GEN_TILE_PAIRS) * h->blobBytes * (interleaved(h) ? 2 : 1) + 64;
	if (gz_mode(h) && h->gzBlobBytes != gzBytes) {
		h->gzBlobBytes = 0;
		for (int f = 0; f < 2; f++) CK(h->d_gzBlobs[f].alloc(f < (interleaved(h) ? 1 : 2) ? gzBytes : 0));
		h->gzBlobBytes = gzBytes;
		CK(h->d_gzLens.alloc((size_t)(h->slabPairs / 16) + 2));
		if (!h->d_gzTab.p) CK(h->d_gzTab.alloc(2));
	}
	if (needHost)
		for (BufferSet& S : h->set)
			for (int f = 0; f < slabFiles; f++)
				if (!S.h_out[f].p) CK(S.h_out[f].alloc(h->slabCap));
	return SSC_OK;
}

// emitted-pair index of the first emitted pair whose planned ID is >= p
int64_t emit_index_of_plan(const ssc_handle* h, int64_t p) {
	if (p <= 0) return 0;
	if (p >= h->plannedPairs) return h->emittedPairs;
	const std::vector<int64_t>& pb = h->planBaseAll;
	size_t b = std::upper_bound(pb.begin(), pb.end(), p) - pb.begin() - 1;   // pb[b] <= p < pb[b+1]
	int64_t emitCount = h->emitBaseAll[b + 1] - h->emitBaseAll[b];
	return h->emitBaseAll[b] + std::min<int64_t>(p - pb[b], emitCount);
}

// Fits the gzip Huffman table of a plan to the first tickets of its first batch (the blobs are in scratch already).
int build_gz_tables(ssc_handle* h, const ssc::GenParams& P, int nTiles) {
	const int sample = std::min(nTiles, 256);
	const size_t pitch = P.blobPitch;
	std::vector<unsigned long long> lens((size_t)sample);
	std::vector<uint8_t> blob((size_t)sample * pitch);
	uint64_t hist[256];
	memset(hist, 0, sizeof(hist));
	CK(cudaStreamSynchronize(h->compute));
	CK(cudaMemcpy(lens.data(), P.tileState, lens.size() * 8, cudaMemcpyDeviceToHost));
	for (int f = 0; f < out_files(h); f++) {
		CK(cudaMemcpy(blob.data(), f ? P.out2 : P.out1, blob.size(), cudaMemcpyDeviceToHost));
		for (int j = 0; j < sample; j++) {
			const size_t n = f ? (size_t)(lens[j] & 0x7fffffffull) : (size_t)(lens[j] >> 31);
			const uint8_t* p = blob.data() + (size_t)j * pitch;
			for (size_t i = 0; i < n; i++) hist[p[i]]++;
		}
	}
	// the gzip and the BGZF tables from the one fit, so that "bgzf" may change between calls and each block is its gzip member
	// with the BC field inserted
	std::vector<ssc::GzTables> tab(2);
	for (int b = 0; b < 2; b++) {
		const char* err = ssc::gz_build_tables(hist, &tab[b], b == 1);
		if (err[0]) return fail(SSC_ERR_INVALID, "gzip tables: %s", err);
	}
	CK(cudaMemcpyAsync(h->d_gzTab.p, tab.data(), 2 * sizeof(ssc::GzTables), cudaMemcpyHostToDevice, h->compute));   // stream order with the deflate kernel
	CK(cudaStreamSynchronize(h->compute));          // tab is freed on return
	h->haveGz = true;
	h->gzBam = h->bam;
	return SSC_OK;
}

// Kernel timing of ssc_generate_device: when the call is timed, records the start event of a piece of work on stream s and
// returns in *end the event the caller records on s after it; the time between the two goes to *sum when the call ends.
// *end is null when the call is not timed.
cudaError_t time_begin(ssc_handle* h, cudaStream_t s, double* sum, cudaEvent_t* end) {
	*end = nullptr;
	if (!h->timeKernels) return cudaSuccess;
	while (h->kev.size() < 2 * (size_t)(h->kevUsed + 1)) {
		Event e;
		const cudaError_t err = create(e, cudaEventDefault);
		if (err != cudaSuccess) return err;
		h->kev.push_back(std::move(e));
	}
	h->kevSum.resize((size_t)h->kevUsed + 1);
	h->kevSum[h->kevUsed] = sum;
	*end = h->kev[2 * h->kevUsed + 1];
	return cudaEventRecord(h->kev[2 * h->kevUsed++], s);
}

// Moves the blobs of the last launched batch to its dense slab with the stand-alone kernel (every batch without the mover;
// with it, the last batch of a call: no later launch runs the mover for it).  Timed as pass 2.
int flush_pending(ssc_handle* h) {
	if (!h->pending.valid) return SSC_OK;
	h->pending.valid = false;
	CK(cudaStreamWaitEvent(h->compute, h->set[h->pending.buf].evScanned, 0));    // the blob offsets, scanned on the mover stream
	cudaEvent_t te;
	CK(time_begin(h, h->compute, &h->stats.compact_kernel_ms, &te));
	CK(ssc::launch_move_blobs(h->pending.P, h->smCount, h->compute));
	if (te) CK(cudaEventRecord(te, h->compute));
	h->stats.launches += 1;
	return SSC_OK;
}

// Copies the BatchResult of buffer set `buf` to its h_result (evResult) once the work queued on stream `after`, which writes it
// last, is done (evScanned).
int result_to_host(ssc_handle* h, int buf, cudaStream_t after) {
	CK(cudaEventRecord(h->set[buf].evScanned, after));
	CK(cudaStreamWaitEvent(h->results, h->set[buf].evScanned, 0));
	CK(cudaMemcpyAsync(h->set[buf].h_result.p, h->set[buf].d_result.p, sizeof(ssc::BatchResult), cudaMemcpyDeviceToHost, h->results));
	CK(cudaEventRecord(h->set[buf].evResult, h->results));
	return SSC_OK;
}

// The launch parameters of batch [emitLo, emitHi) every generation kernel reads (tables, plan, Philox keys), and the batch's
// statistics (one generation launch, its distinct bin records).  qsmem8: the fast kernel with every quality row in shared memory.
ssc::GenParams batch_params(ssc_handle* h, int64_t emitLo, int64_t emitHi, bool qsmem8) {
	h->stats.gen_launches += 1;
	{
		// distinct bins of the batch (statistics: the algorithmic bin-record bytes of the roofline)
		const std::vector<int64_t>& eb = h->devEmitBase;
		const size_t bLo = std::upper_bound(eb.begin(), eb.end(), emitLo) - eb.begin() - 1;
		const size_t bHi = std::lower_bound(eb.begin(), eb.end(), emitHi) - eb.begin();
		h->stats.bin_bytes += (uint64_t)(bHi > bLo ? bHi - bLo : 0) * sizeof(ssc::DevBin);
	}
	ssc::GenParams P;
	memset(&P, 0, sizeof(P));
	P.t = h->dt;
	P.hap2 = h->d_hap2.p; P.hapN = h->d_hapN.p;
	P.bins = h->d_bins.p; P.emitBase = h->d_emitBase.p; P.nBins = h->nDevBins;
	P.riskyAttempt = h->d_risky.p; P.names = h->d_names.p;
	P.seed = h->seed; P.emitLo = emitLo; P.emitHi = emitHi; P.one = 1; P.noSplice = h->noSplice ? 1 : 0;
	P.qstride = qsmem8 ? (uint32_t)h->dt.qualBins * 68u : 68u;   // F_QROW of gen_fast.cu (unused by the 16-bit-key mode)
	P.insLim = h->dt.insEnable ? h->dt.insT + 1u : 0u;
	P.delLim = h->dt.delEnable ? h->dt.delT + 1u : 0u;
	P.alwaysSlow = (h->dt.insEnable && h->dt.insT == 0xFFFFFFFFu) || (h->dt.delEnable && h->dt.delT == 0xFFFFFFFFu);
	P.rg = h->d_rg.p; P.rgLen = h->rgLen;
	for (int r = 0; r < 10; r++) {
		P.rk[2 * r] = (uint32_t)h->seed + (uint32_t)r * 0x9E3779B9u;
		P.rk[2 * r + 1] = (uint32_t)(h->seed >> 32) + (uint32_t)r * 0xBB67AE85u;
	}
	return P;
}

// Launches batch [emitLo, emitHi) into buffer set `buf`; its evResult marks the BatchResult in its h_result.  Fast kernel,
// plain output: pass 1 on the compute stream, then the scan of the blob lengths on the mover stream; the blobs are moved to
// the set's dense slabs d_out by the mover under the next launch_batch, or by flush_pending (right after the scan when the
// mover is off).  Every other mode leaves the finished slabs in d_out when its kernels have run on the compute stream.
int launch_batch(ssc_handle* h, int buf, int64_t emitLo, int64_t emitHi) {
	int qsmem = 0; size_t fastSmem = 0;
	const bool fast = use_fast(h, &qsmem, &fastSmem);
	const int tp = fast ? FG_CHUNK : GEN_TILE_PAIRS;
	int nTiles = (int)((emitHi - emitLo + tp - 1) / tp);
	cudaStream_t s = h->compute;
	BufferSet& S = h->set[buf];
	CK(cudaStreamWaitEvent(s, S.evResult, 0));                // the copy of the BatchResult this buffer set held before
	CK(cudaMemsetAsync(S.d_tileState.p, 0, sizeof(unsigned long long) * nTiles, s));
	CK(cudaMemsetAsync(S.d_ticket.p, 0, sizeof(unsigned int), s));
	CK(cudaMemsetAsync(S.d_result.p, 0, sizeof(ssc::BatchResult), s));
	CK(ssc::launch_locate(h->d_emitBase.p, h->nDevBins, emitLo, tp, nTiles, S.d_tileStart.p, s));
	h->stats.launches += 1;
	ssc::GenParams P = batch_params(h, emitLo, emitHi, fast && qsmem == 8);
	P.tileStartBin = S.d_tileStart.p; P.nTiles = nTiles;
	P.tileState = S.d_tileState.p; P.ticket = S.d_ticket.p; P.blobPrefix = S.d_blobPrefix.p;
	P.out1 = S.d_out[0].p; P.out2 = S.d_out[1].p;
	P.cap1 = h->slabCap; P.cap2 = h->slabCap;
	P.result = S.d_result.p;
	int grid = std::min(nTiles, h->smCount);
	const bool ilv = interleaved(h);
	cudaEvent_t te;
	const bool gz = gz_mode(h);
	if (fast || gz) {
		// the generation kernel writes one blob per ticket and file into the scratch, pass 2 (scan of the blob lengths + one move per
		// blob, in gzip mode per member) the dense slab.  Interleaved: one blob per ticket over both halves of the scratch, so twice
		// the per-file pitch
		P.dense1 = P.out1; P.dense2 = P.out2;
		P.out1 = S.d_slots.p; P.out2 = S.file2Off ? S.d_slots.p + S.file2Off : nullptr;
		P.blobPitch = h->blobBytes * (ilv ? 2u : 1u);
		P.file2Off = (uint32_t)S.file2Off;
	}
	if (fast) {
		h->stats.gen_kernel = 1; h->stats.gen_nch = ssc::fast_nch(h->dt.RL); h->stats.gen_qmode = qsmem;
		h->stats.gen_smem_bytes = (int32_t)fastSmem;
		if (!gz) {
			int movedBuf = -1;
			if (h->pending.valid) {
				// pass 2b of the previous batch on the mover stream, under this batch's generation kernel (which leaves it the SMs);
				// only the mover leaves a batch pending between launches.  Its scan is ahead of it on that stream.
				const ssc::GenParams& Q = h->pending.P;
				movedBuf = buf ^ 1;
				CK(cudaEventRecord(h->evPre, s));                          // everything this launch had to wait for (copies, ...)
				CK(cudaStreamWaitEvent(h->mover, h->evPre, 0));
				CK(time_begin(h, h->mover, &h->stats.mover_kernel_ms, &te));
				CK(ssc::launch_move_blobs_tma(Q, h->moverCtas, h->mover));
				if (te) CK(cudaEventRecord(te, h->mover));
				CK(cudaEventRecord(h->set[movedBuf].evMoved, h->mover));
				h->pending.valid = false;
				h->stats.launches += 1;
			}
			grid = std::min((nTiles + FG_GEN - 1) / FG_GEN, h->smCount - (movedBuf >= 0 ? h->moverCtas : 0));
			if (h->maxCtas > 0) grid = std::min(grid, h->maxCtas);
			CK(time_begin(h, s, &h->stats.gen_kernel_ms, &te));
			CK(ssc::launch_generate_fast(P, qsmem, fastSmem, grid, s, ilv, false));
			if (te) CK(cudaEventRecord(te, s));
			// pass 2a on the mover stream, behind the previous batch's move: only the moves and the host need its offsets and
			// totals, so the compute stream goes straight on to the next batch
			CK(cudaEventRecord(h->evPre, s));
			CK(cudaStreamWaitEvent(h->mover, h->evPre, 0));
			CK(time_begin(h, h->mover, &h->stats.compact_kernel_ms, &te));
			CK(ssc::launch_scan_blobs(P, h->mover));
			if (te) CK(cudaEventRecord(te, h->mover));
			const int rc = result_to_host(h, buf, h->mover);
			if (rc) return rc;
			h->pending.P = P; h->pending.buf = buf; h->pending.valid = true;
			h->stats.launches += 2;
			if (h->moverCtas == 0) return flush_pending(h);              // stand-alone move right after the scan
			// later work on this stream (the next launch reuses the blob scratch, copies read the dense slab) comes after the mover
			if (movedBuf >= 0) CK(cudaStreamWaitEvent(s, h->set[movedBuf].evMoved, 0));
			return SSC_OK;
		}
		int rc = flush_pending(h);
		if (rc) return rc;
		grid = std::min((nTiles + FG_GEN - 1) / FG_GEN, h->smCount);
		if (h->maxCtas > 0) grid = std::min(grid, h->maxCtas);
		CK(time_begin(h, s, &h->stats.gen_kernel_ms, &te));
		CK(ssc::launch_generate_fast(P, qsmem, fastSmem, grid, s, ilv, h->bam));
		if (te) CK(cudaEventRecord(te, s));
		h->stats.launches += 1;
	} else {
		int rc = flush_pending(h);
		if (rc) return rc;
		ssc::GenVariant v = ssc::choose_variant(h->dt, h->fp64, h->smemLimit);
		if (!v.ok) return fail(SSC_ERR_INVALID, "no kernel variant for read length %d / kmer %d", h->dt.RL, h->dt.K);
		h->stats.gen_kernel = v.fp64 ? 4 : v.k3 ? 2 : 3; h->stats.gen_nch = GEN_NCH; h->stats.gen_qmode = -1;
		h->stats.gen_smem_bytes = (int32_t)v.smemBytes;
		CK(ssc::launch_generate(P, v, grid, s, ilv, gz, h->bam));
		h->stats.launches += 1;
	}
	if (gz) {
		// blobs -> (first batch of a plan or of a changed format, FASTQ or BAM: fit the Huffman table to a sample) -> one gzip member
		// per blob -> pass 2 on the members
		CK(time_begin(h, s, &h->stats.compact_kernel_ms, &te));
		if (!h->haveGz || h->gzBam != h->bam) { const int rc = build_gz_tables(h, P, nTiles); if (rc) return rc; }
		CK(cudaMemsetAsync(h->d_gzLens.p, 0, sizeof(unsigned long long) * nTiles, s));
		CK(ssc::launch_deflate_blobs(P.out1, P.out2, P.tileState, nTiles, P.blobPitch, h->d_gzBlobs[0].p, h->d_gzBlobs[1].p, h->d_gzLens.p,
		                             P.blobPitch, h->d_gzTab.p + (bgzf_mode(h) ? 1 : 0), h->smCount, s));
		ssc::GenParams P2 = P;
		P2.out1 = h->d_gzBlobs[0].p; P2.out2 = h->d_gzBlobs[1].p; P2.tileState = h->d_gzLens.p;
		CK(ssc::launch_pass2(P2, h->smCount, s));
		if (te) CK(cudaEventRecord(te, s));
		h->stats.launches += 3;
	}
	return result_to_host(h, buf, s);
}

// error exit of a pipelined call: nothing of it may still be running when the caller sees the code, no batch stays pending
// for the next call, and the kernel timing of ssc_generate_device ends with the call
int bail(ssc_handle* h, int rc) {
	const std::string msg = g_err;
	cudaDeviceSynchronize();
	h->pending.valid = false;
	h->timeKernels = false;
	h->kevUsed = 0;
	g_err = msg;
	return rc;
}

int check_result(ssc_handle* h, const ssc::BatchResult& r) {
	if (r.errorFlags & 1u) return fail(SSC_ERR_OVERFLOW, "output slab overflow (internal capacity estimate too small)");
	if (r.errorFlags & 2u) return fail(SSC_ERR_OVERFLOW, "a read outgrew the per-read scratch (insertions > 96 bases)");
	if (r.errorFlags & 4u) return fail(SSC_ERR_OVERFLOW, "more than 32 indel events or 128 inserted bases in one read");
	h->stats.pairs_emitted += r.pairs;
	h->stats.reads_emitted += r.reads;
	h->stats.bases_emitted += r.bases;
	h->stats.fastq_bytes += gz_mode(h) ? r.rawBytes : r.bytes1 + r.bytes2;
	if (gz_mode(h)) h->stats.gz_bytes += r.bytes1 + r.bytes2;
	h->stats.hap_bytes += r.hapBytes;
	return SSC_OK;
}

}  // namespace

extern "C" {

const char* ssc_last_error(void) { return g_err.c_str(); }
int ssc_version(void) { return 1; }

static int init_handle(ssc_handle* h, int device) {
	h->device = device;
	memset(&h->stats, 0, sizeof(h->stats));
	cudaDeviceProp prop;
	CK(cudaGetDeviceProperties(&prop, device));
	h->smCount = prop.multiProcessorCount;
	// 9 of 148 SMs, 0 below 64 SMs.  On the 3 Gb XTen job (B200, tools/pipeline_probe.py) 9 are the fewest under which the scan
	// and the move of a batch finish before the generation launch on the others does: 8 SMs need 3.88 ms for the move, 9
	// need 3.46 (+ 0.06 for the scan) under a 3.69 ms launch.  GAIIx and HiSeq2500 move fewer bytes per pair and run 1.4 and
	// 0.5 % faster on 7 and 8 SMs, but what a profile needs depends on its generation time as much as on its bytes, and one SM
	// too few costs 4-6 % (the mover sets the step) where one too many costs 0.5-0.7 %: every profile gets the count XTen needs.
	h->moverCtas = h->smCount >= 64 ? (h->smCount * 9 + 74) / 148 : 0;   // < smCount
	h->smemLimit = (int)prop.sharedMemPerBlockOptin - 1024;
	CK(create(h->compute)); CK(create(h->copy)); CK(create(h->copy2)); CK(create(h->mover)); CK(create(h->results));
	CK(create(h->evPre)); CK(create(h->evCaller));
	CK(create(h->evStart, cudaEventDefault)); CK(create(h->evStop, cudaEventDefault));
	for (Event& e : h->evStage) CK(create(e));
	for (BufferSet& S : h->set) {
		for (Event* e : {&S.evDense, &S.evScanned, &S.evResult, &S.evMoved, &S.evCopy, &S.evCopy2}) CK(create(*e));
		CK(S.d_result.alloc(1));
		CK(S.h_result.alloc(1));
	}
	return SSC_OK;
}

int ssc_create(int device, ssc_handle** out) {
	if (!out) return fail(SSC_ERR_INVALID, "out is null");
	*out = nullptr;
	int count = 0;
	cudaError_t e = cudaGetDeviceCount(&count);
	if (e != cudaSuccess || count == 0)
		return fail(SSC_ERR_CUDA, "no CUDA device available (%s); this library has no CPU fallback",
		            e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
	if (device < 0 || device >= count) return fail(SSC_ERR_INVALID, "device %d out of range (%d devices)", device, count);
	CK(cudaSetDevice(device));
	ssc_handle* h = new ssc_handle();
	const int rc = init_handle(h, device);
	if (rc) { const std::string msg = g_err; ssc_destroy(h); g_err = msg; return rc; }   // nothing of a half-built handle leaks
	*out = h;
	return SSC_OK;
}

int ssc_destroy(ssc_handle* h) {
	if (!h) return SSC_OK;
	if (h->prefetchThread.joinable()) h->prefetchThread.join();
	// the members free their memory, streams and events as they are destroyed: with the handle's device current, and only
	// once nothing queued on it can still use them
	cudaSetDevice(h->device);
	cudaDeviceSynchronize();
	delete h;
	return SSC_OK;
}

int ssc_set_option(ssc_handle* h, const char* key, int64_t value) {
	if (!h || !key) return fail(SSC_ERR_INVALID, "null argument");
	if (!strcmp(key, "batch_pairs")) {
		if (value < GEN_TILE_PAIRS) return fail(SSC_ERR_INVALID, "batch_pairs must be >= %d", GEN_TILE_PAIRS);
		h->batchPairs = value;
		return SSC_OK;
	}
	if (!strcmp(key, "gzip")) { h->gzip = value != 0; return SSC_OK; }
	if (!strcmp(key, "bgzf")) { h->bgzf = value != 0; return SSC_OK; }        // takes effect with gzip, at the next call
	if (!strcmp(key, "interleave")) { h->interleave = value != 0; return SSC_OK; }   // slabs re-sized at the next call if they must
	if (!strcmp(key, "bam")) { h->bam = value != 0; return SSC_OK; }                 // likewise; the Huffman table is refitted
	if (!strcmp(key, "concurrent_move")) {
		if (value < 0 || value > 64) return fail(SSC_ERR_INVALID, "concurrent_move: 0 (off) .. 64 SMs");
		h->moverCtas = value < h->smCount ? (int)value : 0;     // the generation kernel needs SMs beside the mover
		return SSC_OK;
	}
	if (!strcmp(key, "fast_qmode")) {
		if (value != -1 && value != 8 && value != 16 && value != 2 && value != 0)
			return fail(SSC_ERR_INVALID, "fast_qmode must be -1 (automatic), 8, 16, 2 or 0");
		if (h->haveProfile) return fail(SSC_ERR_STATE, "fast_qmode must be set before ssc_set_profile");
		h->fastQmode = (int)value;
		return SSC_OK;
	}
	if (!strcmp(key, "max_ctas")) { if (value < 0) return fail(SSC_ERR_INVALID, "max_ctas must be >= 0"); h->maxCtas = (int)value; return SSC_OK; }
	if (!strcmp(key, "no_splice")) { h->noSplice = value != 0; return SSC_OK; }
	if (!strcmp(key, "force_generic")) { h->forceGeneric = value != 0; h->slabPairs = 0; return SSC_OK; }
	if (!strcmp(key, "fp64_search")) {
		if (h->havePlan) return fail(SSC_ERR_STATE, "fp64_search must be set before ssc_set_plan");
		h->fp64 = value != 0;
		return SSC_OK;
	}
	return fail(SSC_ERR_INVALID, "unknown option %s", key);
}

int ssc_set_profile(ssc_handle* h, const ssc_profile_tables* t) {
	if (!h || !t) return fail(SSC_ERR_INVALID, "null argument");
	CK(cudaSetDevice(h->device));
	const char* err = ssc::build_tables(t, &h->th);
	if (err[0]) return fail(SSC_ERR_INVALID, "profile rejected: %s", err);
	if (t->read_length > 320) return fail(SSC_ERR_INVALID, "read_length %d > 320 is not supported", t->read_length);
	cudaStream_t s = h->compute;
	ssc::DeviceTablesHost& th = h->th;
	CK(h->d_isizeT.upload(th.isize.T, s)); CK(h->d_isizeSym.upload(th.isize.sym, s));
	CK(h->d_insT.upload(th.insLen.T, s)); CK(h->d_insSym.upload(th.insLen.sym, s));
	CK(h->d_delT.upload(th.delLen.T, s)); CK(h->d_delSym.upload(th.delLen.sym, s));
	CK(h->d_qualT.upload(th.qualT, s)); CK(h->d_qualSym.upload(th.qualSym, s));
	CK(h->d_qualDiagT.upload(th.qualDiagT, s)); CK(h->d_qualDiagSym.upload(th.qualDiagSym, s));
	std::vector<uint4> sub(th.sub.size());
	for (size_t i = 0; i < sub.size(); i++) sub[i] = make_uint4(th.sub[i].s0, th.sub[i].s1, th.sub[i].s2, th.sub[i].base);
	CK(h->d_sub.upload(sub, s));
	std::vector<int8_t> lut(th.asciiCode, th.asciiCode + 256);
	CK(h->d_lut.upload(lut, s));
	size_t nsub = (size_t)th.nRows * th.B * 4, nq = (size_t)16 * th.B * th.Q;
	auto up = [&](DevBuf<double>& d, const double* p, size_t n) -> cudaError_t {
		std::vector<double> v(p ? p : nullptr, p ? p + n : nullptr);
		return d.upload(v, s);
	};
	CK(up(h->d_fIsize, t->isize_cdf, t->n_isize > 0 ? t->n_isize : 0));
	CK(up(h->d_fIns, t->ins_cdf, t->n_ins));
	CK(up(h->d_fDel, t->del_cdf, t->n_del));
	CK(up(h->d_fSub1, t->subs_cdf1, nsub));
	CK(up(h->d_fSub2, t->use_cdf2 ? t->subs_cdf2 : nullptr, t->use_cdf2 ? nsub : 0));
	CK(up(h->d_fQual, t->quality_cdf, nq));
	CK(cudaStreamSynchronize(s));

	ssc::DevTables& d = h->dt;
	memset(&d, 0, sizeof(d));
	d.N = th.N; d.K = th.K; d.B = th.B; d.Q = th.Q; d.minQ = th.minQ; d.RL = th.RL; d.paired = th.paired;
	d.useCdf2 = th.useCdf2; d.fixedInsert = th.fixedInsert; d.minIS = th.minIS; d.nRows = th.nRows;
	d.insT = th.insT; d.delT = th.delT; d.insEnable = th.insEnable; d.delEnable = th.delEnable;
	d.nIsize = (int)th.isize.T.size(); d.nInsLen = (int)th.insLen.T.size(); d.nDelLen = (int)th.delLen.T.size();
	d.isizeT = h->d_isizeT.p; d.isizeSym = h->d_isizeSym.p;
	d.insLenT = h->d_insT.p; d.insLenSym = h->d_insSym.p;
	d.delLenT = h->d_delT.p; d.delLenSym = h->d_delSym.p;
	d.sub = h->d_sub.p; d.nSub = th.nRows * th.B;
	d.qualT = h->d_qualT.p; d.qualSym = h->d_qualSym.p; d.qualPitch = th.qualPitch; d.nQualRows = 16 * th.B;
	d.maxQualRow = th.maxQualRow; d.fastQmode = h->fastQmode;
	d.qualBins = ssc::fast_choose_qbins(th.B, th.RL);
	d.qualDiagT = h->d_qualDiagT.p; d.qualDiagSym = h->d_qualDiagSym.p; d.qualDiagPitch = th.diagPitch;
	d.compLut = th.compLut;
	d.baseChars = (uint32_t)(uint8_t)th.baseChar[0] | ((uint32_t)(uint8_t)th.baseChar[1] << 8) |
	              ((uint32_t)(uint8_t)th.baseChar[2] << 16) | ((uint32_t)(uint8_t)th.baseChar[3] << 24);
	d.f_isize = h->d_fIsize.p; d.f_ins = h->d_fIns.p; d.f_del = h->d_fDel.p;
	d.f_sub1 = h->d_fSub1.p; d.f_sub2 = h->d_fSub2.p; d.f_qual = h->d_fQual.p;
	d.f_nIsize = t->n_isize; d.f_nIns = t->n_ins; d.f_nDel = t->n_del;
	d.insertRate = t->insert_rate;
	volatile double one_minus = 1 - t->insert_rate;
	d.delThresh = t->del_rate / one_minus;
	{
		// the conflict-scored bin pitch of the shared quality image must not cost the all-rows-in-shared-memory mode
		int qm = 0; size_t sb = 0;
		if (d.qualPitch == 8 && !(ssc::fast_supported(d, h->smemLimit, &qm, &sb) && qm == 8)) d.qualBins = d.B;
	}
	h->haveProfile = true;
	h->havePlan = false;
	h->haveGz = false;
	return SSC_OK;
}

int ssc_genome_reserve(ssc_handle* h, uint64_t total_bases) {
	if (!h) return fail(SSC_ERR_INVALID, "null handle");
	if (!h->haveProfile) return fail(SSC_ERR_STATE, "ssc_set_profile must precede ssc_genome_reserve (codes follow the profile's base order)");
	// checked before anything is allocated (k_winA / k_winB of gen_fast.cu; the 32-bit index is a deliberate saving)
	if (total_bases > SSC_MAX_STORE_BASES)
		return fail(SSC_ERR_INVALID, "haplotype store of %llu bases (limit %llu)", (unsigned long long)total_bases,
		            (unsigned long long)SSC_MAX_STORE_BASES);
	CK(cudaSetDevice(h->device));
	uint64_t groups = (total_bases + SSC_GPAD + 31) / 32 + 2;
	CK(h->d_hap2.alloc(groups * 2 + 64));
	CK(h->d_hapN.alloc(groups + 64));
	CK(cudaMemsetAsync(h->d_hap2.p, 0, (groups * 2 + 64) * 4, h->compute));
	CK(cudaMemsetAsync(h->d_hapN.p, 0, (groups + 64) * 4, h->compute));
	for (int i = 0; i < 2; i++) {
		if (!h->h_stage[i].p) CK(h->h_stage[i].alloc(h->stageBytes));
		if (!h->d_stage[i].p) CK(h->d_stage[i].alloc(h->stageBytes));
	}
	h->genomeCap = total_bases;
	h->genomeSize = 0;
	h->havePlan = false;
	return SSC_OK;
}

int ssc_genome_append(ssc_handle* h, const char* ascii, uint64_t n, uint64_t* first_base) {
	if (!h || (!ascii && n)) return fail(SSC_ERR_INVALID, "null argument");
	if (h->genomeSize + n > h->genomeCap) return fail(SSC_ERR_INVALID, "genome append exceeds the reserved %llu bases", (unsigned long long)h->genomeCap);
	CK(cudaSetDevice(h->device));
	if (first_base) *first_base = h->genomeSize;
	uint64_t done = 0;
	int k = 0;
	while (done < n) {
		uint64_t chunk = std::min<uint64_t>(h->stageBytes, n - done);
		CK(cudaEventSynchronize(h->evStage[k]));           // staging buffer k free again
		memcpy(h->h_stage[k].p, ascii + done, chunk);
		CK(cudaMemcpyAsync(h->d_stage[k].p, h->h_stage[k].p, chunk, cudaMemcpyHostToDevice, h->compute));
		CK(ssc::launch_pack(h->d_stage[k].p, chunk, SSC_GPAD + h->genomeSize + done, h->d_hap2.p, h->d_hapN.p, h->d_lut.p, h->compute));
		CK(cudaEventRecord(h->evStage[k], h->compute));
		h->stats.launches += 1;
		h->stats.h2d_bytes += chunk;
		done += chunk;
		k ^= 1;
	}
	h->genomeSize += n;
	return SSC_OK;
}

int ssc_reference_upload(ssc_handle* h, const char* ascii, uint64_t n) {
	if (!h || (!ascii && n)) return fail(SSC_ERR_INVALID, "null argument");
	CK(cudaSetDevice(h->device));
	if (h->d_ref.n < n) CK(h->d_ref.alloc((size_t)n + (size_t)n / 8 + 4096));
	CK(cudaStreamSynchronize(h->compute));          // earlier ssc_genome_append_ref launches still read the old reference
	// in stream order with the pack kernels that read it: a plain cudaMemcpy from pageable memory runs on the legacy stream,
	// which the (non-blocking) compute stream does not wait for, and may return before the DMA has landed
	if (n) CK(cudaMemcpyAsync(h->d_ref.p, ascii, (size_t)n, cudaMemcpyHostToDevice, h->compute));
	CK(cudaStreamSynchronize(h->compute));          // the caller may free the chromosome string
	h->refSize = n;
	h->stats.h2d_bytes += n;
	return SSC_OK;
}

}  // extern "C"

namespace {
// One FASTA record: file -> pinned staging (pread) -> raw (device) -> unfold kernel -> ref (device); returns when the
// unfolded record and the count of IUPAC characters are there.  `slot` 0 = the foreground set of staging buffers, 1 = the
// prefetch set.  Thread-safe against a concurrent call on the other slot (nothing of the handle is shared but the device).
int upload_fasta_record(ssc_handle* h, int slot, cudaStream_t s, DevBuf<uint8_t>& ref, DevBuf<uint8_t>& raw, DevBuf<unsigned long long>& otherBuf,
                        cudaEvent_t waitFor, int fd, uint64_t file_offset, uint64_t raw_len, uint64_t n_bases, uint32_t line_bases,
                        uint32_t line_width, uint64_t* n_other) {
	CK(cudaSetDevice(h->device));
	if (ref.n < n_bases + 16) CK(ref.alloc((size_t)n_bases + (size_t)n_bases / 8 + 4096));
	if (raw.n < raw_len) CK(raw.alloc((size_t)raw_len + (size_t)raw_len / 8 + 4096));
	if (!otherBuf.p) CK(otherBuf.alloc(1));
	const int NR = ssc_handle::FA_READERS, b0 = slot * NR;
	for (int i = b0; i < b0 + NR; i++) {
		if (!h->h_fa[i].p) CK(h->h_fa[i].alloc(h->faBytes));
		if (!h->evFa[i]) CK(create(h->evFa[i]));
	}
	if (waitFor) CK(cudaStreamWaitEvent(s, waitFor, 0));         // earlier readers of `ref` (pack kernels of the record before the last)
	CK(cudaMemsetAsync(otherBuf.p, 0, 8, s));
	// NR staging buffers, each fed by its own host thread (chunk c goes to reader c mod NR): the page-cache copy of pread is the
	// slow part, so two run at a time, under the DMA of earlier chunks
	const uint64_t nChunks = (raw_len + h->faBytes - 1) / h->faBytes;
	int rcs[ssc_handle::FA_READERS] = {SSC_OK, SSC_OK};
	std::string errMsg[ssc_handle::FA_READERS];
	auto feed = [&](int k) {
		if (cudaSetDevice(h->device) != cudaSuccess) { rcs[k] = SSC_ERR_CUDA; errMsg[k] = "cudaSetDevice failed"; return; }
		uint8_t* buf = h->h_fa[b0 + k].p;
		cudaEvent_t ev = h->evFa[b0 + k];
		for (uint64_t c = (uint64_t)k; c < nChunks; c += NR) {
			const uint64_t done = c * h->faBytes;
			const size_t chunk = (size_t)std::min<uint64_t>(h->faBytes, raw_len - done);
			cudaError_t e = cudaEventSynchronize(ev);                     // staging buffer free again
			size_t got = 0;
			while (e == cudaSuccess && got < chunk) {
				const ssize_t r = pread(fd, buf + got, chunk - got, (off_t)(file_offset + done + got));
				if (r < 0) { if (errno == EINTR) continue; rcs[k] = SSC_ERR_INVALID; errMsg[k] = std::string("reading the FASTA file failed: ") + strerror(errno); return; }
				if (r == 0) break;                                         // a last line without a line feed ends the file early
				got += (size_t)r;
			}
			if (got < chunk) memset(buf + got, '\n', chunk - got);
			if (e == cudaSuccess) e = cudaMemcpyAsync(raw.p + done, buf, chunk, cudaMemcpyHostToDevice, s);
			if (e == cudaSuccess) e = cudaEventRecord(ev, s);
			if (e != cudaSuccess) { rcs[k] = SSC_ERR_CUDA; errMsg[k] = std::string("staging the FASTA record failed: ") + cudaGetErrorString(e); return; }
		}
	};
	{
		std::vector<std::thread> readers;
		for (int k = 1; k < NR && (uint64_t)k < nChunks; k++) readers.emplace_back(feed, k);
		feed(0);
		for (auto& t : readers) t.join();
	}
	for (int k = 0; k < NR; k++) if (rcs[k]) return fail(rcs[k], "%s", errMsg[k].c_str());
	CK(ssc::launch_unfold(raw.p, raw_len, n_bases, line_bases, line_width, ref.p, otherBuf.p, s));
	unsigned long long other = 0;
	CK(cudaMemcpyAsync(&other, otherBuf.p, 8, cudaMemcpyDeviceToHost, s));
	CK(cudaStreamSynchronize(s));
	if (n_other) *n_other = other;
	return SSC_OK;
}

int check_fasta_geometry(uint64_t n_bases, uint32_t line_bases, uint32_t line_width) {
	if (n_bases >= (1ull << 32) - 64 || (n_bases && (line_bases == 0 || line_width < line_bases)))
		return fail(SSC_ERR_INVALID, "FASTA record geometry not supported (%llu bases, %u per line of %u bytes)",
		            (unsigned long long)n_bases, line_bases, line_width);
	return SSC_OK;
}
}  // namespace

extern "C" {

int ssc_reference_upload_fasta(ssc_handle* h, int fd, uint64_t file_offset, uint64_t raw_len, uint64_t n_bases,
                               uint32_t line_bases, uint32_t line_width, uint64_t* n_other) {
	if (!h || fd < 0) return fail(SSC_ERR_INVALID, "bad argument");
	if (h->prefetching) return fail(SSC_ERR_STATE, "a prefetched FASTA record is waiting: adopt it first");
	int rc = check_fasta_geometry(n_bases, line_bases, line_width);
	if (rc) return rc;
	rc = upload_fasta_record(h, 0, h->compute, h->d_ref, h->d_raw, h->d_other, nullptr, fd, file_offset, raw_len, n_bases, line_bases, line_width, n_other);
	if (rc) return rc;
	h->refSize = n_bases;
	h->stats.h2d_bytes += raw_len;
	h->stats.launches += 1;
	return SSC_OK;
}

int ssc_reference_prefetch_fasta(ssc_handle* h, int fd, uint64_t file_offset, uint64_t raw_len, uint64_t n_bases,
                                 uint32_t line_bases, uint32_t line_width) {
	if (!h || fd < 0) return fail(SSC_ERR_INVALID, "bad argument");
	if (h->prefetching) return fail(SSC_ERR_STATE, "one FASTA record can be prefetched at a time");
	int rc = check_fasta_geometry(n_bases, line_bases, line_width);
	if (rc) return rc;
	CK(cudaSetDevice(h->device));
	if (!h->upload) CK(create(h->upload));
	if (!h->evRefFree) CK(create(h->evRefFree));
	// the second buffer set was the current reference until the last adoption: its readers are in the compute stream by now
	CK(cudaEventRecord(h->evRefFree, h->compute));
	h->prefetching = true;
	h->prefetchRc = 0; h->prefetchErr.clear();
	h->prefetchBases = n_bases; h->prefetchRaw = raw_len; h->prefetchOther = 0;
	h->prefetchThread = std::thread([=]() {
		h->prefetchRc = upload_fasta_record(h, 1, h->upload, h->d_ref2, h->d_raw2, h->d_other2, h->evRefFree, fd, file_offset, raw_len, n_bases,
		                                    line_bases, line_width, &h->prefetchOther);
		if (h->prefetchRc) h->prefetchErr = g_err;          // (this thread's message, for the adopting thread)
	});
	return SSC_OK;
}

int ssc_reference_adopt_prefetched(ssc_handle* h, uint64_t* n_other) {
	if (!h) return fail(SSC_ERR_INVALID, "null handle");
	if (!h->prefetching) return fail(SSC_ERR_STATE, "no FASTA record was prefetched");
	h->prefetchThread.join();
	h->prefetching = false;
	if (h->prefetchRc) return fail(h->prefetchRc, "%s", h->prefetchErr.c_str());
	std::swap(h->d_ref, h->d_ref2); std::swap(h->d_raw, h->d_raw2); std::swap(h->d_other, h->d_other2);
	h->refSize = h->prefetchBases;
	h->stats.h2d_bytes += h->prefetchRaw;
	h->stats.launches += 1;
	if (n_other) *n_other = h->prefetchOther;
	return SSC_OK;
}

int ssc_genome_append_ref(ssc_handle* h, uint64_t ref_off, uint64_t len, int32_t reps, uint64_t* first_base) {
	if (!h || reps < 0) return fail(SSC_ERR_INVALID, "bad argument");
	if (ref_off + len > h->refSize) return fail(SSC_ERR_INVALID, "reference range outside the uploaded chromosome");
	if (h->genomeSize + len * (uint64_t)reps > h->genomeCap) return fail(SSC_ERR_INVALID, "genome append exceeds the reserved %llu bases", (unsigned long long)h->genomeCap);
	CK(cudaSetDevice(h->device));
	if (first_base) *first_base = h->genomeSize;
	for (int32_t r = 0; r < reps && len; r++) {
		CK(ssc::launch_pack(h->d_ref.p + ref_off, len, SSC_GPAD + h->genomeSize, h->d_hap2.p, h->d_hapN.p, h->d_lut.p, h->compute));
		h->genomeSize += len;
		h->stats.launches += 1;
	}
	return SSC_OK;
}

int ssc_genome_poke(ssc_handle* h, const int64_t* store_pos, const char* chars, int64_t n) {
	if (!h || n < 0 || (n && (!store_pos || !chars))) return fail(SSC_ERR_INVALID, "null argument");
	if (n == 0) return SSC_OK;
	CK(cudaSetDevice(h->device));
	for (int64_t i = 0; i < n; i++)
		if (store_pos[i] < 0 || (uint64_t)store_pos[i] >= h->genomeSize) return fail(SSC_ERR_INVALID, "poke %lld outside the haplotype store", (long long)i);
	DevBuf<int64_t> d_pos; DevBuf<uint8_t> d_ch;
	CK(d_pos.alloc((size_t)n)); CK(d_ch.alloc((size_t)n));
	CK(cudaMemcpyAsync(d_pos.p, store_pos, (size_t)n * 8, cudaMemcpyHostToDevice, h->compute));
	CK(cudaMemcpyAsync(d_ch.p, chars, (size_t)n, cudaMemcpyHostToDevice, h->compute));
	CK(ssc::launch_poke(h->d_hap2.p, h->d_hapN.p, d_pos.p, d_ch.p, n, h->d_lut.p, h->compute));
	CK(cudaStreamSynchronize(h->compute));
	h->stats.launches += 1;
	return SSC_OK;
}

int ssc_genome_read(ssc_handle* h, uint64_t start, uint64_t n, char* out) {
	if (!h || (!out && n)) return fail(SSC_ERR_INVALID, "null argument");
	if (start + n > h->genomeSize) return fail(SSC_ERR_INVALID, "range outside the haplotype store");
	if (n == 0) return SSC_OK;
	CK(cudaSetDevice(h->device));
	DevBuf<uint8_t> d_out;
	CK(d_out.alloc((size_t)n));
	CK(ssc::launch_unpack(h->d_hap2.p, h->d_hapN.p, SSC_GPAD + start, n, h->dt.baseChars, d_out.p, h->compute));
	CK(cudaMemcpyAsync(out, d_out.p, (size_t)n, cudaMemcpyDeviceToHost, h->compute));
	CK(cudaStreamSynchronize(h->compute));
	h->stats.launches += 1;
	return SSC_OK;
}

int ssc_genome_size(ssc_handle* h, uint64_t* n_bases) {
	if (!h || !n_bases) return fail(SSC_ERR_INVALID, "null argument");
	*n_bases = h->genomeSize;
	return SSC_OK;
}

int ssc_gc_census(ssc_handle* h, const int64_t* starts, const int32_t* lens, int64_t n, int32_t* gc, int32_t* nn) {
	if (!h || n < 0 || (n && (!starts || !lens || !gc || !nn))) return fail(SSC_ERR_INVALID, "null argument");
	if (!h->haveProfile || !h->d_hap2.p) return fail(SSC_ERR_STATE, "ssc_genome_append must precede ssc_gc_census");
	if (n == 0) return SSC_OK;
	if (n > 0x7fffffffLL * 8) return fail(SSC_ERR_INVALID, "too many intervals");
	CK(cudaSetDevice(h->device));
	for (int64_t i = 0; i < n; i++)
		if (starts[i] < 0 || lens[i] < 0 || (uint64_t)(starts[i] + lens[i]) > h->genomeSize)
			return fail(SSC_ERR_INVALID, "interval %lld outside the haplotype store", (long long)i);
	uint32_t gcCodes = 0;
	for (int k = 0; k < 4; k++) if (h->th.baseChar[k] == 'G' || h->th.baseChar[k] == 'C') gcCodes |= 1u << k;
	cudaStream_t s = h->compute;
	const bool timing = getenv("SIMUSCOP_TIMING") != nullptr;
	auto now = []() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
	double t0 = now();
	if (timing) { cudaStreamSynchronize(s); fprintf(stderr, "[simuscop timing] gc_census: drained the upload queue in %.3f s\n", now() - t0); t0 = now(); }
	// census buffers live in the handle and only grow (a cudaMalloc/cudaFree pair per call stalls for up to 0.7 s)
	DevBuf<int64_t>& d_starts = h->d_cenStarts; DevBuf<int32_t>& d_lens = h->d_cenLens; DevBuf<int32_t>& d_gc = h->d_cenGc; DevBuf<int32_t>& d_nn = h->d_cenNn;
	if (d_starts.n < (size_t)n) {
		const size_t cap = (size_t)n + (size_t)n / 2 + 1024;
		CK(d_starts.alloc(cap)); CK(d_lens.alloc(cap)); CK(d_gc.alloc(cap)); CK(d_nn.alloc(cap));
	}
	CK(cudaMemcpyAsync(d_starts.p, starts, (size_t)n * 8, cudaMemcpyHostToDevice, s));
	CK(cudaMemcpyAsync(d_lens.p, lens, (size_t)n * 4, cudaMemcpyHostToDevice, s));
	CK(ssc::launch_gc_census(h->d_hap2.p, h->d_hapN.p, d_starts.p, d_lens.p, n, gcCodes, d_gc.p, d_nn.p, s));
	CK(cudaMemcpyAsync(gc, d_gc.p, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
	CK(cudaMemcpyAsync(nn, d_nn.p, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
	CK(cudaStreamSynchronize(s));
	if (timing) fprintf(stderr, "[simuscop timing] gc_census: %lld intervals in %.3f s\n", (long long)n, now() - t0);
	h->stats.launches += 1;
	h->stats.h2d_bytes += (uint64_t)n * 12; h->stats.d2h_bytes += (uint64_t)n * 8;
	return SSC_OK;
}

int ssc_set_plan(ssc_handle* h, uint64_t seed, const ssc_bin* bins, int64_t n_bins, const ssc_segment* segs,
                 int64_t n_segs, const char* names, int64_t names_len, int64_t* planned_pairs, int64_t* emitted_pairs) {
	if (!h || (!bins && n_bins) || (!segs && n_segs) || (!names && names_len)) return fail(SSC_ERR_INVALID, "null argument");
	if (!h->haveProfile) return fail(SSC_ERR_STATE, "ssc_set_profile must precede ssc_set_plan");
	CK(cudaSetDevice(h->device));
	const ssc::DevTables& t = h->dt;
	const int RL = t.RL;
	const bool paired = t.paired != 0;
	h->seed = seed;
	h->havePlan = false;
	h->haveGz = false;
	h->pending.valid = false;

	// The per-bin passes below run on a few host threads over contiguous bin / segment ranges (a 3 Gb diploid plan has
	// 6 M bins); every result is position-determined, so the plan does not depend on the thread count.
	const unsigned T = (unsigned)std::max<int64_t>(1, std::min<int64_t>({16, (int64_t)std::thread::hardware_concurrency(), n_bins / 65536 + 1}));
	auto parallel = [&](int64_t n, const std::function<void(int64_t, int64_t, unsigned)>& fn) {
		if (T == 1 || n < 2) { fn(0, n, 0); return; }
		std::vector<std::thread> th;
		for (unsigned k = 1; k < T; k++) th.emplace_back(fn, n * k / T, n * (k + 1) / T, k);
		fn(0, n / T, 0);
		for (auto& x : th) x.join();
	};

	// ---- validate, planned pairs, risky bins
	std::vector<int64_t>& pb = h->planBaseAll;
	pb.assign(n_bins + 1, 0);
	std::vector<int32_t> planned(n_bins), emit(n_bins);
	std::vector<int32_t> riskyBase(n_bins, -1);
	int maxName = 0;
	if (names_len < 0 || names_len >= (1 << 17)) return fail(SSC_ERR_INVALID, "name blob of %lld bytes (limit 131071)", (long long)names_len);
	for (int64_t s = 0; s < n_segs; s++) {
		if (segs[s].first_bin < 0 || segs[s].n_bins < 0 || segs[s].first_bin + segs[s].n_bins > n_bins)
			return fail(SSC_ERR_INVALID, "segment %lld: bin range out of bounds", (long long)s);
		// a name is "@" + popu + "#" + chr + "#" (the '@' is written as part of it, 1..64 bytes)
		if (segs[s].name_len < 1 || segs[s].name_len > 64 || segs[s].name_offset < 0 || segs[s].name_offset + segs[s].name_len > names_len ||
		    names[segs[s].name_offset] != '@')
			return fail(SSC_ERR_INVALID, "segment %lld: bad name (1..64 bytes starting with '@')", (long long)s);
		maxName = std::max(maxName, (int)segs[s].name_len);
	}
	struct BinError { int64_t bin = -1; const char* what = nullptr; };
	std::vector<BinError> errs(T);
	std::vector<std::vector<int64_t>> riskyOf(T);              // bins that can fail, per thread range (ascending)
	parallel(n_bins, [&](int64_t lo, int64_t hi, unsigned tid) {
		for (int64_t i = lo; i < hi; i++) {
			const ssc_bin& b = bins[i];
			const int64_t n = b.read_count > 0 ? (paired ? ((int64_t)b.read_count + 1) / 2 : (int64_t)b.read_count) : 0;
			if (n > 0 && errs[tid].bin < 0) {
				const char* what = nullptr;
				if (b.segment < 0 || b.segment >= n_segs) what = "bad segment";
				else if (b.spos < 0 || b.epos < b.spos) what = "bad range";
				else if (b.segsize == 0) what = "segsize 0 (copy number 0 segments cannot emit reads)";
				else if (b.hap_base < 0 || b.contig_end < b.hap_base || (uint64_t)b.contig_end > h->genomeSize) what = "haplotype range outside the store";
				else if (n > 0x7fffffff) what = "too many reads";
				if (what) { errs[tid].bin = i; errs[tid].what = what; }
			}
			planned[i] = (int32_t)n;
			emit[i] = (int32_t)n;
			if (n > 0) {
				// an attempt fails iff min(want, contig_end - (hap_base+pos)) < RL  (Segment.cpp:753)
				bool risky = (int64_t)b.epos > b.contig_end - b.hap_base - RL;
				if (!paired && ((int64_t)b.epos - b.spos + 1) < RL) risky = true;
				if (paired && t.nIsize == 0 && t.fixedInsert < RL) risky = true;
				if (paired && t.nIsize > 0 && t.minIS < RL) risky = true;          // an insert-size table that reaches below the read length
				if (risky) riskyOf[tid].push_back(i);
			}
		}
	});
	for (unsigned k = 0; k < T; k++)
		if (errs[k].bin >= 0) return fail(SSC_ERR_INVALID, "bin %lld: %s", (long long)errs[k].bin, errs[k].what);
	for (int64_t i = 0; i < n_bins; i++) pb[i + 1] = pb[i] + planned[i];
	h->plannedPairs = pb[n_bins];
	std::vector<ssc::CensusBin> census;
	std::vector<int64_t> censusOf;            // census index -> bin
	int64_t riskyTotal = 0;
	for (unsigned k = 0; k < T; k++)
		for (int64_t i : riskyOf[k]) {
			const ssc_bin& b = bins[i];
			const int64_t n = planned[i];
			ssc::CensusBin c;
			c.hap_base = b.hap_base + SSC_GPAD; c.contig_end = b.contig_end + SSC_GPAD; c.plan_base = pb[i];
			c.spos = b.spos; c.epos = b.epos; c.planned = (int32_t)n; c.risky_base = (int32_t)riskyTotal;
			if (riskyTotal + n > 0x7fffffff) return fail(SSC_ERR_INVALID, "too many pairs in bins that can fail");
			riskyBase[i] = (int32_t)riskyTotal;
			riskyTotal += n;
			census.push_back(c);
			censusOf.push_back(i);
		}

	// ---- census on the device
	cudaStream_t s = h->compute;
	CK(h->d_risky.alloc((size_t)std::max<int64_t>(riskyTotal, 1)));
	if (!census.empty()) {
		DevBuf<ssc::CensusBin> d_census;
		DevBuf<int32_t> d_emitted;
		CK(d_census.upload(census, s));
		CK(d_emitted.alloc(census.size()));
		CK(ssc::launch_census(t, h->fp64, d_census.p, (int)census.size(), seed, h->d_risky.p, d_emitted.p, s));
		std::vector<int32_t> em(census.size());
		CK(cudaMemcpyAsync(em.data(), d_emitted.p, em.size() * 4, cudaMemcpyDeviceToHost, s));
		CK(cudaStreamSynchronize(s));
		h->stats.launches += 1;
		for (size_t k = 0; k < census.size(); k++) emit[censusOf[k]] = em[k];
	}

	// ---- prefix sums, compaction
	std::vector<int64_t>& eb = h->emitBaseAll;
	eb.assign(n_bins + 1, 0);
	for (int64_t i = 0; i < n_bins; i++) eb[i + 1] = eb[i] + emit[i];
	h->emittedPairs = eb[n_bins];
	// device bins of segment sIdx go to dev[segOff[sIdx] ...): bins must be listed segment by segment in order, otherwise
	// emit order != bin order
	std::vector<int64_t> segOff(n_segs + 1, 0);
	std::vector<const char*> segErr(T, nullptr);
	std::vector<int64_t> segErrAt(T, -1);
	parallel(n_segs, [&](int64_t lo, int64_t hi, unsigned tid) {
		for (int64_t sIdx = lo; sIdx < hi; sIdx++) {
			int64_t cnt = 0, fragBase = 0;
			for (int64_t i = segs[sIdx].first_bin; i < segs[sIdx].first_bin + segs[sIdx].n_bins; i++) {
				if (emit[i] > 0) {
					cnt++;
					if (segErrAt[tid] < 0 && bins[i].segment != sIdx) { segErrAt[tid] = i; segErr[tid] = "does not belong to the segment that lists it"; }
					if (segErrAt[tid] < 0 && fragBase + emit[i] > 0x7fffffff) { segErrAt[tid] = i; segErr[tid] = "fragment counter overflow of its segment"; }
				}
				fragBase += emit[i];
			}
			segOff[sIdx + 1] = cnt;
		}
	});
	for (unsigned k = 0; k < T; k++) if (segErrAt[k] >= 0) return fail(SSC_ERR_INVALID, "bin %lld %s", (long long)segErrAt[k], segErr[k]);
	for (int64_t sIdx = 0; sIdx < n_segs; sIdx++) segOff[sIdx + 1] += segOff[sIdx];
	const size_t nDev = (size_t)segOff[n_segs];
	std::vector<int64_t>& devEmitBase = h->devEmitBase;
	devEmitBase.assign(nDev + 1, 0);
	// The device bins (64 bytes each, 384 MB for a 3 Gb diploid plan) are formatted straight into the two pinned staging
	// buffers, a run of whole segments at a time, and copied from there: no pageable image of the table is ever built.
	for (int i = 0; i < 2; i++) {
		if (!h->h_stage[i].p) CK(h->h_stage[i].alloc(h->stageBytes));
		CK(cudaEventSynchronize(h->evStage[i]));
	}
	CK(h->d_bins.alloc(std::max<size_t>(nDev, 1)));
	const size_t perChunk = h->stageBytes / sizeof(ssc::DevBin);
	int stage = 0;
	for (int64_t s0 = 0; s0 < n_segs;) {
		int64_t s1 = s0;
		while (s1 < n_segs && (size_t)(segOff[s1 + 1] - segOff[s0]) <= perChunk) s1++;
		if (s1 == s0) return fail(SSC_ERR_INVALID, "segment %lld has more than %zu bins", (long long)s0, perChunk);
		const int64_t o0 = segOff[s0], cnt = segOff[s1] - o0;
		if (cnt > 0) {
			CK(cudaEventSynchronize(h->evStage[stage]));
			ssc::DevBin* out = (ssc::DevBin*)h->h_stage[stage].p;
			parallel(s1 - s0, [&](int64_t lo, int64_t hi, unsigned) {
				for (int64_t sIdx = s0 + lo; sIdx < s0 + hi; sIdx++) {
					int64_t fragBase = 0, o = segOff[sIdx];
					for (int64_t i = segs[sIdx].first_bin; i < segs[sIdx].first_bin + segs[sIdx].n_bins; i++) {
						if (emit[i] > 0) {
							ssc::DevBin d;
							d.hap_base = bins[i].hap_base + SSC_GPAD; d.contig_end = bins[i].contig_end + SSC_GPAD;
							d.plan_base = pb[i]; d.emit_base = eb[i];
							d.spos = bins[i].spos; d.epos = bins[i].epos; d.segsize = bins[i].segsize;
							d.frag_base = (int32_t)fragBase;
							d.name_off = segs[sIdx].name_offset; d.name_len = segs[sIdx].name_len;
							d.risky_base = riskyBase[i]; d.segment = (int32_t)sIdx;
							out[o - o0] = d;
							devEmitBase[(size_t)o] = eb[i];
							o++;
						}
						fragBase += emit[i];
					}
				}
			});
			CK(cudaMemcpyAsync(h->d_bins.p + o0, out, (size_t)cnt * sizeof(ssc::DevBin), cudaMemcpyHostToDevice, s));
			CK(cudaEventRecord(h->evStage[stage], s));
			stage ^= 1;
		}
		s0 = s1;
	}
	devEmitBase[nDev] = h->emittedPairs;
	for (size_t k = 1; k + 1 < devEmitBase.size(); k++)
		if (devEmitBase[k] <= devEmitBase[k - 1]) return fail(SSC_ERR_INVALID, "segments must list their bins in increasing, non-overlapping order");
	h->nDevBins = (int64_t)nDev;
	CK(h->d_emitBase.upload(devEmitBase, s));
	std::vector<char> nm(names, names + names_len);
	nm.push_back(0);
	CK(h->d_names.upload(nm, s));
	CK(cudaStreamSynchronize(s));
	h->names.swap(nm);
	h->segNameOff.resize((size_t)n_segs); h->segNameLen.resize((size_t)n_segs);
	for (int64_t k = 0; k < n_segs; k++) { h->segNameOff[(size_t)k] = segs[k].name_offset; h->segNameLen[(size_t)k] = segs[k].name_len; }
	// BAM output takes names made of the SAM QNAME characters [!-?A-~] only: the first segment with another byte after its '@'
	h->badQnameSeg = -1;
	for (int64_t k = 0; k < n_segs && h->badQnameSeg < 0; k++)
		for (int32_t i = 1; i < segs[k].name_len; i++) {
			const uint8_t c = (uint8_t)h->names[(size_t)(segs[k].name_offset + i)];
			if (c < '!' || c > '~' || c == '@') { h->badQnameSeg = k; h->badQnameByte = c; break; }
		}
	h->maxName = maxName;
	h->stats.h2d_bytes += nDev * sizeof(ssc::DevBin) + devEmitBase.size() * 8;
	// worst-case record bytes per pair per file: header + 2*(RL + 96) + 4
	h->maxRecBytes = maxName + 10 + 1 + 10 + 3 + 2 * (RL + 96) + 4;
	h->havePlan = true;
	if (planned_pairs) *planned_pairs = h->plannedPairs;
	if (emitted_pairs) *emitted_pairs = h->emittedPairs;
	return SSC_OK;
}

// BAM output of a plan whose read names are not all valid QNAMEs is refused before anything is generated
static int check_bam_names(const ssc_handle* h) {
	if (!h->bam || h->badQnameSeg < 0) return SSC_OK;
	return fail(SSC_ERR_INVALID, "bam: segment %lld: its name holds byte 0x%02x, which a BAM read name may not hold (SAM QNAME [!-?A-~])",
	            (long long)h->badQnameSeg, h->badQnameByte);
}

// The pipeline of ssc_generate.  Every error return goes through bail() in ssc_generate.
static int generate_batches(ssc_handle* h, int64_t pair_lo, int64_t pair_hi, ssc_sink_fn sink, void* user) {
	int rc = ensure_batch_resources(h, true);
	if (rc) return rc;
	const int64_t eLo = emit_index_of_plan(h, pair_lo), eHi = emit_index_of_plan(h, pair_hi);
	if (eHi <= eLo) return SSC_OK;
	const int nFiles = out_files(h);
	struct Batch { int64_t lo, hi; };
	std::vector<Batch> batches;
	for (int64_t e = eLo; e < eHi; e += h->slabPairs) batches.push_back({e, std::min(eHi, e + h->slabPairs)});
	const int nb = (int)batches.size();
	// pipeline: the launch of batch k+1 (under which the mover completes the dense slab of batch k) runs under the device->host
	// copies of batch k-1 (file 1 / file 2 on two streams), which run under the sink of batch k-2.  h_out[k & 1] was consumed by
	// the sink of batch k-2 an iteration before the copy of batch k is issued.
	int qm = 0; size_t sb = 0;
	const bool moverCompletes = use_fast(h, &qm, &sb) && !gz_mode(h) && h->moverCtas > 0;   // batch k's dense slab under launch k+1
	auto launch = [&](int k) -> int {
		// the dense slab this launch writes: d_out[(k-1) & 1] when the mover completes the previous batch under it, else
		// d_out[k & 1]; its last reader is the copy of the batch two before the one that now lands there
		const int target = moverCompletes ? (k + 1) & 1 : k & 1;
		CK(cudaStreamWaitEvent(h->compute, h->set[target].evCopy, 0));
		CK(cudaStreamWaitEvent(h->compute, h->set[target].evCopy2, 0));
		int r = launch_batch(h, k & 1, batches[k].lo, batches[k].hi);
		if (r) return r;
		if (!moverCompletes) CK(cudaEventRecord(h->set[k & 1].evDense, h->compute));     // the dense slab of batch k is complete with its own launch
		return SSC_OK;
	};
	rc = launch(0);
	if (rc) return rc;
	ssc::BatchResult res[2];
	for (int k = 0; k < nb; k++) {
		const int buf = k & 1;
		rc = k + 1 < nb ? launch(k + 1) : flush_pending(h);         // after this the dense slab of batch k is in the stream
		if (rc) return rc;
		if (moverCompletes) CK(cudaEventRecord(h->set[buf].evDense, h->compute));    // (its pass 2b came with the launch of batch k+1)
		CK(cudaEventSynchronize(h->set[buf].evResult));
		res[buf] = *h->set[buf].h_result.p;
		rc = check_result(h, res[buf]);
		if (rc) return rc;
		CK(cudaStreamWaitEvent(h->copy, h->set[buf].evDense, 0));
		CK(cudaMemcpyAsync(h->set[buf].h_out[0].p, h->set[buf].d_out[0].p, res[buf].bytes1, cudaMemcpyDeviceToHost, h->copy));
		CK(cudaEventRecord(h->set[buf].evCopy, h->copy));
		if (nFiles == 2) {
			CK(cudaStreamWaitEvent(h->copy2, h->set[buf].evDense, 0));
			CK(cudaMemcpyAsync(h->set[buf].h_out[1].p, h->set[buf].d_out[1].p, res[buf].bytes2, cudaMemcpyDeviceToHost, h->copy2));
		}
		CK(cudaEventRecord(h->set[buf].evCopy2, h->copy2));
		h->stats.d2h_bytes += res[buf].bytes1 + res[buf].bytes2;
		if (k >= 1) {
			const int pb = (k - 1) & 1;
			CK(cudaEventSynchronize(h->set[pb].evCopy));
			CK(cudaEventSynchronize(h->set[pb].evCopy2));
			int src = sink(user, (const char*)h->set[pb].h_out[0].p, res[pb].bytes1, nFiles == 2 ? (const char*)h->set[pb].h_out[1].p : nullptr,
			               nFiles == 2 ? res[pb].bytes2 : 0, batches[k - 1].lo, batches[k - 1].hi - batches[k - 1].lo);
			if (src) return fail(SSC_ERR_SINK, "sink returned %d", src);
		}
	}
	{
		const int pb = (nb - 1) & 1;
		CK(cudaEventSynchronize(h->set[pb].evCopy));
		CK(cudaEventSynchronize(h->set[pb].evCopy2));
		int src = sink(user, (const char*)h->set[pb].h_out[0].p, res[pb].bytes1, nFiles == 2 ? (const char*)h->set[pb].h_out[1].p : nullptr,
		               nFiles == 2 ? res[pb].bytes2 : 0, batches[nb - 1].lo, batches[nb - 1].hi - batches[nb - 1].lo);
		if (src) return fail(SSC_ERR_SINK, "sink returned %d", src);
	}
	return SSC_OK;
}

int ssc_generate(ssc_handle* h, int64_t pair_lo, int64_t pair_hi, ssc_sink_fn sink, void* user) {
	if (!h || !sink) return fail(SSC_ERR_INVALID, "null argument");
	if (!h->havePlan) return fail(SSC_ERR_STATE, "ssc_set_plan must precede ssc_generate");
	if (pair_lo < 0 || pair_hi < pair_lo) return fail(SSC_ERR_INVALID, "bad pair range");
	if (check_bam_names(h)) return SSC_ERR_INVALID;
	CK(cudaSetDevice(h->device));
	const int rc = generate_batches(h, pair_lo, pair_hi, sink, user);
	return rc ? bail(h, rc) : SSC_OK;
}

// The pipeline of ssc_generate_device; the totals are added to *b1, *b2, *nb.  Every error return goes through bail() in
// ssc_generate_device.
static int generate_device_batches(ssc_handle* h, int64_t pair_lo, int64_t pair_hi, uint64_t* b1, uint64_t* b2, uint64_t* nb,
                                   float* ms) {
	int rc = ensure_batch_resources(h, false);
	if (rc) return rc;
	const int64_t eLo = emit_index_of_plan(h, pair_lo), eHi = emit_index_of_plan(h, pair_hi);
	if (eHi <= eLo) return SSC_OK;
	h->timeKernels = true; h->kevUsed = 0;
	CK(cudaEventRecord(h->evStart, h->compute));
	int k = 0;
	for (int64_t e = eLo; e < eHi; e += h->slabPairs, k++) {
		const int buf = k & 1;
		if (k >= 2) {
			CK(cudaEventSynchronize(h->set[buf].evResult));
			ssc::BatchResult r = *h->set[buf].h_result.p;
			rc = check_result(h, r);
			if (rc) return rc;
			*b1 += r.bytes1; *b2 += r.bytes2; *nb += r.bases;
		}
		rc = launch_batch(h, buf, e, std::min(eHi, e + h->slabPairs));
		if (rc) return rc;
	}
	rc = flush_pending(h);                      // the last batch's blobs: stand-alone move, timed with the scans as "pass 2"
	if (rc) return rc;
	CK(cudaEventRecord(h->evStop, h->compute));    // the compute stream has waited for the mover stream's last work
	CK(cudaEventSynchronize(h->evStop));
	for (int j = std::max(0, k - 2); j < k; j++) {
		CK(cudaEventSynchronize(h->set[j & 1].evResult));
		ssc::BatchResult r = *h->set[j & 1].h_result.p;
		rc = check_result(h, r);
		if (rc) return rc;
		*b1 += r.bytes1; *b2 += r.bytes2; *nb += r.bases;
	}
	CK(cudaEventElapsedTime(ms, h->evStart, h->evStop));
	h->stats.device_ms += *ms;
	h->timeKernels = false;
	for (int i = 0; i < h->kevUsed; i++) {
		float t = 0;
		CK(cudaEventElapsedTime(&t, h->kev[2 * i], h->kev[2 * i + 1]));
		*h->kevSum[i] += t;
		if (h->kevSum[i] == &h->stats.gen_kernel_ms) h->stats.timed_batches += 1;
	}
	return SSC_OK;
}

int ssc_generate_device(ssc_handle* h, int64_t pair_lo, int64_t pair_hi, uint64_t* bytes1, uint64_t* bytes2,
                        uint64_t* bases, double* device_ms) {
	if (!h) return fail(SSC_ERR_INVALID, "null handle");
	if (!h->havePlan) return fail(SSC_ERR_STATE, "ssc_set_plan must precede ssc_generate_device");
	if (pair_lo < 0 || pair_hi < pair_lo) return fail(SSC_ERR_INVALID, "bad pair range");
	if (check_bam_names(h)) return SSC_ERR_INVALID;
	CK(cudaSetDevice(h->device));
	uint64_t b1 = 0, b2 = 0, nb = 0;
	float ms = 0;
	const int rc = generate_device_batches(h, pair_lo, pair_hi, &b1, &b2, &nb, &ms);
	if (rc) return bail(h, rc);
	if (bytes1) *bytes1 = b1;
	if (bytes2) *bytes2 = b2;
	if (bases) *bases = nb;
	if (device_ms) *device_ms = ms;
	return SSC_OK;
}

// bytes between the base rows of two consecutive reads' slots: RL + 96 (the longest read emitted) rounded up to 16
static int32_t read_pitch(const ssc_handle* h) { return (h->dt.RL + 96 + 15) / 16 * 16; }

int ssc_read_shape(ssc_handle* h, int64_t pair_lo, int64_t pair_hi, int64_t* n_pairs, int32_t* n_mates, int32_t* pitch) {
	if (!h || !n_pairs || !n_mates || !pitch) return fail(SSC_ERR_INVALID, "null argument");
	if (!h->havePlan) return fail(SSC_ERR_STATE, "ssc_set_plan must precede ssc_read_shape");
	if (pair_lo < 0 || pair_hi < pair_lo) return fail(SSC_ERR_INVALID, "bad pair range");
	*n_pairs = emit_index_of_plan(h, pair_hi) - emit_index_of_plan(h, pair_lo);
	*n_mates = h->dt.paired ? 2 : 1;
	*pitch = read_pitch(h);
	return SSC_OK;
}

int ssc_segment_name(ssc_handle* h, int32_t segment, char* out, int32_t cap) {
	if (!h || !out) return fail(SSC_ERR_INVALID, "null argument");
	if (!h->havePlan) return fail(SSC_ERR_STATE, "ssc_set_plan must precede ssc_segment_name");
	if (segment < 0 || (size_t)segment >= h->segNameOff.size())
		return fail(SSC_ERR_INVALID, "segment %d out of range (%zu segments)", segment, h->segNameOff.size());
	const int32_t len = h->segNameLen[(size_t)segment];
	if (cap < len + 1) return fail(SSC_ERR_INVALID, "segment name of %d bytes needs a buffer of %d bytes, got %d", len, len + 1, cap);
	memcpy(out, h->names.data() + h->segNameOff[(size_t)segment], (size_t)len);
	out[len] = 0;
	return SSC_OK;
}

// The batches of ssc_generate_reads, emitted pairs [eLo, eHi), back to back on the compute stream.  Every error return goes
// through bail() in ssc_generate_reads.
static int generate_read_batches(ssc_handle* h, int64_t eLo, int64_t eHi, const ssc_read_arrays* out, cudaStream_t caller, int qmode,
                                 size_t smem) {
	const int M = h->dt.paired ? 2 : 1;
	const uint64_t perPair = (uint64_t)M * 2u * (uint64_t)out->pitch;
	// the kernel addresses a batch's slots with 32-bit offsets
	const int64_t pairs = std::min<int64_t>({h->batchPairs, eHi - eLo, (int64_t)(((1ull << 32) - 1) / perPair)});
	const int maxTiles = (int)((pairs + FG_CHUNK - 1) / FG_CHUNK);
	if (h->d_rdTileStart.n < (size_t)maxTiles) CK(h->d_rdTileStart.alloc((size_t)maxTiles));
	if (!h->d_rdTicket.p) CK(h->d_rdTicket.alloc(1));
	if (!h->d_rdResult.p) CK(h->d_rdResult.alloc(1));
	cudaStream_t s = h->compute;
	CK(cudaEventRecord(h->evCaller, caller));         // work the caller queued before the call (e.g. on the output arrays) goes first
	CK(cudaStreamWaitEvent(s, h->evCaller, 0));
	CK(cudaMemsetAsync(h->d_rdResult.p, 0, sizeof(ssc::BatchResult), s));
	h->stats.gen_kernel = 1; h->stats.gen_nch = ssc::fast_nch(h->dt.RL); h->stats.gen_qmode = qmode;
	h->stats.gen_smem_bytes = (int32_t)smem;
	for (int64_t lo = eLo; lo < eHi; lo += pairs) {
		const int64_t hi = std::min(eHi, lo + pairs), row = lo - eLo;
		const int nTiles = (int)((hi - lo + FG_CHUNK - 1) / FG_CHUNK);
		CK(cudaMemsetAsync(h->d_rdTicket.p, 0, sizeof(unsigned int), s));
		CK(ssc::launch_locate(h->d_emitBase.p, h->nDevBins, lo, FG_CHUNK, nTiles, h->d_rdTileStart.p, s));
		ssc::GenParams P = batch_params(h, lo, hi, qmode == 8);
		P.tileStartBin = h->d_rdTileStart.p; P.nTiles = nTiles; P.ticket = h->d_rdTicket.p; P.result = h->d_rdResult.p;
		P.out1 = out->reads + (uint64_t)row * perPair;
		P.rdLength = out->length + row * M; P.rdPairId = out->pair_id + row;
		P.rdSegment = out->segment + row; P.rdPos = out->pos + row; P.rdFrag = out->frag + row;
		P.pitch = (uint32_t)out->pitch;
		// nothing to move: every SM generates
		int grid = std::min((nTiles + FG_GEN - 1) / FG_GEN, h->smCount);
		if (h->maxCtas > 0) grid = std::min(grid, h->maxCtas);
		CK(ssc::launch_generate_reads(P, qmode, smem, grid, s));
		h->stats.launches += 2;
	}
	ssc::BatchResult r;
	CK(cudaMemcpyAsync(&r, h->d_rdResult.p, sizeof(r), cudaMemcpyDeviceToHost, s));
	CK(cudaStreamSynchronize(s));
	return check_result(h, r);
}

int ssc_generate_reads(ssc_handle* h, int64_t pair_lo, int64_t pair_hi, const ssc_read_arrays* out, void* stream, int64_t* n_pairs) {
	if (!h || !out) return fail(SSC_ERR_INVALID, "null argument");
	if (!h->havePlan) return fail(SSC_ERR_STATE, "ssc_set_plan must precede ssc_generate_reads");
	if (pair_lo < 0 || pair_hi < pair_lo) return fail(SSC_ERR_INVALID, "bad pair range");
	if (!out->reads || !out->length || !out->pair_id || !out->segment || !out->pos || !out->frag)
		return fail(SSC_ERR_INVALID, "ssc_generate_reads: null array pointer in ssc_read_arrays");
	if (((uintptr_t)out->reads & 15) || ((uintptr_t)out->length & 1) || ((uintptr_t)out->pair_id & 7) || ((uintptr_t)out->segment & 3) ||
	    ((uintptr_t)out->pos & 3) || ((uintptr_t)out->frag & 3))
		return fail(SSC_ERR_INVALID, "ssc_generate_reads: reads must be 16-byte aligned, the other arrays aligned to their element size");
	if (out->pitch != read_pitch(h))
		return fail(SSC_ERR_INVALID, "ssc_generate_reads: pitch %d, the plan's read length %d needs %d (ssc_read_shape)", out->pitch, h->dt.RL,
		            read_pitch(h));
	const int64_t eLo = emit_index_of_plan(h, pair_lo), eHi = emit_index_of_plan(h, pair_hi);
	if (out->capacity < eHi - eLo)
		return fail(SSC_ERR_INVALID, "ssc_generate_reads: capacity %lld pairs, the range emits %lld", (long long)out->capacity,
		            (long long)(eHi - eLo));
	if (h->fp64) return fail(SSC_ERR_INVALID, "array output needs the fast kernel; fp64_search selects the FP64 ground-truth kernel");
	if (h->forceGeneric) return fail(SSC_ERR_INVALID, "array output needs the fast kernel; force_generic selects the generic kernel");
	int qmode = 0; size_t smem = 0;
	if (!use_fast(h, &qmode, &smem))
		return fail(SSC_ERR_INVALID, "array output needs the fast kernel (kmer 3, read length 33..160, tables within shared memory); "
		            "this profile has kmer %d, read length %d", h->dt.K, h->dt.RL);
	CK(cudaSetDevice(h->device));
	if (eHi > eLo) {
		const int rc = generate_read_batches(h, eLo, eHi, out, (cudaStream_t)stream, qmode, smem);
		if (rc) return bail(h, rc);
	}
	if (n_pairs) *n_pairs = eHi - eLo;
	return SSC_OK;
}

int ssc_table_lookup_host(const double* cdf, int n, uint32_t u) {
	if (!cdf || n < 1) return -1;
	ssc::CompressedCdf c = ssc::compress_cdf(cdf, n);
	size_t k = 0;
	while (k + 1 < c.T.size() && c.T[k] < u) k++;
	return (int)c.sym[k];
}

int ssc_sub_lookup_host(const double* cdf4, uint32_t u) {
	if (!cdf4) return -1;
	ssc::SubRow r = ssc::make_sub_row(cdf4);
	return (int)(r.base + (u > r.s0) + (u > r.s1) + (u > r.s2));
}

int64_t ssc_gzip_member_host(const uint8_t* in, uint32_t n, const uint8_t* sample, size_t sample_n, uint8_t* out, size_t cap) {
	if (!in || !out || n == 0) return -1;
	uint64_t hist[256];
	memset(hist, 0, sizeof(hist));
	for (size_t i = 0; i < sample_n; i++) hist[sample[i]]++;
	ssc::GzTables tab;
	const char* err = ssc::gz_build_tables(hist, &tab);
	if (err[0]) { fail(SSC_ERR_INVALID, "gzip tables: %s", err); return -1; }
	return (int64_t)ssc::gz_member_host(&tab, in, n, out, cap);
}

// a read group id: 1..64 bytes of [!-~]
static bool valid_read_group(const char* id, size_t n) {
	if (n < 1 || n > 64) return false;
	for (size_t i = 0; i < n; i++) if ((uint8_t)id[i] < '!' || (uint8_t)id[i] > '~') return false;
	return true;
}

int ssc_set_read_group(ssc_handle* h, const char* id) {
	if (!h) return fail(SSC_ERR_INVALID, "null handle");
	const size_t n = id ? strlen(id) : 0;
	if (n == 0) { h->rgLen = 0; return SSC_OK; }
	if (!valid_read_group(id, n)) return fail(SSC_ERR_INVALID, "read group id must be 1..64 printable characters without spaces ([!-~])");
	CK(cudaSetDevice(h->device));
	if (!h->d_rg.p) CK(h->d_rg.alloc(64));
	// in stream order behind the kernels of earlier calls, which read the old id
	CK(cudaMemcpyAsync(h->d_rg.p, id, n, cudaMemcpyHostToDevice, h->compute));
	CK(cudaStreamSynchronize(h->compute));
	h->rgLen = (int)n;
	return SSC_OK;
}

int64_t ssc_bam_header(const char* read_group, uint8_t* out, size_t cap) {
	const size_t n = read_group ? strlen(read_group) : 0;
	if ((n && !valid_read_group(read_group, n)) || (!out && cap)) { fail(SSC_ERR_INVALID, "ssc_bam_header: bad argument"); return -1; }
	std::string text = "@HD\tVN:1.6\tSO:unsorted\tGO:query\n";
	if (n) text += "@RG\tID:" + std::string(read_group, n) + "\tSM:" + std::string(read_group, n) + "\n";
	std::vector<uint8_t> raw = {'B', 'A', 'M', 1};
	auto le32 = [](std::vector<uint8_t>& v, uint32_t x) { for (int k = 0; k < 4; k++) v.push_back((uint8_t)(x >> (8 * k))); };
	le32(raw, (uint32_t)text.size());
	raw.insert(raw.end(), text.begin(), text.end());
	le32(raw, 0);                                   // n_ref
	// one stored BGZF block: header with the BC field, a final stored DEFLATE block, CRC-32, ISIZE
	const size_t total = raw.size() + ssc::GZ_BGZF_STORED_EXTRA;
	if (cap < total) return 0;
	std::vector<uint8_t> b = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0, (uint8_t)((total - 1) & 0xff), (uint8_t)((total - 1) >> 8),
	                          1, (uint8_t)(raw.size() & 0xff), (uint8_t)(raw.size() >> 8), (uint8_t)(~raw.size() & 0xff), (uint8_t)((~raw.size() >> 8) & 0xff)};
	b.insert(b.end(), raw.begin(), raw.end());
	le32(b, ssc::gz_crc32_host(raw.data(), raw.size()));
	le32(b, (uint32_t)raw.size());
	memcpy(out, b.data(), b.size());
	return (int64_t)b.size();
}

int ssc_issue_floor(ssc_handle* h, int mode, int read_length, int64_t n_pairs, int reps, double* ms_per_launch) {
	if (!h || !ms_per_launch) return fail(SSC_ERR_INVALID, "null argument");
	if (mode < 0 || mode > 1 || read_length < 33 || read_length > 160 || n_pairs < FG_CHUNK || n_pairs > (1 << 22) || reps < 1)
		return fail(SSC_ERR_INVALID, "ssc_issue_floor: mode 0/1, read_length 33..160, n_pairs 32..4194304, reps >= 1");
	CK(cudaSetDevice(h->device));
	const int64_t nTiles = (n_pairs + FG_CHUNK - 1) / FG_CHUNK;
	const uint32_t blobPitch = FG_CHUNK * FG_SLOT;
	DevBuf<uint32_t> scratch; DevBuf<uint8_t> blobs;
	CK(scratch.alloc(1 + (size_t)h->smCount * FG_WORKERS));
	const size_t fileBytes = (size_t)nTiles * blobPitch + 256;
	if (mode == 1) {
		if (2 * fileBytes >= (1ull << 32)) return fail(SSC_ERR_INVALID, "ssc_issue_floor: n_pairs too large for 32-bit blob cursors");
		CK(blobs.alloc(2 * fileBytes));
	}
	cudaStream_t s = h->compute;
	const int grid = (int)std::min<int64_t>((nTiles + FG_WORKERS - 1) / FG_WORKERS, h->smCount);
	CK(ssc::launch_issue_floor(mode, read_length, n_pairs, h->seed, grid, scratch.p, blobs.p, blobPitch, (uint32_t)fileBytes, s));   // warm-up
	CK(cudaEventRecord(h->evStart, s));
	for (int r = 0; r < reps; r++)
		CK(ssc::launch_issue_floor(mode, read_length, n_pairs, h->seed + 1 + (uint64_t)r, grid, scratch.p, blobs.p, blobPitch, (uint32_t)fileBytes, s));
	CK(cudaEventRecord(h->evStop, s));
	CK(cudaEventSynchronize(h->evStop));
	float ms = 0;
	CK(cudaEventElapsedTime(&ms, h->evStart, h->evStop));
	*ms_per_launch = (double)ms / reps;
	h->stats.launches += (uint64_t)reps + 1;
	return SSC_OK;
}

int ssc_get_stats(ssc_handle* h, ssc_stats* out) {
	if (!h || !out) return fail(SSC_ERR_INVALID, "null argument");
	*out = h->stats;
	return SSC_OK;
}

int ssc_reset_stats(ssc_handle* h) {
	if (!h) return fail(SSC_ERR_INVALID, "null handle");
	memset(&h->stats, 0, sizeof(h->stats));
	return SSC_OK;
}

}  // extern "C"
