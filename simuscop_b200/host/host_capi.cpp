// host_capi.cpp -- C ABI of include/simuscop_host.h and the file sink of the drop-in run.
#include <fcntl.h>
#include <sys/mman.h>
#include <unistd.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <iostream>
#include <string>
#include <cerrno>
#include <condition_variable>
#include <mutex>
#include <thread>
#include <vector>

#include "../../include/simuscop_host.h"
#include "host.h"

struct ssh_job {
	sschost::Job job;
};

// ------------------------------------------------------------------------------------------------
// Output side: SeqWriter's role (lib/seqwriter/SeqWriter.cpp:41-54: append the slab(s) to the FASTQ file(s), both files
// advancing together) at the rate a GPU produces slabs.  The call returns when the slab is in the file (page cache), because
// the pinned slab is reused afterwards.
//
// What bounds it (tools/fs_probe.c on the pool's boxes, profiles/r02w_fs_probe.jsonl): buffered writes to ONE file serialise
// on its inode lock -- 3.6-5.4 GB/s into one file with 1, 4 or 16 threads, against 15-38 GB/s into 4-16 separate files --
// and stores through a shared mapping of the file do not take that lock but pay a page fault per 4 KB (tmpfs 6-7 GB/s per
// file with 4-16 threads, ext4 3-4).  So a slab of ~0.7 GB per file is cut into 8 MB chunks and written from both ends:
//   * one STREAM thread per file pwrite()s the file's chunks front to back (threads 0 and 1 of the pool);
//   * in the modes with mappings the other threads, and a stream thread whose file is finished, copy chunks into a
//     MAP_SHARED mapping of the slab's file range, back to front, in whichever file has more left.
// SIMUSCOP_WRITER_MODE = pwrite (streams only) | mmap (mappings only) | hybrid (both; needs more than two threads).
// A writer on a descriptor the caller opened (ssh_writer_open_fd: standard output, a pipe to an aligner) writes one stream with
// write() from the caller's thread: a pipe has no offsets for pwrite() and no pages to map.
// ------------------------------------------------------------------------------------------------
struct ssh_writer {
	enum Mode { PWRITE = 0, MMAP = 1, HYBRID = 2 };
	static const size_t CH = 8u << 20;
	int fd[2] = {-1, -1};
	uint64_t off[2] = {0, 0};
	bool seq = false;             // ssh_writer_open_fd: sequential write() on fd[0], which the writer does not close
	int nThreads = 1;
	int mode = PWRITE;
	std::vector<std::thread> pool;
	std::mutex mu;
	std::condition_variable cvWork, cvDone;
	// the slab of one file in flight: chunks [front, back) are still to be taken
	struct FileJob { int fd = -1; const char* p = nullptr; size_t len = 0; uint64_t off = 0; char* base = nullptr; size_t front = 0, back = 0; bool seq = false; };
	FileJob job[2];
	size_t inFlight = 0;
	bool stop = false, noMap = false;
	int err = 0;
	// turnstile for several producers (one per GPU) that deliver batches out of order: batch k is written when every
	// batch before it has been
	int64_t turn = 0;
	std::condition_variable cvTurn;
	// ssh_writer_bgzf: every slab is whole BGZF blocks.  Their starts go to a .gzi per stream as the slabs arrive (the layout of
	// htslib's bgzf_index_dump: uint64 count, then (compressed, uncompressed) offset pairs of every block after the first, all
	// little-endian; the count is patched at close), and the EOF block is appended at close
	bool bgzf = false;
	int gzi[2] = {-1, -1};
	uint64_t gziEntries[2] = {0, 0};
	uint64_t blocks[2] = {0, 0};      // data blocks so far
	uint64_t uoff[2] = {0, 0};        // uncompressed bytes so far (the running sum of ISIZE)
	static constexpr uint8_t BGZF_EOF[28] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};

	static int pwrite_all(int fd, const char* p, size_t n, uint64_t off) {
		while (n > 0) {
			ssize_t w = pwrite(fd, p, n, (off_t)off);
			if (w < 0) { if (errno == EINTR) continue; return errno ? errno : EIO; }
			p += w; n -= (size_t)w; off += (uint64_t)w;
		}
		return 0;
	}
	// EPIPE when the reader has gone (the process ignores SIGPIPE): the sink fails and the run ends with SSC_ERR_SINK
	static int write_all(int fd, const char* p, size_t n) {
		while (n > 0) {
			ssize_t w = write(fd, p, n);
			if (w < 0) { if (errno == EINTR) continue; return errno ? errno : EIO; }
			p += w; n -= (size_t)w;
		}
		return 0;
	}
	static int put(const FileJob& j, size_t chunk, bool mapped) {
		const size_t o = chunk * CH, n = std::min(CH, j.len - o);
		if (j.seq) return write_all(j.fd, j.p + o, n);
		if (!mapped) return pwrite_all(j.fd, j.p + o, n, j.off + o);
		char* dst = j.base + o;
#ifdef MADV_POPULATE_WRITE
		// fault the chunk's pages in one call (page-aligned interior) instead of one trap per page
		{
			const uintptr_t a = ((uintptr_t)dst + 4095) & ~(uintptr_t)4095, b = ((uintptr_t)dst + n) & ~(uintptr_t)4095;
			if (b > a) madvise((void*)a, b - a, MADV_POPULATE_WRITE);
		}
#endif
		memcpy(dst, j.p + o, n);
		return 0;
	}
	static void put_le64(std::vector<uint8_t>& v, uint64_t x) { for (int k = 0; k < 8; k++) v.push_back((uint8_t)(x >> (8 * k))); }
	// Walks the BGZF blocks of a slab of stream f that starts at compressed offset off[f]: the index entries of the blocks in *e
	// and the stream's counts after it in *nb / *u.  EINVAL unless the slab is a whole number of well-formed blocks (the header
	// checks of htslib's reader, a BSIZE within the slab, at least the 28 bytes of an empty block, ISIZE <= 64 KiB).
	int walk_bgzf(int f, const char* p, size_t n, std::vector<uint8_t>* e, uint64_t* nb, uint64_t* u) const {
		*nb = blocks[f]; *u = uoff[f];
		uint64_t c = off[f];
		for (size_t at = 0; at < n;) {
			const uint8_t* b = (const uint8_t*)p + at;
			if (n - at < 18 || b[0] != 0x1f || b[1] != 0x8b || b[2] != 8 || !(b[3] & 4) || b[10] != 6 || b[11] != 0 || b[12] != 'B' ||
			    b[13] != 'C' || b[14] != 2 || b[15] != 0)
				return EINVAL;
			const size_t bs = (size_t)(b[16] | b[17] << 8) + 1;
			if (bs < 28 || bs > n - at) return EINVAL;
			const uint32_t isize = b[bs - 4] | b[bs - 3] << 8 | b[bs - 2] << 16 | (uint32_t)b[bs - 1] << 24;
			if (isize > 65536) return EINVAL;
			if (*nb > 0 && gzi[f] >= 0) { put_le64(*e, c); put_le64(*e, *u); }   // block 0 at (0, 0) has no entry
			++*nb; c += bs; *u += isize; at += bs;
		}
		return 0;
	}
	// The index entries of both slabs of a write_slabs call, or EINVAL (and nothing written) if either is not BGZF blocks.
	int index_slabs(const char* const* bufs, const size_t* lens) {
		std::vector<uint8_t> e[2];
		uint64_t nb[2], u[2];
		for (int f = 0; f < 2; f++) {
			const int r = walk_bgzf(f, bufs[f], lens[f], &e[f], &nb[f], &u[f]);
			if (r) return r;
		}
		for (int f = 0; f < 2; f++) {
			if (!e[f].empty()) {
				const int r = pwrite_all(gzi[f], (const char*)e[f].data(), e[f].size(), 8 + gziEntries[f] * 16);
				if (r) return r;
				gziEntries[f] += e[f].size() / 16;
			}
			blocks[f] = nb[f]; uoff[f] = u[f];
		}
		return 0;
	}
	// close: the EOF block behind each stream, and the entry count at the head of each index
	int finish_bgzf() {
		int r = 0;
		for (int f = 0; f < 2 && !r; f++) {
			if (fd[f] < 0) continue;
			r = seq ? write_all(fd[f], (const char*)BGZF_EOF, 28) : pwrite_all(fd[f], (const char*)BGZF_EOF, 28, off[f]);
			if (!r) off[f] += 28;
			if (!r && gzi[f] >= 0) {
				std::vector<uint8_t> cnt;
				put_le64(cnt, gziEntries[f]);
				r = pwrite_all(gzi[f], (const char*)cnt.data(), 8, 0);
			}
		}
		return r;
	}
	bool left() const { return job[0].front < job[0].back || job[1].front < job[1].back; }
	// the next chunk for pool thread `id` (called with mu held): false when there is nothing this thread may take
	bool take(int id, int* file, size_t* chunk, bool* mapped) {
		const bool streams = mode != MMAP;
		if (streams && id < 2 && job[id].front < job[id].back) { *file = id; *chunk = job[id].front++; *mapped = false; return true; }
		// a mapper, or a stream thread without work of its own: the file with more left, from the back
		int f = (job[0].back - job[0].front) >= (job[1].back - job[1].front) ? 0 : 1;
		for (int k = 0; k < 2; k++, f ^= 1) {
			FileJob& j = job[f];
			if (j.front >= j.back) continue;
			if (j.base) { *file = f; *chunk = --j.back; *mapped = true; return true; }
			// not mapped: left to the file's own stream -- or, where there are no streams (mmap mode that could not map), to anybody
			if (!streams) { *file = f; *chunk = j.front++; *mapped = false; return true; }
		}
		return false;
	}
	void worker(int id) {
		std::unique_lock<std::mutex> lk(mu);
		while (true) {
			int f = 0; size_t c = 0; bool mapped = false, got = false;
			cvWork.wait(lk, [&] { return stop || (got = take(id, &f, &c, &mapped)); });
			if (!got) return;                                  // stop
			inFlight++;
			const FileJob j = job[f];
			lk.unlock();
			const int e = put(j, c, mapped);
			lk.lock();
			if (e && !err) err = e;
			inFlight--;
			if (!left() && inFlight == 0) cvDone.notify_all();
		}
	}
	// Both slabs to their files at the running offsets; returns when written.
	int write_slabs(const char* b1, size_t l1, const char* b2, size_t l2) {
		std::unique_lock<std::mutex> lk(mu);
		// a stream that failed once (the reader of the pipe has gone) takes no more bytes; nor does a BGZF stream (its index
		// would no longer match the file)
		if ((seq || bgzf) && err) return err;
		const char* bufs[2] = {b1, b2}; const size_t lens[2] = {l1, fd[1] >= 0 ? l2 : 0};
		if (bgzf) {
			const int e = index_slabs(bufs, lens);
			if (e) { if (!err) err = e; return err; }
		}
		void* maps[2] = {nullptr, nullptr}; size_t mapLen[2] = {0, 0};
		for (int f = 0; f < 2; f++) {
			job[f] = FileJob();
			if (!lens[f]) continue;
			job[f].fd = fd[f]; job[f].p = bufs[f]; job[f].len = lens[f]; job[f].off = off[f]; job[f].seq = seq;
			job[f].back = (lens[f] + CH - 1) / CH;
			const bool wantMap = !pool.empty() && !noMap && (mode == MMAP || (mode == HYBRID && nThreads > 2));
			if (wantMap) {
				const uint64_t a = off[f] & ~(uint64_t)4095;
				if (ftruncate(fd[f], (off_t)(off[f] + lens[f])) == 0) {
					void* m = mmap(nullptr, (size_t)(off[f] + lens[f] - a), PROT_READ | PROT_WRITE, MAP_SHARED, fd[f], (off_t)a);
					if (m != MAP_FAILED) { maps[f] = m; mapLen[f] = (size_t)(off[f] + lens[f] - a); job[f].base = (char*)m + (off[f] - a); }
					else noMap = true;
				} else noMap = true;
			}
			off[f] += lens[f];
		}
		if (!left()) return err;
		if (pool.empty()) {           // single-threaded (and the sequential stream): write here
			for (int f = 0; f < 2; f++) {
				for (size_t c = job[f].front; c < job[f].back; c++) { const int e = put(job[f], c, false); if (e && !err) err = e; }
				job[f] = FileJob();
			}
			return err;
		}
		cvWork.notify_all();
		cvDone.wait(lk, [&] { return !left() && inFlight == 0; });
		for (int f = 0; f < 2; f++) { if (maps[f]) munmap(maps[f], mapLen[f]); job[f] = FileJob(); }
		return err;
	}
};

namespace {

// sink of a single producer: batches arrive in order
int writer_sink(void* user, const char* b1, size_t l1, const char* b2, size_t l2, int64_t, int64_t) {
	return ((ssh_writer*)user)->write_slabs(b1, l1, b2, l2) ? 1 : 0;
}

// sink of one of several producers: `batch` is the global index of the (single) batch this ssc_generate call covers
struct TurnSink { ssh_writer* w; int64_t batch; };
int turn_sink(void* user, const char* b1, size_t l1, const char* b2, size_t l2, int64_t, int64_t) {
	TurnSink* t = (TurnSink*)user;
	ssh_writer* w = t->w;
	{
		std::unique_lock<std::mutex> lk(w->mu);
		w->cvTurn.wait(lk, [&] { return w->turn == t->batch || w->err; });
		if (w->err) return 1;
	}
	const int e = w->write_slabs(b1, l1, b2, l2);
	{
		std::lock_guard<std::mutex> lk(w->mu);
		w->turn = t->batch + 1;
	}
	w->cvTurn.notify_all();
	return e ? 1 : 0;
}

// Read group of sample s in BAM output: its stem, which a BAM read group id takes when it is 1..64 bytes of [!-~].  A longer
// stem (an abundance file with several or long population names) keeps its first bytes and ends in "~<s>", which keeps the ids
// of one run distinct; other bytes become '_'.
std::string bam_read_group(const std::string& stem, int s) {
	std::string id = stem;
	for (char& c : id) if ((unsigned char)c < '!' || (unsigned char)c > '~') c = '_';
	if (id.size() > 64) {
		const std::string tail = "~" + std::to_string(s);
		id = id.substr(0, 64 - tail.size()) + tail;
	}
	return id.empty() ? "sample~" + std::to_string(s) : id;
}

// SIMUSCOP_TRUTH_VCF=1: <output>/<stem>.truth.vcf of sample s, written once the sample is prepared
int write_truth(sschost::Job& J, int s) {
	const char* t = getenv("SIMUSCOP_TRUTH_VCF");
	if (!t || atoi(t) == 0) return 0;
	const std::string path = J.cfg.str["output"] + "/" + J.samples[s].stem + ".truth.vcf";
	if (J.write_truth_vcf(s, path)) { std::cerr << "Error: can not write the truth VCF " << path << std::endl; return SSC_ERR_SINK; }
	return 0;
}

}  // namespace

extern "C" {

int ssh_open(const char* config_path, uint64_t seed, ssh_job** out) {
	if (!config_path || !out) return SSC_ERR_INVALID;
	ssh_job* j = new ssh_job();
	j->job.seed = seed;
	j->job.open(config_path);
	*out = j;
	return SSC_OK;
}

int ssh_close(ssh_job* job) { delete job; return SSC_OK; }
int ssh_num_samples(ssh_job* job) { return (int)job->job.samples.size(); }
const char* ssh_sample_stem(ssh_job* job, int s) { return job->job.samples.at(s).stem.c_str(); }
int ssh_paired(ssh_job* job) { return job->job.cfg.paired() ? 1 : 0; }
int ssh_read_length(ssh_job* job) { return job->job.prof.RL; }
const char* ssh_output_dir(ssh_job* job) { return job->job.cfg.str["output"].c_str(); }

int ssh_prepare_sample(ssh_job* job, int s, ssc_handle* dev, const char* dump_path, int64_t* planned, int64_t* emitted) {
	if (!job || s < 0 || s >= (int)job->job.samples.size()) return SSC_ERR_INVALID;
	return job->job.prepare_sample(s, dev, dump_path ? dump_path : "", planned, emitted);
}

int ssh_write_truth_vcf(ssh_job* job, int s, const char* path) {
	if (!job || !path || s < 0 || s >= (int)job->job.samples.size()) return SSC_ERR_INVALID;
	if (s != job->job.lastPrepared) return SSC_ERR_STATE;
	return job->job.write_truth_vcf(s, path);
}

int ssh_selftest_splices(ssh_job* job, int64_t* segments_checked, int64_t* with_indels) {
	// Host-only check of the splice-list construction the device path uses for segments with insertion / deletion variants
	// (Job::segment_splices + the substitution mapping of Job::device_weights) against the string construction
	// (Job::build_haplotypes, which the CPU suite pins against the instrumented reference): every haplotype of every segment
	// of every population, materialised from its splice list, must equal the string.  Returns the number of mismatches.
	if (!job) return -1;
	sschost::Job& J = job->job;
	J.begin_plan();
	const int ploidy = J.cfg.num["ploidy"];
	int64_t bad = 0, checked = 0, indel = 0;
	for (auto& popu : J.cfg.popu)
		for (auto& chr : J.chroms) {
			const std::string& chrSeq = J.fasta.chromosome(chr);
			for (auto& seg : J.segs[popu][chr]) {
				std::vector<std::string> want;
				J.build_haplotypes(seg, popu, want);
				const size_t refOff = (size_t)(seg.start - 1);
				const size_t refLen = std::min((size_t)seg.refSize(), chrSeq.size() > refOff ? chrSeq.size() - refOff : 0);
				if (refLen == 0) continue;
				std::vector<int> reps; std::vector<sschost::Poke> pokes;
				J.segment_copies_and_pokes(seg, popu, reps, pokes);
				std::vector<std::vector<sschost::Piece>> ropes;
				J.segment_splices(seg, popu, refLen, reps, ropes);
				if (!J.segment_is_copy_only(seg, popu)) indel++;
				for (int h = 0; h < ploidy; h++) {
					std::string got;
					std::vector<std::pair<size_t, char>> pk;
					for (const sschost::Piece& p : ropes[h]) {
						if (p.copy >= 0) {
							for (const sschost::Poke& q : pokes) if (q.hap == h && q.off >= p.a && q.off < p.b) pk.push_back({got.size() + (size_t)(q.off - p.a), q.c});
							got.append(chrSeq, refOff + (size_t)p.a, (size_t)(p.b - p.a));
						} else got += p.lit;
					}
					for (auto& q : pk) got[q.first] = (char)toupper((unsigned char)q.second);
					checked++;
					if (got != want[h]) bad++;
				}
			}
		}
	if (segments_checked) *segments_checked = checked;
	if (with_indels) *with_indels = indel;
	return (int)bad;
}

int ssh_writer_open(const char* path1, const char* path2, int threads, ssh_writer** out) {
	if (!path1 || !out) return SSC_ERR_INVALID;
	ssh_writer* w = new ssh_writer();
	w->fd[0] = open(path1, O_WRONLY | O_CREAT | O_TRUNC, 0644);
	if (path2 && path2[0]) w->fd[1] = open(path2, O_WRONLY | O_CREAT | O_TRUNC, 0644);
	if (w->fd[0] < 0 || (path2 && path2[0] && w->fd[1] < 0)) {
		if (w->fd[0] >= 0) close(w->fd[0]);
		if (w->fd[1] >= 0) close(w->fd[1]);
		delete w;
		return SSC_ERR_SINK;
	}
	w->nThreads = threads < 1 ? 1 : (threads > 64 ? 64 : threads);
	if (const char* m = getenv("SIMUSCOP_WRITER_MODE"))
		w->mode = strcmp(m, "mmap") == 0 ? ssh_writer::MMAP : (strcmp(m, "hybrid") == 0 ? ssh_writer::HYBRID : ssh_writer::PWRITE);
	if (w->mode == ssh_writer::PWRITE && w->nThreads > 2) w->nThreads = 2;   // one stream per file: more threads would only queue on the inode locks
	if (w->nThreads > 1) for (int i = 0; i < w->nThreads; i++) w->pool.emplace_back([w, i] { w->worker(i); });
	*out = w;
	return SSC_OK;
}

int ssh_writer_open_fd(int fd, ssh_writer** out) {
	if (fd < 0 || !out) return SSC_ERR_INVALID;
	ssh_writer* w = new ssh_writer();
	w->fd[0] = fd;
	w->seq = true;
	*out = w;
	return SSC_OK;
}

int ssh_writer_bgzf(ssh_writer* w, const char* index1, const char* index2) {
	if (!w) return SSC_ERR_INVALID;
	if (w->bgzf || w->off[0] || w->off[1]) return SSC_ERR_STATE;
	if (index2 && w->fd[1] < 0) return SSC_ERR_INVALID;
	const char* idx[2] = {index1, index2};
	for (int f = 0; f < 2; f++) {
		if (!idx[f]) continue;
		const uint8_t zero[8] = {0, 0, 0, 0, 0, 0, 0, 0};         // the entry count, patched at close
		w->gzi[f] = open(idx[f], O_WRONLY | O_CREAT | O_TRUNC, 0644);
		if (w->gzi[f] < 0 || ssh_writer::pwrite_all(w->gzi[f], (const char*)zero, 8, 0)) {
			for (int k = 0; k <= f; k++) if (w->gzi[k] >= 0) { close(w->gzi[k]); w->gzi[k] = -1; }
			return SSC_ERR_SINK;
		}
	}
	w->bgzf = true;
	return SSC_OK;
}

ssc_sink_fn ssh_writer_sink(void) { return writer_sink; }

int ssh_writer_close(ssh_writer* w, uint64_t* bytes1, uint64_t* bytes2) {
	if (!w) return SSC_OK;
	{
		std::lock_guard<std::mutex> lk(w->mu);
		w->stop = true;
	}
	w->cvWork.notify_all();
	for (auto& t : w->pool) t.join();
	// a BGZF stream that failed gets no EOF block: a reader then sees it is truncated
	if (w->bgzf && !w->err) w->err = w->finish_bgzf();
	int rc = w->err ? SSC_ERR_SINK : SSC_OK;
	for (int f = 0; f < 2; f++) if (w->gzi[f] >= 0 && close(w->gzi[f]) != 0) rc = SSC_ERR_SINK;
	if (!w->seq)
		for (int f = 0; f < 2; f++) if (w->fd[f] >= 0 && close(w->fd[f]) != 0) rc = SSC_ERR_SINK;
	if (bytes1) *bytes1 = w->off[0];
	if (bytes2) *bytes2 = w->off[1];
	delete w;
	return rc;
}

int ssh_run(ssh_job* job, int device) {
	if (getenv("SIMUSCOP_PLAN_ONLY")) {
		// host logic only (no GPU): write the SSCPLAN1 dumps of every sample and stop
		const char* prefix = getenv("SIMUSCOP_DUMP_PLAN");
		if (!prefix) { std::cerr << "Error: SIMUSCOP_PLAN_ONLY needs SIMUSCOP_DUMP_PLAN" << std::endl; return 1; }
		for (int s = 0; s < (int)job->job.samples.size(); s++) {
			int64_t a, b;
			int r = job->job.prepare_sample(s, nullptr, std::string(prefix) == "none" ? std::string() : std::string(prefix) + "." + std::to_string(s) + ".plan", &a, &b);
			if (r) return r;
			r = write_truth(job->job, s);
			if (r) return r;
		}
		return 0;
	}
	// devices: SIMUSCOP_DEVICES="0,1,2,..." shards every sample by pair-ID range over the listed GPUs
	std::vector<int> devIds;
	if (const char* dl = getenv("SIMUSCOP_DEVICES")) {
		for (const std::string& t : sschost::split(dl, ',')) if (!sschost::trim(t).empty()) devIds.push_back(atoi(t.c_str()));
	}
	if (devIds.empty()) devIds.push_back(device);
	sschost::Job& J = job->job;
	// SIMUSCOP_STDOUT=1: the reads of the one sample go to standard output (PE interleaved) and no FASTQ file is written;
	// SIMUSCOP_INTERLEAVE=1: a PE sample is written to <output>/<stem>.fq[.gz], mate 1 and mate 2 of each pair in turn;
	// SIMUSCOP_BAM=1: every sample, PE or SE, is written as unaligned BAM to <output>/<stem>.bam, read group = the stem (see
	// bam_read_group; takes
	// precedence over SIMUSCOP_GZIP, SIMUSCOP_BGZF and SIMUSCOP_INTERLEAVE)
	const char* soEnv = getenv("SIMUSCOP_STDOUT");
	const bool toStdout = soEnv && atoi(soEnv) != 0;
	const char* bamEnv = getenv("SIMUSCOP_BAM");
	const bool bam = bamEnv && atoi(bamEnv) != 0;
	const char* ilEnv = getenv("SIMUSCOP_INTERLEAVE");
	const bool interleave = !bam && J.cfg.paired() && (toStdout || (ilEnv && atoi(ilEnv) != 0));
	if (toStdout && J.samples.size() > 1) {
		std::cerr << "Error: SIMUSCOP_STDOUT=1 writes one sample, this configuration yields " << J.samples.size()
		          << " (one per row of the abundance file); write them to files instead" << std::endl;
		return 1;
	}
	std::vector<ssc_handle*> devs;
	int rc = 0;
	for (int id : devIds) {
		ssc_handle* h = nullptr;
		rc = ssc_create(id, &h);
		if (rc) { std::cerr << "Error: " << ssc_last_error() << std::endl; for (auto* d : devs) ssc_destroy(d); return rc; }
		devs.push_back(h);
	}
	const char* dumpPrefix = getenv("SIMUSCOP_DUMP_PLAN");
	if (const char* bp = getenv("SIMUSCOP_BATCH_PAIRS")) for (auto* d : devs) ssc_set_option(d, "batch_pairs", atoll(bp));
	// SIMUSCOP_GZIP=1: the same FASTQ, compressed on the GPU, written as <name>.fq.gz (concatenated gzip members)
	// SIMUSCOP_BGZF=1: the same, each member a BGZF block, the file ended by the BGZF EOF block, and <name>.fq.gz.gzi beside it
	// (the block index `bgzip -i` writes; none on standard output); implies SIMUSCOP_GZIP=1
	const char* gzEnv = getenv("SIMUSCOP_GZIP");
	const char* bgzfEnv = getenv("SIMUSCOP_BGZF");
	const bool bgzf = !bam && bgzfEnv && atoi(bgzfEnv) != 0;
	const bool gz = !bam && (bgzf || (gzEnv && atoi(gzEnv) != 0));
	if (bam) for (auto* d : devs) ssc_set_option(d, "bam", 1);
	if (gz) for (auto* d : devs) ssc_set_option(d, "gzip", 1);
	if (bgzf) for (auto* d : devs) ssc_set_option(d, "bgzf", 1);
	if (interleave) for (auto* d : devs) ssc_set_option(d, "interleave", 1);
	const int G = (int)devs.size();
	for (int s = 0; s < (int)J.samples.size() && !rc; s++) {
		const std::string prefix = J.cfg.str["output"] + "/" + J.samples[s].stem;
		const bool paired = J.cfg.paired();
		const std::string ext = bam ? ".bam" : gz ? ".fq.gz" : ".fq";
		const bool twoFiles = paired && !interleave && !bam;
		const std::string f1 = toStdout ? "<standard output>" : (twoFiles ? prefix + "_1" + ext : prefix + ext);
		const std::string f2 = twoFiles ? prefix + "_2" + ext : "";
		std::string dump;
		if (dumpPrefix) dump = std::string(dumpPrefix) + "." + std::to_string(s) + ".plan";
		int64_t planned = 0, emitted = 0;
		rc = J.prepare_sample_multi(s, devs, dump, &planned, &emitted);
		if (rc) { std::cerr << "Error: " << ssc_last_error() << std::endl; break; }
		rc = write_truth(J, s);
		if (rc) break;
		const std::string rg = bam_read_group(J.samples[s].stem, s);
		if (bam) {
			for (auto* d : devs)
				if ((rc = ssc_set_read_group(d, rg.c_str()))) break;
			// the read names are checked before the output is opened: an empty range runs the check and generates nothing
			if (!rc) rc = ssc_generate(devs[0], 0, 0, [](void*, const char*, size_t, const char*, size_t, int64_t, int64_t) { return 0; }, nullptr);
		}
		if (rc) { std::cerr << "Error: " << ssc_last_error() << std::endl; break; }
		// one ordered writer per sample.  One GPU: a single ssc_generate call over the whole job (the library pipelines kernel,
		// device->host copy and sink).  Several GPUs: the job is cut into batches, batch k goes to GPU k mod G, and every
		// finished slab waits at the writer's turnstile until all earlier batches are in the file -- one pass of I/O, no part
		// files, output identical to the single-GPU run.
		ssh_writer* w = nullptr;
		int wthreads = 4;
		if (const char* wt = getenv("SIMUSCOP_WRITER_THREADS")) wthreads = atoi(wt);
		if (toStdout ? ssh_writer_open_fd(1, &w) : ssh_writer_open(f1.c_str(), twoFiles ? f2.c_str() : nullptr, wthreads, &w))
			sschost::die(-1, "Error: can not open fastq file to save results:\n" + f1);
		if (bgzf) {
			const std::string i1 = f1 + ".gzi", i2 = f2 + ".gzi";
			if (ssh_writer_bgzf(w, toStdout ? nullptr : i1.c_str(), twoFiles ? i2.c_str() : nullptr))
				sschost::die(-1, "Error: can not open the BGZF index file of:\n" + f1);
		}
		if (bam) {
			// BGZF blocks without an index (unaligned records have no coordinates), the header block in front of turn 0
			uint8_t hdr[512];
			const int64_t n = ssc_bam_header(rg.c_str(), hdr, sizeof(hdr));
			if (n <= 0 || ssh_writer_bgzf(w, nullptr, nullptr) || w->write_slabs((const char*)hdr, (size_t)n, nullptr, 0)) {
				std::cerr << "Error: writing the BAM header of " << f1 << " failed" << std::endl;
				ssh_writer_close(w, nullptr, nullptr);
				rc = SSC_ERR_SINK;
				break;
			}
		}
		if (G == 1) {
			rc = ssc_generate(devs[0], 0, planned, writer_sink, w);
			if (rc) std::cerr << "Error: " << ssc_last_error() << std::endl;
		} else {
			int64_t bp = 1 << 20;
			if (const char* bpe = getenv("SIMUSCOP_BATCH_PAIRS")) bp = std::max<int64_t>(32, atoll(bpe));
			const int64_t nBatches = (planned + bp - 1) / bp;
			std::vector<int> rcs(G, 0);
			std::vector<std::string> errs(G);
			auto work = [&](int g) {
				for (int64_t k = g; k < nBatches; k += G) {
					TurnSink ts{w, k};
					// a batch without emitted pairs never reaches the sink: pass its turn on here
					bool called = false;
					struct Ctx { TurnSink* ts; bool* called; } ctx{&ts, &called};
					auto thunk = [](void* u, const char* b1, size_t l1, const char* b2, size_t l2, int64_t a, int64_t n) -> int {
						Ctx* c = (Ctx*)u; *c->called = true; return turn_sink(c->ts, b1, l1, b2, l2, a, n);
					};
					rcs[g] = ssc_generate(devs[g], k * bp, std::min(planned, (k + 1) * bp), thunk, &ctx);
					if (rcs[g]) { errs[g] = ssc_last_error(); std::lock_guard<std::mutex> lk(w->mu); if (!w->err) w->err = EIO; w->cvTurn.notify_all(); return; }
					if (!called) {
						std::unique_lock<std::mutex> lk(w->mu);
						w->cvTurn.wait(lk, [&] { return w->turn == k || w->err; });
						w->turn = k + 1;
						lk.unlock();
						w->cvTurn.notify_all();
					}
				}
			};
			std::vector<std::thread> th;
			for (int g = 1; g < G; g++) th.emplace_back(work, g);
			work(0);
			for (auto& t : th) t.join();
			for (int g = 0; g < G; g++) if (rcs[g]) { std::cerr << "Error: " << errs[g] << std::endl; rc = rcs[g]; }
		}
		if (ssh_writer_close(w, nullptr, nullptr) && !rc) { std::cerr << "Error: writing " << f1 << " failed" << std::endl; rc = SSC_ERR_SINK; }
	}
	for (auto* d : devs) ssc_destroy(d);
	return rc;
}

}  // extern "C"
