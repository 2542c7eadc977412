/*
 * simuscop.h -- C ABI of the B200 read-generation hot path (libsimuscop_cuda.so).
 *
 * This is the drop-in boundary for the per-read loop of SimuSCoP's `simuReads`.
 * The reference has no FFI for this path; it enters it through a C function
 * pointer and process-wide singletons:
 *
 *   threadPool->pool_add_work(&Segment::yieldReads, &chrSegs[k], n++)
 *                                     reference lib/genome/Genome.cpp:881, :949
 *   void* Segment::yieldReads(const void* seg)      lib/segment/Segment.cpp:673-871
 *   char* Profile::predict(char* refSeq, int isRead1)  lib/profile/Profile.cpp:1586-1701
 *   int   Profile::yieldInsertSize()                lib/profile/Profile.cpp:1486-1493
 *   swp->write(char*[, char*])                      lib/seqwriter/SeqWriter.cpp:41-54
 *
 * The entry points below are what a maintainer binds where Genome::yieldReads
 * dispatched segments to the thread pool (INTEGRATION.md shows the stub).
 * Conventions: plain pointers and sizes only; every function returns SSC_OK (0)
 * or an SSC_ERR_* code and records a message readable with ssc_last_error();
 * no exception crosses the boundary; host pointers are borrowed for the duration
 * of the call only; one handle per GPU; a handle is not thread-safe, distinct
 * handles may be used from distinct host threads.  There is no CPU fallback:
 * without a CUDA device ssc_create() fails.
 */
#ifndef SIMUSCOP_H
#define SIMUSCOP_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SSC_OK            0
#define SSC_ERR_INVALID   1   /* bad argument / unsupported configuration */
#define SSC_ERR_CUDA      2   /* CUDA runtime error */
#define SSC_ERR_STATE     3   /* call order violated (e.g. generate before set_plan) */
#define SSC_ERR_NOMEM     4
#define SSC_ERR_SINK      5   /* the sink callback returned non-zero */
#define SSC_ERR_OVERFLOW  6   /* a read outgrew the per-read scratch (see DESIGN.md, limits) */

typedef struct ssc_handle ssc_handle;

/*
 * Profile tables -- the FP64 CDFs exactly as the reference builds them
 * (Profile::load -> normParas(true) -> initCDFs, lib/profile/Profile.cpp:934-1434;
 * Matrix::normalize/cumsum, lib/matrix/Matrix.h:482-522).  Row-major:
 *   subs_cdf1/2 [n_kmer_rows][bins][n_bases]      (Profile::subsCdf1/2)
 *   quality_cdf [n_bases*n_bases][bins][n_qual]   (Profile::qualityCdf)
 *   isize_cdf   [n_isize]  value k <-> insert size min_insert_size+k (Profile::iSizeCdf)
 *   ins_cdf/del_cdf [n_ins]/[n_del]               (Profile::insCdf/delCdf)
 * n_isize == 0 means "no insert-size table": every fragment uses fixed_insert_size
 * (Profile::yieldInsertSize, Profile.cpp:1487-1489).  use_cdf2 == 0 means read 2
 * uses subs_cdf1 (Profile::getSubBaseIndx2, Profile.cpp:1546-1549).
 */
typedef struct ssc_profile_tables {
	int32_t n_bases;            /* N, must be 4 */
	int32_t kmer;               /* K */
	int32_t bins;               /* B */
	int32_t n_qual;             /* Q = 94 */
	int32_t min_qual;           /* 33 */
	int32_t read_length;        /* RL */
	int32_t paired;             /* layout == "PE" */
	int32_t use_cdf2;
	int32_t fixed_insert_size;  /* config insertSize */
	int32_t min_insert_size;
	int32_t n_isize;
	int32_t n_ins;
	int32_t n_del;
	int32_t n_kmer_rows;        /* sum_{p=1..K} N^p */
	double insert_rate;
	double del_rate;
	char bases[8];              /* e.g. "ACTG", NUL padded */
	const double* isize_cdf;
	const double* ins_cdf;
	const double* del_cdf;
	const double* subs_cdf1;
	const double* subs_cdf2;
	const double* quality_cdf;
} ssc_profile_tables;

/*
 * One sampling bin of the read plan (Segment::fragStartPos/fragEndPos/hapIndxs/fragRCs,
 * lib/segment/Segment.h:44-48), flattened so that the device needs no segment objects.
 * Bins are given in the reference's threads=1 emission order
 * (population -> chromosome -> segment -> bin); bins of one segment are contiguous.
 */
typedef struct ssc_bin {
	int64_t hap_base;     /* index in the haplotype store of the first base of this
	                         segment's haplotype string (segSequences[hap]) */
	int64_t contig_end;   /* one past the last base of the (population, chromosome,
	                         haplotype index) contig: the concatenation of the same-index
	                         haplotype strings of the chromosome's segments, which is what
	                         Segment::getFragSequence + Genome::produceFragment walk
	                         (Segment.cpp:1077-1103, Genome.cpp:599-632) */
	int32_t spos, epos;   /* start position is drawn in [spos, epos] */
	uint32_t segsize;     /* seqSize/CN, the modulus of the position in read names */
	int32_t read_count;   /* fragRCs[i] */
	int32_t segment;      /* index into the segment array */
	int32_t reserved;
} ssc_bin;

typedef struct ssc_segment {
	int64_t first_bin;
	int64_t n_bins;
	int32_t name_offset;  /* "@<popu>#<chr>#" inside the name blob (Segment.cpp:780,809,824) */
	int32_t name_len;     /* 1..64 bytes, the first one '@'; the blob is < 2^17 bytes */
} ssc_segment;

typedef struct ssc_stats {
	double   device_ms;        /* sum of CUDA-event durations of the generation kernels */
	uint64_t launches;         /* kernels launched by this handle since creation */
	uint64_t gen_launches;     /* launches of the fused generation kernel */
	uint64_t pairs_emitted;
	uint64_t reads_emitted;
	uint64_t bases_emitted;    /* sum of emitted read lengths */
	uint64_t fastq_bytes;      /* bytes of FASTQ written to HBM ("bam": bytes of the BAM records before compression) */
	uint64_t hap_bytes;        /* algorithmic haplotype bytes read: ceil(len/4)+ceil(len/8) per fragment */
	uint64_t d2h_bytes;
	uint64_t h2d_bytes;
	double   gen_kernel_ms;    /* CUDA-event time of the generation kernel alone (ssc_generate_device) */
	double   compact_kernel_ms;/* CUDA-event time of the compaction kernel alone (ssc_generate_device) */
	uint64_t timed_batches;    /* launches covered by gen_kernel_ms */
	uint64_t gz_bytes;         /* gzip mode: compressed bytes written to the slabs, BGZF blocks with "bgzf" or "bam" (fastq_bytes stays the plain size) */
	uint64_t bin_bytes;        /* algorithmic bin-record bytes read: 64 bytes per distinct bin of every generated batch */
	double   mover_kernel_ms;  /* CUDA-event time of the concurrent blob mover (concurrent_move > 0) on its own stream, under the
	                              generation kernel of the next batch (ssc_generate_device) */
	/* the generation kernel of the most recent launch (0 before the first): */
	int32_t  gen_kernel;       /* 1 = fast kernel (K = 3, RL 33..160), 2 = generic kernel with the K = 3 substitution tables in
	                              shared memory, 3 = generic kernel with the tables in global memory, 4 = FP64 linear search */
	int32_t  gen_nch;          /* chunks of 32 cycles of the instance: 2..5 for the fast kernel, 10 for the generic kernels */
	int32_t  gen_qmode;        /* fast kernel: where the quality tables live (8 / 16 / 2 / 0, see "fast_qmode"); -1 otherwise */
	int32_t  gen_smem_bytes;   /* dynamic shared memory of the launch */
} ssc_stats;

/*
 * Sink for finished FASTQ slabs, called in pair order.  buf1/buf2 point to pinned host
 * memory owned by the handle and valid only during the call (SeqWriter::write(char*,char*)
 * semantics, SeqWriter.cpp:49-54: the callee copies or writes synchronously).  In SE
 * layout buf2 == NULL and len2 == 0.  With the "interleave" option a PE plan follows the SE
 * contract too: buf1/len1 hold pair i mate 1, pair i mate 2, ... in pair order, and
 * buf2 == NULL, len2 == 0.  Return 0 to continue.
 */
typedef int (*ssc_sink_fn)(void* user, const char* buf1, size_t len1, const char* buf2, size_t len2,
                           int64_t first_pair, int64_t n_pairs);

const char* ssc_last_error(void);
int ssc_version(void);

int ssc_create(int device, ssc_handle** out);
int ssc_destroy(ssc_handle* h);

/* "batch_pairs" (pairs per kernel launch), "fp64_search" (0/1: use the FP64 linear-search
 * ground-truth kernel instead of the integer-threshold kernel), "force_generic" (0/1), "gzip" (0/1: the slabs
 * handed to the sink hold concatenated gzip members -- a valid .gz stream of the same FASTQ bytes -- compressed on
 * the GPU, one member per 32 pairs, Huffman-coded with a table fitted to the first batch, or stored where that code would
 * expand the member past its bytes + 23, so gzip mode fails only where plain output does, with every kernel and profile; the plain bytes of
 * SeqWriter::write are the default), "bgzf" (0/1, default 0; no effect without gzip: every gzip member is written as a BGZF
 * block -- FLG = FEXTRA and the 8 bytes 06 00 'B' 'C' 02 00 BSIZE(2, = block length - 1) after the 10-byte header, the
 * DEFLATE data unchanged, a stored block raw + 31 bytes -- so bgzip, samtools and other htslib readers can decompress in
 * parallel and seek.  A block holds the records of 32 pairs (interleaved: of both mates), at most 32 x the plan's worst-case
 * record (header + 2 x (read length + 96) + 4 bytes; both mates interleaved) + 31 bytes: 39 199 up to read length 160, 59 167
 * at read length 320 with 64-byte names, interleaved; in PE output
 * block k of file 1 and block k of file 2 hold the same pairs.  The slabs and ssc_generate_device hold whole blocks, gz_bytes
 * counts them.  The library does not write the 28-byte BGZF end-of-file block, since it cannot know which call is the last:
 * the writer appends 1f 8b 08 04 00 00 00 00 00 ff 06 00 42 43 02 00 1b 00 03 00 00 00 00 00 00 00 00 00 (ssh_writer_bgzf
 * does it).  Like gzip it may be set between calls and takes effect at the next one), "interleave" (0/1: a PE plan writes ONE stream, pair i mate 1 then pair i mate 2 in pair
 * order, byte for byte the interleave of the _1 / _2 records without the option, "/1" and "/2" suffixes included -- what
 * `bwa mem -p` and `bowtie2 --interleaved` read; the sink gets it as buf1/len1 with buf2 == NULL, len2 == 0,
 * ssc_generate_device returns it in *bytes1 with *bytes2 = 0, ssc_stats counts the same fastq_bytes / gz_bytes totals; with
 * gzip, one member per 32 pairs of both mates; no effect on SE plans and on ssc_generate_reads; like gzip it may be set
 * between calls and takes effect at the next one), "bam" (0/1, default 0: the slabs hold BGZF blocks of unaligned BAM records
 * (SAM specification v1, section 4.2) instead of FASTQ, whatever "gzip", "bgzf" and "interleave" say.  Each read is one record:
 * refID, pos, next_refID, next_pos -1, mapq 0, bin 4680, no CIGAR, tlen 0, flag 77 / 141 for PE mate 1 / 2 and 4 for SE (0x10 is
 * never set: a read is stored as its FASTQ record has it), read_name = the FASTQ name without '@' and without "/1" or "/2"
 * (both mates of a pair have the same name), l_seq = the read's length, the FASTQ bases as 4-bit codes (first base in the
 * high nibble, a zero pad nibble behind an odd-length read), the FASTQ qualities - 33, and RG:Z:<id> when
 * ssc_set_read_group has set an id.  The records are those of the interleaved FASTQ of the same range, in the same order; a
 * PE plan writes ONE stream (buf1/len1 of the sink, *bytes1 of ssc_generate_device), mate 1 and mate 2 of each pair in turn.
 * A block holds the records of 32 pairs (both mates), at most 32 x 2 x (36 + name + 21 + (RL + 97) / 2 + RL + 96 + 68) + 31
 * bytes.  The Huffman table is fitted to the first batch of BAM records, and fitted anew at the next call whenever the option
 * changes.  gz_bytes counts the BGZF bytes, fastq_bytes the BAM record bytes.  A plan whose segment names hold, after the
 * '@', a byte outside the SAM QNAME characters [!-?A-~] is refused with SSC_ERR_INVALID before anything is generated (the
 * message names the segment and the byte), also for an empty pair range, so that a caller can check a plan that way before
 * it opens its output; the handle stays usable.  The library writes neither the BAM header
 * (ssc_bam_header) nor the BGZF end-of-file block: the caller's writer does (ssh_writer_bgzf appends the EOF block).  No
 * effect on ssc_generate_reads; may be set between calls and takes effect at the next one), "concurrent_move" (n > 0: the blobs of batch k are moved by a
 * bulk-copy kernel on n SMs, on a second stream, while the generation kernel of batch k+1 runs on the others; default 9 of
 * 148 SMs, 0 below 64 SMs; 0, or n at least the GPU's SM count: a stand-alone kernel after every batch), "max_ctas" (> 0 caps the grid of the generation
 * kernel; 0 = one CTA per SM), "no_splice" (0/1, tests: reads with indel events take the position-by-position path
 * of the fast kernel instead of the spliced packed read), "fast_qmode" (tests; set before ssc_set_profile: -1 = automatic,
 * the default; 8 / 16 / 2 / 0 = the fast kernel may only keep its quality tables that way: 8 = every row in shared memory
 * as 32-bit thresholds (5..8 live symbols per row), 16 = every row as 16-bit keys with an exact repeat on ties (<= 40 live
 * symbols), 2 = only the ref == call rows in shared memory, 0 = all in global memory.  A mode that does not apply or does
 * not fit the shared memory leaves the profile to the generic kernel; ssc_stats shows what ran). */
int ssc_set_option(ssc_handle* h, const char* key, int64_t value);

/* Read group of the "bam" output: every record then ends in the tag RG:Z:<id>.  id: 1..64 bytes of [!-~]; NULL or "" removes
 * the tag (the default).  Anything else is refused with SSC_ERR_INVALID.  May be set between calls. */
int ssc_set_read_group(ssc_handle* h, const char* id);

/* Host-only (no GPU, no handle): the header of a BAM stream as one stored BGZF block -- "BAM\1", l_text and the text
 * "@HD\tVN:1.6\tSO:unsorted\tGO:query\n", plus "@RG\tID:<id>\tSM:<id>\n" when read_group is neither NULL nor "", and
 * n_ref = 0 -- written to out.  A BAM file of the "bam" option is this block, the handles' blocks, then the BGZF EOF block.
 * Returns the block size, 0 when it does not fit `cap`, or -1 on a bad read group (see ssc_set_read_group). */
int64_t ssc_bam_header(const char* read_group, uint8_t* out, size_t cap);

int ssc_set_profile(ssc_handle* h, const ssc_profile_tables* t);

/* Haplotype store: 2-bit codes (in the profile's `bases` order) + 1-bit non-ACGT mask,
 * packed on the device from ASCII (any case; every non-ACGT character behaves as N).
 * Append the haplotype strings contig by contig; *first_base receives the store index of
 * the first appended base.  ssc_genome_reserve refuses (SSC_ERR_INVALID, before allocating) a store of more than
 * 2^36 - 32 bases: the fast kernel addresses a read's window by a 32-bit index of 16-base words. */
int ssc_genome_reserve(ssc_handle* h, uint64_t total_bases);
int ssc_genome_append(ssc_handle* h, const char* ascii, uint64_t n, uint64_t* first_base);
int ssc_genome_size(ssc_handle* h, uint64_t* n_bases);

/* Reference-relative construction of haplotype strings on the device (the copy-and-substitute part of
 * Segment::generateSegSequences, lib/segment/Segment.cpp:124-311: a haplotype of a segment without indel variants is
 * the reference slice repeated once per copy, with SNP / SNV alleles poked in).  The chromosome is uploaded once
 * (ssc_reference_upload, any case, ASCII); ssc_genome_append_ref appends `reps` copies of reference bases
 * [ref_off, ref_off+len) to the store exactly as ssc_genome_append would append that string; ssc_genome_poke then
 * overwrites single bases (store indices, distinct) with the given characters.  ssc_genome_read decodes store bases
 * back to upper-case ASCII (non-ACGT -> 'N'), a diagnostic for tests. */
int ssc_reference_upload(ssc_handle* h, const char* ascii, uint64_t n);
/* The same from the FASTA file itself (FastaReference::getSequence, lib/fastahack/Fasta.cpp:304-334, and the upper-casing
 * of Genome::getSubSequence done on the device): the sequence lines of one record are read from `fd` (raw_len bytes at
 * file_offset, straight into pinned staging buffers) and unfolded on the GPU with the geometry of the record's .fai entry
 * (n_bases bases, line_bases bases per line in line_width bytes).  *n_other receives the number of characters that are
 * neither ACGT nor N in either case (IUPAC codes). */
int ssc_reference_upload_fasta(ssc_handle* h, int fd, uint64_t file_offset, uint64_t raw_len, uint64_t n_bases,
                               uint32_t line_bases, uint32_t line_width, uint64_t* n_other);
/* The same in the background: ssc_reference_prefetch_fasta starts reading and unfolding a record into a second set of
 * buffers (own thread, own stream) and returns; the caller goes on working with the current reference (ssc_genome_append_ref,
 * ssc_gc_census, host work) and later calls ssc_reference_adopt_prefetched, which waits for the record and makes it the
 * current reference.  One record may be in flight. */
int ssc_reference_prefetch_fasta(ssc_handle* h, int fd, uint64_t file_offset, uint64_t raw_len, uint64_t n_bases,
                                 uint32_t line_bases, uint32_t line_width);
int ssc_reference_adopt_prefetched(ssc_handle* h, uint64_t* n_other);
int ssc_genome_append_ref(ssc_handle* h, uint64_t ref_off, uint64_t len, int32_t reps, uint64_t* first_base);
int ssc_genome_poke(ssc_handle* h, const int64_t* store_pos, const char* chars, int64_t n);
int ssc_genome_read(ssc_handle* h, uint64_t start, uint64_t n, char* out);

/* GC census of haplotype-store intervals: the device half of the GC-weighted read plan
 * (Segment::getWeightedLength, lib/segment/Segment.cpp:567-624, which calls calculateGCPercent,
 * lib/mydefine/MyDefine.cpp:279-303, once per 1 kb window / capture target).  For interval i =
 * store bases [starts[i], starts[i]+lens[i]) (lens[i] >= 0, inside the appended store) it returns
 * gc[i] = number of G or C bases and nn[i] = number of non-ACGT bases; the caller forms the
 * reference's integer percentage (nn > 0 ? -1 : 100*gc/len).  Host arrays, copied inside. */
int ssc_gc_census(ssc_handle* h, const int64_t* starts, const int32_t* lens, int64_t n,
                  int32_t* gc, int32_t* nn);

/* Uploads the plan, runs the fragment census (failCount > 1000 rule, Segment.cpp:753-762)
 * for `seed`, and computes pair / fragCount prefix sums.  *planned_pairs = number of pair
 * IDs (PE: sum ceil(read_count/2); SE: sum read_count). */
int ssc_set_plan(ssc_handle* h, uint64_t seed,
                 const ssc_bin* bins, int64_t n_bins,
                 const ssc_segment* segs, int64_t n_segs,
                 const char* names, int64_t names_len,
                 int64_t* planned_pairs, int64_t* emitted_pairs);

/* Generates planned pair IDs [pair_lo, pair_hi) and streams the FASTQ bytes to `sink`
 * through pinned double buffers (host copies inside). */
int ssc_generate(ssc_handle* h, int64_t pair_lo, int64_t pair_hi, ssc_sink_fn sink, void* user);

/* Same work, output left in the handle's device slab (no device->host copy of FASTQ):
 * the device-resident measurement leg.  Any of the out pointers may be NULL.  Interleaved
 * PE output: the whole stream in *bytes1, *bytes2 = 0. */
int ssc_generate_device(ssc_handle* h, int64_t pair_lo, int64_t pair_hi,
                        uint64_t* bytes1, uint64_t* bytes2, uint64_t* bases, double* device_ms);

/*
 * Array output: the reads of a pair range written straight into caller-owned device arrays (e.g. torch tensors) for a
 * consumer on the same GPU -- no FASTQ text, no host copy.  The bytes are the FASTQ record's own; n = capacity in pairs,
 * M = 1 (SE) or 2 (PE).  Pair i of the range (FASTQ order) is row i.
 */
typedef struct ssc_read_arrays {      /* device pointers, caller-owned */
	uint8_t* reads;    /* [n][M][2][pitch], 16-byte aligned: row 0 = the base characters of the FASTQ record, row 1 = its
	                      quality characters (phred + 33, as written); every byte past the read's length is 0 */
	int16_t* length;   /* [n][M]: read length (RL +- indels, as in the FASTQ record) */
	int64_t* pair_id;  /* [n]: planned pair ID (the Philox address; abandoned pairs are absent, as in the FASTQ) */
	int32_t* segment;  /* [n]: index into the ssc_segment array of ssc_set_plan: the name prefix "@<popu>#<chr>#" */
	int32_t* pos;      /* [n]: position field of the read name (pos % segsize) */
	int32_t* frag;     /* [n]: fragment-counter field of the read name */
	int64_t capacity;  /* pairs */
	int32_t pitch;     /* must equal the value ssc_read_shape reports */
} ssc_read_arrays;

/* Pairs emitted by planned pair IDs [pair_lo, pair_hi), mates per pair, and the slot pitch: RL + 96 (the longest read the
 * library emits) rounded up to a multiple of 16. */
int ssc_read_shape(ssc_handle* h, int64_t pair_lo, int64_t pair_hi, int64_t* n_pairs, int32_t* n_mates, int32_t* pitch);
/* Generates planned pair IDs [pair_lo, pair_hi) into `out` on the fast kernel (kmer 3, read length 33..160; force_generic,
 * fp64_search and other profiles are refused with SSC_ERR_INVALID; the gzip option does not apply).  `stream` is a
 * cudaStream_t (0 = the legacy default stream): work queued on it before the call is ordered before the first write.  Returns
 * once the arrays are complete; *n_pairs (may be NULL) = the pairs written.  Null or misaligned pointers, a capacity below the
 * range, or a wrong pitch are refused before anything is written.  A read longer than RL + 96 fails with SSC_ERR_OVERFLOW.
 * ssc_stats counts pairs, reads, bases and launches as for FASTQ output; fastq_bytes is unchanged.  Device memory of the
 * handle: per-batch bookkeeping only (no FASTQ slab, blob scratch or pinned host buffers). */
int ssc_generate_reads(ssc_handle* h, int64_t pair_lo, int64_t pair_hi, const ssc_read_arrays* out, void* stream,
                       int64_t* n_pairs);
/* The read-name prefix "@<popu>#<chr>#" of a segment, NUL-terminated; cap >= its length + 1. */
int ssc_segment_name(ssc_handle* h, int32_t segment, char* out, int32_t cap);

/* Host-only diagnostic (no GPU needed): the symbol the integer-threshold table built from
 * `cdf` selects for the 32-bit draw u.  Must equal the reference's
 * randIndx(cdf, n) with r = 2.2204e-16 + (1 - 2.2204e-16) * (u / 2^32) for every u
 * (lib/mydefine/MyDefine.cpp:176-184); tests sweep the table boundaries with it. */
int ssc_table_lookup_host(const double* cdf, int n, uint32_t u);
/* Same for a 4-symbol substitution row encoded as {S0,S1,S2,base}. */
int ssc_sub_lookup_host(const double* cdf4, uint32_t u);

/* Host-only diagnostic (no GPU needed): one gzip member of in[0..n) built with the device encoder's own tables
 * (Huffman code fitted to the byte histogram of `sample`, CRC-32 by the kernel's lane-strided algebra) and bit
 * packing, stored instead when coding would make it longer than n + 23 bytes, as on the device.  Returns the member size,
 * 0 when it does not fit `cap`, or -1.  Tests inflate it with zlib and compare it with the device's members. */
int64_t ssc_gzip_member_host(const uint8_t* in, uint32_t n, const uint8_t* sample, size_t sample_n, uint8_t* out, size_t cap);

/* Measurement aid (no reference counterpart): the instruction-issue ceiling of the generation kernel on this GPU.
 * mode 0 = Philox4x32-10 only, one block per lane-cycle in the generation kernel's launch shape (the cost of the reference's
 * four uniform draws per base, Profile.cpp:1560/1569/1534/1578, and nothing else); mode 1 = the same plus the per-base table
 * work and byte stores of an indel-free read on synthetic tables.  Runs `reps` launches over n_pairs pairs of read_length
 * cycles per mate and returns the mean CUDA-event time of a launch.  bench.py reports it as roofline.issue. */
int ssc_issue_floor(ssc_handle* h, int mode, int read_length, int64_t n_pairs, int reps, double* ms_per_launch);

int ssc_get_stats(ssc_handle* h, ssc_stats* out);
int ssc_reset_stats(ssc_handle* h);

#ifdef __cplusplus
}
#endif
#endif
