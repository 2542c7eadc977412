/*
 * simuscop_host.h -- C ABI of the host front end (libsimuscop_host.so).
 *
 * Replaces, for the simuReads path, what the reference does between reading the
 * configuration file and dispatching segments:
 *   config.loadConfig(); genome.loadData(); profile.train(file);
 *   genome.generateSegments(); genome.yieldReads()            src/simuReads.cpp:48-74
 * ssh_open() covers everything up to generateSegments(); ssh_prepare_sample() is the
 * host half of Genome::yieldReads (read budget, GC-weighted bins, haplotype strings;
 * lib/genome/Genome.cpp:827-960) and hands the result to a device handle of
 * simuscop.h.  Samples must be prepared in increasing order (plan RNG state is shared,
 * as in the reference).  Errors in the input files terminate the process with the
 * reference's own messages and exit codes (exit(1) / exit(-1)), like the reference.
 */
#ifndef SIMUSCOP_HOST_H
#define SIMUSCOP_HOST_H

#include <stdint.h>
#include "simuscop.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ssh_job ssh_job;

int ssh_open(const char* config_path, uint64_t seed, ssh_job** out);
int ssh_close(ssh_job* job);
int ssh_num_samples(ssh_job* job);
/* file-name stem of sample s: "<popu>" or "<p1>_0.300+<p2>_0.250..." (Genome.cpp:857-866, 899-929) */
const char* ssh_sample_stem(ssh_job* job, int s);
int ssh_paired(ssh_job* job);
int ssh_read_length(ssh_job* job);
const char* ssh_output_dir(ssh_job* job);
/* dump_path may be NULL; otherwise an SSCPLAN1 file of the sample is written there */
int ssh_prepare_sample(ssh_job* job, int s, ssc_handle* dev, const char* dump_path,
                       int64_t* planned_pairs, int64_t* emitted_pairs);
/* The answer key of sample s: a VCFv4.2 file at `path` with every SNV and indel the sample's haplotypes hold, one phased
 * allele per copy (GT:HCN in the column of every population the sample draws from, '.' in the others; INFO/EAF the expected
 * allele fraction in this sample) and one <CNV> record per copy-number segment of the variation file (CN:MCN:HCN).  Call it
 * right after ssh_prepare_sample(job, s, ...) and before the next sample is prepared: it reads the phasing state as it stands
 * (a segment the reference leaves without a major set is phased again for the next sample).  Draws nothing from the plan RNG,
 * so the plans of later samples do not change.  The CLI writes it as <output>/<stem>.truth.vcf when SIMUSCOP_TRUTH_VCF=1.
 * Returns SSC_ERR_STATE unless s is the sample prepared last, SSC_ERR_SINK when the file cannot be written. */
int ssh_write_truth_vcf(ssh_job* job, int s, const char* path);
/* Host-only self test (no GPU): the splice lists from which the device assembles haplotypes with insertion / deletion
 * variants, materialised on the host, against the string construction of Segment::generateSegSequences
 * (lib/segment/Segment.cpp:124-460).  Returns the number of differing haplotypes. */
int ssh_selftest_splices(ssh_job* job, int64_t* haplotypes_checked, int64_t* segments_with_indels);

/* Output side (the role of SeqWriter, lib/seqwriter/SeqWriter.cpp:41-54): an ordered FASTQ file writer whose sink can be
 * handed to ssc_generate with user = the writer.  path2 NULL = single-end.  threads <= 1: slabs are written by the caller's
 * thread; otherwise one pwrite() stream per file, the two files side by side (a file is a serial resource under its inode
 * lock, so the default mode never uses more than two threads).  Environment SIMUSCOP_WRITER_MODE = mmap | hybrid: `threads`
 * workers copy 8 MB chunks into shared mappings of the slab's file ranges (hybrid: beside the two streams). */
typedef struct ssh_writer ssh_writer;
int ssh_writer_open(const char* path1, const char* path2, int threads, ssh_writer** out);
/* A single-stream writer on a descriptor the caller opened and closes (standard output, a pipe to an aligner): slabs are
 * written in order with write() from the calling thread, so descriptors that cannot seek work.  buf2 must be NULL (SE or
 * interleaved PE).  A failed write (EPIPE once the reader has gone, with SIGPIPE ignored) makes the sink return non-zero. */
int ssh_writer_open_fd(int fd, ssh_writer** out);
/* BGZF output (the handles' "gzip" and "bgzf" options): call after ssh_writer_open / ssh_writer_open_fd and before the first
 * slab.  From then on every slab must be a whole number of well-formed BGZF blocks (else the sink returns non-zero, takes no
 * more slabs, and ssh_writer_close reports SSC_ERR_SINK); ssh_writer_close appends the 28-byte BGZF EOF block to each stream
 * (also on a descriptor) unless a write failed.  index1 / index2 (either may be NULL; index2 needs a second file): a .gzi block
 * index of stream 1 / 2 in the layout of htslib's bgzf_index_dump -- uint64 entry count, then one (compressed offset,
 * uncompressed offset) uint64 pair per data block after the first (block 0 at (0, 0) is implicit, the EOF block has none), all
 * little-endian.  Entries are written as the slabs arrive and the count at close: 16 bytes per block of 32 pairs, ~150 MB per
 * file of a 3 Gb x 30x PE run.  Returns SSC_ERR_STATE after the first slab or a second call, SSC_ERR_SINK when an index
 * cannot be created. */
int ssh_writer_bgzf(ssh_writer* w, const char* index1, const char* index2);
ssc_sink_fn ssh_writer_sink(void);
int ssh_writer_close(ssh_writer* w, uint64_t* bytes1, uint64_t* bytes2);

/* The whole drop-in run: every sample -> FASTQ files in the output directory, on `device`.  Environment:
 * SIMUSCOP_INTERLEAVE=1 writes a PE sample to <output>/<stem>.fq (.fq.gz with SIMUSCOP_GZIP=1), mate 1 and mate 2 of each pair
 * in turn, instead of <stem>_1 / <stem>_2; SIMUSCOP_STDOUT=1 writes the reads (PE interleaved) to standard output and no
 * FASTQ file, and refuses a configuration with more than one sample; SIMUSCOP_BGZF=1 (implies SIMUSCOP_GZIP=1) writes every
 * .fq.gz as BGZF, ended by the EOF block, with its block index <name>.fq.gz.gzi beside it (standard output: no index);
 * SIMUSCOP_BAM=1 writes every sample, PE or SE, as unaligned BAM to <output>/<stem>.bam (standard output with SIMUSCOP_STDOUT=1):
 * the header block of ssc_bam_header with read group <stem>, the records of the handles' "bam" option (RG:Z:<stem>), the BGZF
 * EOF block, and no index; it takes precedence over SIMUSCOP_GZIP, SIMUSCOP_BGZF and SIMUSCOP_INTERLEAVE.  A stem longer than
 * the 64 bytes of a read group id gives its first bytes and "~<sample index>"; bytes outside [!-~] become '_'.  A sample whose
 * read names are not valid BAM names is refused before its file is opened. */
int ssh_run(ssh_job* job, int device);

#ifdef __cplusplus
}
#endif
#endif
