// host.h -- host front end of the drop-in simuReads: everything the reference does ONCE per run
// (config, FASTA, SNP / variation / target / abundance inputs, .profile -> FP64 CDF tables,
// segmentation, haplotype construction, GC-weighted read plan) restated in C++17, producing the
// flat plan that include/simuscop.h consumes.  The per-read loop itself lives on the GPU.
//
// Each function cites the reference lines whose semantics (and bits) it reproduces.
#pragma once
#include <cstdint>
#include <map>
#include <random>
#include <string>
#include <vector>

#include "../../include/simuscop.h"

namespace sschost {

[[noreturn]] void die(int code, const std::string& msg);   // prints to stderr and exits like the reference

std::string trim(const std::string& s, const char* chars = " \t\r\n");
std::vector<std::string> split(const std::string& s, char delim);
std::string abbr_chr(const std::string& chr);               // abbrOfChr, lib/mydefine/MyDefine.cpp:212-225

// ---- configuration file (lib/config/Config.cpp:14-175)
struct Config {
	std::map<std::string, std::string> str;
	std::map<std::string, int> num;
	std::map<std::string, double> real;
	std::vector<std::string> popu;
	void load(const std::string& path);
	bool paired() const { return str.at("layout") == "PE"; }
	bool verbose() const { return num.at("verbose") != 0; }
};

// ---- FASTA + .fai (lib/fastahack/Fasta.cpp)
struct FastaEntry { std::string name; long length; long long offset; int line_blen, line_len; };
class Fasta {
public:
	void open(const std::string& path);                      // builds <path>.fai when missing
	std::vector<std::string> names;                          // chr/chrom prefix stripped, index order
	long length(const std::string& chr) const;               // 0 when unknown
	// upper-cased bases [start, start+len) of chr (Genome::getSubSequence, lib/genome/Genome.cpp:423-429)
	const std::string& chromosome(const std::string& chr);   // whole chromosome, cached one at a time
	// positions of the cached chromosome that hold neither ACGT nor N (IUPAC codes): calculateGCPercent
	// (lib/mydefine/MyDefine.cpp:279-303) counts only a literal 'N' as unknown, the device mask every non-ACGT character
	bool other_in(size_t a, size_t b) const;
	const FastaEntry* entry(const std::string& chr) const;   // .fai geometry of a record, nullptr when unknown
	std::vector<FastaEntry> records;                         // every .fai record in index order, named by the first word of its header line
	int fd();                                                // the FASTA file, opened read-only on first use
	~Fasta();
private:
	int fd_ = -1;
	std::vector<size_t> cachedOther_;
	std::string path_;
	std::map<std::string, FastaEntry> idx_;
	std::string cachedName_, cached_;
};

// ---- sequencing profile (lib/profile/Profile.cpp:934-1434)
struct ProfileModel {
	std::string bases; int N = 0, K = 0, B = 0, RL = 0, Q = 94, minQ = 33, rows = 0;
	double insertRate = 0, delRate = 0, stdISize = 0, gcStd = 0;
	double gcMeans[101];
	std::vector<double> insCdf, delCdf, sub1, sub2, qual, isizeCdf;
	int minIS = 0; bool useCdf2 = false;
	void load(const std::string& path, Config& cfg);         // load + normParas(true) + initCDFs
	void fill(ssc_profile_tables* t, const Config& cfg) const;
	// GC factor samplers (Profile.cpp:1409-1415, 1507-1517)
	std::vector<std::default_random_engine> gcEng;
	std::vector<std::normal_distribution<double>> gcDist;
	void seed_gc(uint64_t seed);
	double gc_factor(int gc);
};

struct Cnv { long spos, epos; float cn, mcn; };
struct Snv { long pos; char ref, alt; bool het; };
struct Ins { long pos; std::string seq; bool het; };
struct Del { long pos; int len; bool het; };
struct Snp { long long pos; char nucleotide; };
struct Target { long spos, epos; };

struct Bin { long spos, epos; int hap; double weight; int rc; };
struct Poke { int hap; long off; char c; };
// A haplotype of a segment with insertion / deletion variants as a splice list: runs of the reference slice (copy t, bases
// [a, b) of the slice) and literal runs (inserted sequences), in order.  The device assembles it from the uploaded chromosome.
struct Piece { int copy; long a, b; std::string lit; long len() const { return copy >= 0 ? b - a : (long)lit.size(); } };   // substitution at offset off of every copy of the reference slice
struct BinSpec { long spos, epos; int hap; int kind; long n; long gcStart, gcLen; };   // a bin before its GC draw (host_plan.cpp)
struct ChrLayout {   // where the haplotype strings of one chromosome live in the device store
	std::vector<std::vector<int64_t>> base;      // [segment][haplotype] store index of the string, -1 = absent
	std::vector<std::vector<size_t>> hapLen;     // [segment][haplotype]
	std::vector<int64_t> contigEnd;              // [haplotype]
};

struct Segment {
	int idx; std::string chr; long start, end; int CN, mCN;
	bool fromCnv = false;                // made from a 'c' record of the variation file (not the ploidy default between them)
	std::vector<int> seqReps, mIndx, targetIdx;
	std::vector<Bin> bins; bool weighted = false;
	std::vector<std::string> hapCache;   // haplotypes kept between the weights pass and materialisation (memory permitting)
	long readCount = 0;
	long refSize() const { return end - start + 1; }
};

struct Sample { std::string stem; std::vector<float> props; };

class Job {
public:
	Config cfg;
	Fasta fasta;
	ProfileModel prof;
	std::vector<std::string> chroms;
	std::map<std::string, std::map<std::string, std::vector<Cnv>>> cnvs;   // popu -> chr -> records (file order)
	std::map<std::string, std::map<std::string, std::vector<Snv>>> snvs;
	std::map<std::string, std::map<std::string, std::vector<Ins>>> inss;
	std::map<std::string, std::map<std::string, std::vector<Del>>> dels;
	std::map<std::string, std::vector<Snp>> snps;
	std::map<std::string, std::vector<Target>> targets;
	std::vector<std::vector<float>> mix;
	std::map<std::string, std::map<std::string, std::vector<Segment>>> segs;   // popu -> chr -> segments
	std::vector<Sample> samples;
	long reads = 0;
	std::map<std::string, double> acn;
	uint64_t seed = 1;
	bool planSeeded = false;

	void open(const std::string& configPath);                // Genome::loadData + Profile::train + generateSegments
	long chrom_len(const std::string& chr) const;
	long genome_length() const;
	long target_length() const;

	// haplotype strings of one segment (Segment::generateSegSequences, lib/segment/Segment.cpp:124-460)
	void build_haplotypes(Segment& seg, const std::string& popu, std::vector<std::string>& haps);
	void phase_segment(Segment& seg);                        // rand()-driven copy-number phasing (Segment.cpp:140-215)
	bool segment_is_copy_only(const Segment& seg, const std::string& popu);
	void segment_copies_and_pokes(Segment& seg, const std::string& popu, std::vector<int>& reps, std::vector<Poke>& pokes);
	// the same from the phasing state as it stands: draws nothing, for a segment that has been phased
	void phased_copies_and_pokes(const Segment& seg, const std::string& popu, std::vector<int>& reps, std::vector<Poke>& pokes);
	// the insert / erase part of Segment::generateSegSequences (Segment.cpp:313-444) on splice lists instead of strings
	void segment_splices(Segment& seg, const std::string& popu, size_t refLen, const std::vector<int>& reps, std::vector<std::vector<Piece>>& ropes);
	// bins + weights (Segment::getWeightedLength, Segment.cpp:550-641)
	double weighted_length(Segment& seg, const std::string& popu);
	double weighted_length_from(Segment& seg, const std::vector<std::string>& haps);
	void enumerate_bins(const Segment& seg, const std::vector<size_t>& hapLen, std::vector<BinSpec>& out);
	double weights_from_gc(Segment& seg, const std::vector<BinSpec>& specs, const int* gc, const double* factors = nullptr);
	// weights pass on the device (ssc_gc_census), streaming the haplotype store at the same time
	int device_weights(const std::string& popu, const std::vector<ssc_handle*>& devs, uint64_t& localSize,
	                   std::map<std::string, ChrLayout>& layout);
	long long hapCacheBudget = 0;                             // bytes of haplotype strings that may stay cached
	void set_read_counts(const std::string& popu, long reads);   // Genome::setReadCounts, Genome.cpp:783-825
	void begin_plan();                                        // reads, ACNs, srand (Genome.cpp:831-852)

	// Streams sample `s` into the device handle: haplotype store + plan.  dumpPath (optional): SSCPLAN1 file.
	int prepare_sample(int s, ssc_handle* dev, const std::string& dumpPath, int64_t* planned, int64_t* emitted);
	// same, replicated into several device handles (one per GPU); an empty list = plan-only mode
	int prepare_sample_multi(int s, const std::vector<ssc_handle*>& devs, const std::string& dumpPath, int64_t* planned, int64_t* emitted);
	int lastPrepared = -1;                                    // the sample prepared last
	// truth.cpp: the variants and copy numbers the haplotypes of sample `s` carry, as a phased per-copy VCF (DESIGN.md section 10).
	// Reads the phasing state as it stands and draws nothing, so it describes sample `s` only while `s` is the sample prepared
	// last (a segment the reference leaves without a major set is phased again for the next sample).  0, or SSC_ERR_SINK when
	// `path` cannot be written.
	int write_truth_vcf(int s, const std::string& path);
private:
	void load_variations();
	void load_snps();
	void load_targets();
	void divide_targets();
	void load_abundance();
	void generate_segments();
	void divide_segment(const std::string& popu, const std::string& chr, long s, long e, int CN, int mCN, int& idx, bool fromCnv);
	long rand_int(long a, long b);                            // randomInteger, lib/mydefine/MyDefine.cpp:192-194
};

}  // namespace sschost
