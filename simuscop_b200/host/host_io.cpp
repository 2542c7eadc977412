// host_io.cpp -- configuration file, FASTA/.fai, SNP / variation / target / abundance loaders.
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <sstream>

#include "host.h"

namespace sschost {

void die(int code, const std::string& msg) {
	std::cerr << msg << std::endl;
	exit(code);
}

std::string trim(const std::string& s, const char* chars) {
	size_t a = s.find_first_not_of(chars);
	if (a == std::string::npos) return "";
	size_t b = s.find_last_not_of(chars);
	return s.substr(a, b - a + 1);
}

// getline-based split: "a,,b" -> {a,"",b}; a trailing delimiter adds no empty field (lib/split/split.cpp:3-15)
std::vector<std::string> split(const std::string& s, char delim) {
	std::vector<std::string> out;
	std::stringstream ss(s);
	std::string item;
	while (std::getline(ss, item, delim)) out.push_back(item);
	return out;
}

std::string abbr_chr(const std::string& chr) {
	size_t i = chr.find("chrom");
	if (i != std::string::npos) return chr.substr(i + 5);
	i = chr.find("chr");
	if (i != std::string::npos) return chr.substr(i + 3);
	return chr;
}

// ------------------------------------------------------------------------------------------------
// Config (lib/config/Config.cpp:14-175): same keys, defaults, messages and exit codes
// ------------------------------------------------------------------------------------------------
void Config::load(const std::string& path) {
	const char* strKeys[] = {"bam", "profile", "ref", "variation", "snp", "vcf", "target", "bases", "output", "abundance", "layout", "samtools"};
	for (const char* k : strKeys) str[k] = "";
	str["layout"] = "SE";
	str["bases"] = "ACTG";
	num = {{"kmer", 0}, {"bins", 0}, {"threads", 1}, {"verbose", 1}, {"readLength", 0}, {"coverage", 0}, {"ploidy", 2}, {"insertSize", 350}};
	real = {{"indelRate", 0.00025}};
	if (path.empty()) die(-1, "Error: configuration file not specified!");
	std::ifstream ifs(path.c_str());
	if (!ifs.is_open()) die(-1, "Error: can not open configuration file" + path);
	std::string line;
	int lineNum = 0;
	while (std::getline(ifs, line)) {
		lineNum++;
		line = trim(line);
		if (line.empty() || line[0] == '#') continue;
		size_t eq = line.find('=');
		if (eq == std::string::npos)
			die(1, "ERROR: line " + std::to_string(lineNum) + " is incorrectly formatted in file " + path + "\n" + line);
		std::string key = trim(line.substr(0, eq)), value = trim(line.substr(eq + 1));
		if (str.count(key)) str[key] = value;
		else if (num.count(key)) num[key] = atoi(value.c_str());
		else if (real.count(key)) real[key] = atof(value.c_str());
		else if (key == "name") {
			popu = split(value, ',');
			for (auto& p : popu) p = trim(p);
		} else
			die(1, "ERROR: unrecognized item \"" + key + "\" @line " + std::to_string(lineNum) + " in file " + path + "\n" + line);
	}
	// checkParas, Config.cpp:101-175
	if (str["profile"].empty()) die(1, "Error: sequencing profile must be specified!");
	if (str["snp"].empty()) std::cerr << "Warning: SNP file not specified!\nNo SNPs will be inserted into the genome." << std::endl;
	if (str["variation"].empty()) std::cerr << "Warning: variation file not specified!\nNo variations will be inserted into the genome." << std::endl;
	if (str["ref"].empty()) die(1, "Error: reference file not specified!");
	if (popu.empty()) die(1, "Error: population names not specified!");
	if (popu.size() > 1 && str["abundance"].empty()) die(1, "Error: abundance file not specified!");
	if (str["output"].empty()) die(1, "Error: output directory not specified!");
	if (str["layout"].empty()) {
		std::cerr << "Warning: sequence layout not specified!\nuse the default value: \"single end\"" << std::endl;
		str["layout"] = "SE";
	} else if (str["layout"] != "SE" && str["layout"] != "PE")
		die(1, "Error: sequence layout incorrectly specified!\nshould be SE or PE");
	if (num["threads"] < 1) die(1, "Error: number of threads should be a positive integer!");
	if (num["coverage"] < 1) die(1, "Error: sequence coverage should be a positive integer!");
	if (num["ploidy"] < 1) die(1, "Error: genome ploidy should be a positive integer!");
	if (str["layout"] == "PE" && num["insertSize"] < num["readLength"]) die(1, "Error: insert size should be not smaller than read length!");
	if (real["indelRate"] < 0 || real["indelRate"] > 0.001) die(1, "Error: indel error rate should be a value between 0 to 0.001!");
}

// ------------------------------------------------------------------------------------------------
// FASTA (lib/fastahack/Fasta.cpp:45-85 index reader, :103-191 indexer, :233-260 open)
// ------------------------------------------------------------------------------------------------
static std::string first_token(const std::string& s) {
	size_t a = s.find_first_not_of(" \t");
	if (a == std::string::npos) return "";
	size_t b = s.find_first_of(" \t", a);
	return s.substr(a, b == std::string::npos ? std::string::npos : b - a);
}

void Fasta::open(const std::string& path) {
	path_ = path;
	FILE* f = fopen(path.c_str(), "r");
	if (!f) die(1, "could not open " + path);
	fclose(f);
	const std::string fai = path + ".fai";
	struct stat st;
	if (stat(fai.c_str(), &st) != 0) {
		std::cerr << "index file " << fai << " not found, generating..." << std::endl;
		std::ifstream in(path.c_str());
		std::vector<FastaEntry> ents;
		FastaEntry cur{"", 0, -1, 0, 0};
		bool have = false, mismatch = false, emptyLine = false;
		std::string line;
		long long offset = 0, lineNo = 0;
		while (std::getline(in, line)) {
			lineNo++;
			int ll = (int)line.length();
			if (!line.empty() && line[0] == ';') {
			} else if (!line.empty() && line[0] == '>') {
				if (have) ents.push_back(cur);
				cur = FastaEntry{line.substr(1), 0, -1, 0, 0};
				have = true; mismatch = false; emptyLine = false;
			} else {
				if (cur.offset == -1) cur.offset = offset;
				cur.length += ll;
				if (cur.line_len) {
					if (mismatch || emptyLine) {
						if (ll == 0) emptyLine = true;
						else die(1, std::string(emptyLine ? "ERROR: embedded newline" : "ERROR: mismatched line lengths") + " at line " +
						             std::to_string(lineNo) + " within sequence " + cur.name + "\nFile not suitable for fasta index generation.");
					}
					if (cur.line_len != ll + 1) { mismatch = true; if (ll == 0) emptyLine = true; }
				} else cur.line_len = ll + 1;
				cur.line_blen = cur.line_len - 1;
			}
			offset += ll + 1;
		}
		if (have) ents.push_back(cur);
		std::stable_sort(ents.begin(), ents.end(), [](const FastaEntry& a, const FastaEntry& b) { return a.offset < b.offset; });
		// written under a private name and renamed, so that concurrent processes never read a partial index
		const std::string tmp = fai + ".tmp." + std::to_string((long)getpid());
		{
			std::ofstream out(tmp.c_str());
			if (!out.is_open()) die(1, "could not open index file " + fai + " for writing!");
			for (auto& e : ents) {
				std::string nm = split(e.name, ' ').empty() ? "" : split(e.name, ' ')[0];
				out << nm << "\t" << e.length << "\t" << e.offset << "\t" << e.line_blen << "\t" << e.line_len << std::endl;
			}
		}
		if (rename(tmp.c_str(), fai.c_str()) != 0) die(1, "could not open index file " + fai + " for writing!");
	}
	std::ifstream in(fai.c_str());
	if (!in.is_open()) die(1, "could not open index file " + fai);
	std::string line;
	long long ln = 0;
	while (std::getline(in, line)) {
		ln++;
		std::vector<std::string> f5 = split(line, '\t');
		if (f5.size() != 5)
			die(1, "Warning: malformed fasta index file " + fai + " does not have enough fields @line " + std::to_string(ln) + "\n" + line);
		std::string name = abbr_chr(first_token(f5[0]));
		names.push_back(name);
		records.push_back(FastaEntry{first_token(f5[0]), atol(f5[1].c_str()), atoll(f5[2].c_str()), atoi(f5[3].c_str()), atoi(f5[4].c_str())});
		idx_.insert(std::make_pair(name, FastaEntry{f5[0], atol(f5[1].c_str()), atoll(f5[2].c_str()), atoi(f5[3].c_str()), atoi(f5[4].c_str())}));
	}
}

// any character other than A, C, G, T, N in bases [a, b) of the cached chromosome
bool Fasta::other_in(size_t a, size_t b) const {
	auto it = std::lower_bound(cachedOther_.begin(), cachedOther_.end(), a);
	return it != cachedOther_.end() && *it < b;
}

const FastaEntry* Fasta::entry(const std::string& chr) const {
	auto it = idx_.find(chr);
	return it == idx_.end() ? nullptr : &it->second;
}

int Fasta::fd() {
	if (fd_ < 0) fd_ = ::open(path_.c_str(), O_RDONLY);
	return fd_;
}

Fasta::~Fasta() { if (fd_ >= 0) ::close(fd_); }

long Fasta::length(const std::string& chr) const {
	auto it = idx_.find(chr);
	return it == idx_.end() ? 0 : it->second.length;
}

const std::string& Fasta::chromosome(const std::string& chr) {
	if (chr == cachedName_) return cached_;
	auto it = idx_.find(chr);
	if (it == idx_.end()) die(1, "unable to find FASTA index entry for '" + chr + "'");
	const FastaEntry& e = it->second;
	FILE* f = fopen(path_.c_str(), "r");
	if (!f) die(1, "could not open " + path_);
	long nl = e.line_blen > 0 ? e.length / e.line_blen : 0;
	size_t raw = (size_t)e.length + (size_t)nl + 1;
	std::string buf(raw, '\0');
	fseeko(f, (off_t)e.offset, SEEK_SET);
	size_t got = fread(&buf[0], 1, raw, f);
	fclose(f);
	cached_.assign((size_t)e.length, 'N');
	cachedOther_.clear();
	size_t w = 0, i = 0;
	while (i < got && w < (size_t)e.length) {
		const char* nlp = (const char*)memchr(buf.data() + i, '\n', got - i);
		size_t lineEnd = nlp ? (size_t)(nlp - buf.data()) : got;
		size_t n = std::min(lineEnd - i, (size_t)e.length - w);
		char* dst = &cached_[w];
		const unsigned char* src = (const unsigned char*)buf.data() + i;
		unsigned other = 0;
		for (size_t k = 0; k < n; k++) {                       // toupper without a table: the loop vectorises
			const unsigned char c = src[k];
			const unsigned char u = (unsigned char)(c - (unsigned char)(((unsigned char)(c - 'a') < 26u) << 5));
			dst[k] = (char)u;
			other |= !((u == 'A') | (u == 'C') | (u == 'G') | (u == 'T') | (u == 'N'));
		}
		if (other)                                             // rare (IUPAC codes): remember where, see Fasta::other_in
			for (size_t k = 0; k < n; k++) {
				const char u = dst[k];
				if (!(u == 'A' || u == 'C' || u == 'G' || u == 'T' || u == 'N')) cachedOther_.push_back(w + k);
			}
		w += n;
		i = lineEnd + 1;
	}
	cached_.resize(w);
	cachedName_ = chr;
	return cached_;
}

// ------------------------------------------------------------------------------------------------
// Genome inputs
// ------------------------------------------------------------------------------------------------
long Job::chrom_len(const std::string& chr) const {
	if (std::find(chroms.begin(), chroms.end(), chr) == chroms.end()) return 0;   // Genome::getChromLen, Genome.cpp:382-396
	return fasta.length(chr);
}

long Job::genome_length() const {
	long n = 0;
	for (auto& c : chroms) n += chrom_len(c);
	return n;
}

long Job::target_length() const {
	if (targets.empty()) return genome_length();
	long n = 0;
	for (auto& kv : targets)
		for (auto& t : kv.second) n += t.epos - t.spos + 1;
	return n;
}

// Genome::loadAbers, lib/genome/Genome.cpp:41-206
void Job::load_variations() {
	const std::string file = cfg.str["variation"];
	if (file.empty()) return;
	std::ifstream ifs(file.c_str());
	if (!ifs.is_open()) die(-1, "can not open file " + file);
	auto knownPopu = [&](const std::string& p) { return std::find(cfg.popu.begin(), cfg.popu.end(), p) != cfg.popu.end(); };
	std::string line;
	int lineNum = 0, nc = 0, ns = 0, ni = 0, nd = 0;
	auto bad = [&](const std::string& what) { die(1, "ERROR: " + what + " at line " + std::to_string(lineNum) + " in file " + file + "\n" + line); };
	auto badFields = [&]() { die(1, "ERROR: line " + std::to_string(lineNum) + " has wrong number of fields in file " + file + "\n" + line); };
	auto hetOf = [&](const std::string& code, const char* what) {
		if (code != "homo" && code != "het") bad(std::string("unrecognized ") + what + " type");
		return code == "het";
	};
	while (std::getline(ifs, line)) {
		lineNum++;
		if (line.empty()) continue;
		std::vector<std::string> f = split(line, '\t');
		const std::string& type = f[0];
		if (type == "c") {
			if (f.size() != 7) badFields();
			if (!knownPopu(f[1])) bad("unrecognized population identifier");
			float cn = (float)atof(f[5].c_str()), mcn = (float)atof(f[6].c_str());
			if (cn < mcn) bad("total copy number should be not lower than major copy number");
			if (cn - mcn > mcn) mcn = cn - mcn;
			cnvs[f[1]][abbr_chr(f[2])].push_back(Cnv{atol(f[3].c_str()), atol(f[4].c_str()), cn, mcn});
			nc++;
		} else if (type == "s") {
			if (f.size() != 7) badFields();
			if (!knownPopu(f[1])) bad("unrecognized population identifier");
			char ref = f[4].at(0), alt = f[5].at(0);
			if (ref == alt) bad("the mutated allele should be not same as the reference allele");
			snvs[f[1]][abbr_chr(f[2])].push_back(Snv{atol(f[3].c_str()), ref, alt, hetOf(f[6], "SNV")});
			ns++;
		} else if (type == "i") {
			if (f.size() != 6) badFields();
			if (!knownPopu(f[1])) bad("unrecognized population identifier");
			inss[f[1]][abbr_chr(f[2])].push_back(Ins{atol(f[3].c_str()), f[4], hetOf(f[5], "insert")});
			ni++;
		} else if (type == "d") {
			if (f.size() != 6) badFields();
			if (!knownPopu(f[1])) bad("unrecognized population identifier");
			dels[f[1]][abbr_chr(f[2])].push_back(Del{atol(f[3].c_str()), atoi(f[4].c_str()), hetOf(f[5], "deletion")});
			nd++;
		} else bad("unrecognized aberraton type");
	}
	std::cerr << "\nDetails of the aberrations loaded from file " << file << " are as follows:" << std::endl;
	std::cerr << "CNV: " << nc << "\nSNV: " << ns << "\nInsert: " << ni << "\nDeletion: " << nd << std::endl;
}

static char complement_char(char c) {   // SNP::getComplement, lib/snp/snp.cpp:86-99
	switch (c) {
	case 'A': return 'T'; case 'T': return 'A'; case 'C': return 'G'; case 'G': return 'C';
	case 'a': return 't'; case 't': return 'a'; case 'c': return 'g'; case 'g': return 'c';
	default: return 'N';
	}
}

// SNPOnChr::readSNPs + SNP::SNP, lib/snp/snp.cpp:12-35, 147-203
void Job::load_snps() {
	const std::string file = cfg.str["snp"];
	if (file.empty()) return;
	FILE* fp = fopen(file.c_str(), "r");
	if (!fp) die(-1, "can not open SNP file " + file);
	char buf[1000];
	long lineNo = 0, n = 0;
	while (fgets(buf, 1000, fp)) {
		lineNo++;
		std::vector<char*> el;
		el.push_back(buf);
		for (char* p = buf; *p; p++)
			if (*p == '\t') { *p = '\0'; el.push_back(p + 1); }
		if (el.size() != 6) {
			std::cerr << "Warning: malformed snp file " << file << ", there should be 6 fields @line " << lineNo << std::endl << buf << std::endl;
			continue;
		}
		n++;
		std::string observed = el[3];
		char strand = *el[4], ref = *el[5];
		std::vector<std::string> al = split(observed, '/');
		if (strand == '-') ref = complement_char(ref);
		char nuc = (al[0].at(0) == ref) ? al[1].at(0) : al[0].at(0);
		if (strand == '-') nuc = complement_char(nuc);
		snps[abbr_chr(el[1])].push_back(Snp{atoll(el[2]), nuc});
	}
	fclose(fp);
	std::cerr << "\n" << n << " SNPs to simulate were loaded from file " << file << std::endl;
}

// Genome::loadTargets, lib/genome/Genome.cpp:238-295
void Job::load_targets() {
	const std::string file = cfg.str["target"];
	if (file.empty()) return;
	std::ifstream ifs(file.c_str());
	if (!ifs.is_open()) die(-1, "can not open target file " + file);
	std::string line;
	int lineNum = 0, cnt = 0;
	while (std::getline(ifs, line)) {
		lineNum++;
		std::vector<std::string> f = split(line, '\t');
		if (f.size() < 3) die(1, "ERROR: line " + std::to_string(lineNum) + " should have at least 3 fields in file " + file + "\n" + line);
		std::string chr = abbr_chr(f[0]);
		long chrLen = chrom_len(chr);
		if (chrLen <= 0) continue;
		Target t;
		t.spos = std::max((long)1, atol(f[1].c_str()) - 50 + 1);
		long e = atol(f[2].c_str());
		long tmp = e <= 0 ? chrLen - (-e) % chrLen : e;
		t.epos = std::min(chrLen, tmp + 50);
		targets[chr].push_back(t);
		cnt++;
	}
	std::cerr << "\ntotal " << cnt << " targets were loaded from file " << file << std::endl;
}

// Genome::divideTargets, lib/genome/Genome.cpp:684-739
void Job::divide_targets() {
	std::map<std::string, std::vector<Target>> out;
	for (auto& kv : targets) {
		for (auto& t : kv.second) {
			long spos = t.spos;
			long size = t.epos - t.spos + 1;
			int k = (int)(size / 1000);
			for (int i = 0; i < k; i++) {
				Target nt;
				nt.spos = spos;
				nt.epos = (i == k - 1) ? t.epos : spos + 1000 - 1;
				spos = nt.epos + 1;
				out[kv.first].push_back(nt);
			}
			if (spos <= t.epos) out[kv.first].push_back(Target{spos, t.epos});
		}
	}
	targets = out;
}

// Genome::loadAbundance, lib/genome/Genome.cpp:297-339
void Job::load_abundance() {
	const std::string file = cfg.str["abundance"];
	if (file.empty()) return;
	std::ifstream ifs(file.c_str());
	if (!ifs.is_open()) die(-1, "can not open abundance file " + file);
	std::string line;
	int lineNum = 0;
	while (std::getline(ifs, line)) {
		lineNum++;
		std::vector<std::string> f = split(line, '\t');
		if (f.size() != cfg.popu.size()) die(1, "ERROR: line " + std::to_string(lineNum) + " has wrong number of fields in file " + file + "\n" + line);
		std::vector<float> props;
		float sum = 0;
		for (auto& s : f) { float p = (float)atof(s.c_str()); sum += p; props.push_back(p); }
		if (fabs(1 - sum) > 0.001) die(1, "ERROR: the sum of abundances is not equal to one at line " + std::to_string(lineNum) + " in file " + file + "\n" + line);
		mix.push_back(props);
	}
	std::cerr << "\ntotal " << mix.size() << " population combinations were loaded from file " << file << std::endl;
}

void Job::open(const std::string& configPath) {
	cfg.load(configPath);
	{
		// haplotype strings may stay in host memory between the two plan passes: 40 % of RAM unless SIMUSCOP_HOST_CACHE_GB says otherwise
		const char* e = getenv("SIMUSCOP_HOST_CACHE_GB");
		long long phys = (long long)sysconf(_SC_PHYS_PAGES) * (long long)sysconf(_SC_PAGE_SIZE);
		hapCacheBudget = e ? (long long)(atof(e) * 1e9) : (long long)(0.4 * (double)phys);
	}
	// Genome::loadData, lib/genome/Genome.cpp:17-30
	load_variations();
	load_snps();
	std::string ref = cfg.str["ref"];
	if (ref.size() > 3 && ref.substr(ref.size() - 3) == ".gz") {   // Genome::loadRefSeq, Genome.cpp:217-236
		std::string plain = ref.substr(0, ref.size() - 3);
		std::string cmd = "gzip -cd " + ref + " > " + plain;
		if (system(cmd.c_str()) != 0) std::cerr << "Warning: gzip failed on " << ref << std::endl;
		ref = plain;
	}
	fasta.open(ref);
	chroms = fasta.names;
	if (chroms.empty()) die(1, "ERROR: reference sequence cannot be empty!");
	std::cerr << "\nReference sequence was loaded from file " << cfg.str["ref"] << std::endl;
	load_targets();
	divide_targets();
	load_abundance();
	// output directory (src/simuReads.cpp:56-60)
	std::string cmd = "test ! -e " + cfg.str["output"] + " && mkdir -m 755 -p " + cfg.str["output"];
	if (system(cmd.c_str())) {}
	prof.load(cfg.str["profile"], cfg);
	generate_segments();
	// sample list (Genome.cpp:857-866, 899-929)
	if (mix.empty()) samples.push_back(Sample{cfg.popu[0], {}});
	else
		for (auto& props : mix) {
			std::string fn;
			char b[1000];
			for (size_t i = 0; i < cfg.popu.size(); i++) {
				snprintf(b, sizeof(b), i == 0 ? "%s_%.3f" : "+%s_%.3f", cfg.popu[i].c_str(), props[i]);
				fn += b;
			}
			samples.push_back(Sample{fn, props});
		}
}

}  // namespace sschost
