// truth.cpp -- the answer key of an output sample: a phased VCF of the small variants and copy numbers its haplotypes carry.
//
// The changes are read off the same splice lists and substitutions the device assembles the haplotypes from
// (Job::segment_splices, Job::phased_copies_and_pokes), copy by copy, not from the input files: the reference's insert /
// erase offset arithmetic can move a deletion across a copy junction, remove an inserted sequence or drop a variant, and
// which copies hold a heterozygous change is decided by the rand()-driven phasing.  Nothing here draws from rand() or
// phases a segment, so the plan (and the FASTQ files) are the same with and without the truth file.  DESIGN.md section 10.
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <map>
#include <tuple>

#include "host.h"

namespace sschost {

namespace {
typedef std::tuple<long, std::string, std::string> VarKey;   // (POS, REF, ALT): the VCF order within a contig

// where a variant is and which copies hold it, for one population
struct VarSite {
	long locus = 0;                                   // the first changed reference base (the anchor of an insertion or SNV)
	std::map<int, std::vector<char>> copies;          // segment index -> allele of each copy of that segment
};

// the changes one copy of a segment holds: its surviving reference runs [a, b) of the slice, the inserted literals, and
// the substitutions of the haplotype index (slice offset -> base, the last one applied)
struct CopyWalk {
	const std::string& chr;                           // the upper-cased chromosome
	long start, refLen;                               // slice = chromosome bases [start, start + refLen), 1-based
	std::vector<std::pair<VarKey, long>> out;         // (record, locus)

	// one record for everything between the surviving slice offsets o1 < o2 (-1 and refLen: the slice's neighbours)
	void gap(long o1, long o2, const std::string& lit) {
		if (o2 == o1 + 1 && lit.empty()) return;
		const long a = start + o1;                    // 1-based anchor to the left
		const long chrLen = (long)chr.size();
		if (a >= 1) {
			if (start + o2 - 1 > chrLen) return;
			std::string ref = chr.substr((size_t)(a - 1), (size_t)(o2 - o1));
			std::string alt = chr.substr((size_t)(a - 1), 1) + lit;
			if (ref != alt) out.push_back({VarKey(a, ref, alt), o2 == o1 + 1 ? a : a + 1});
		} else {                                      // a change in front of chromosome position 1: anchored to the right
			const long r = start + o2;                // 1-based
			if (r > chrLen) return;
			std::string ref = chr.substr(0, (size_t)r);
			std::string alt = lit + chr.substr((size_t)(r - 1), 1);
			if (ref != alt) out.push_back({VarKey(1, ref, alt), 1});
		}
	}
	void snv(long o, char c) {
		const char b = (char)toupper((unsigned char)c);
		const long p = start + o;
		if (b != chr[(size_t)(p - 1)]) out.push_back({VarKey(p, chr.substr((size_t)(p - 1), 1), std::string(1, b)), p});
	}
};

// the segments of one population on one chromosome that hold a position, in plan order (more than one where 'c' records
// overlap): a binary search over the starts, then back while the running maximum of the ends still reaches the position
struct SegIndex {
	std::vector<size_t> order;                        // segment indices by start
	std::vector<long> start, maxEnd;
	explicit SegIndex(const std::vector<Segment>& v) {
		order.resize(v.size());
		for (size_t k = 0; k < v.size(); k++) order[k] = k;
		std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return v[a].start < v[b].start; });
		long m = 0;
		for (size_t k : order) { start.push_back(v[k].start); m = std::max(m, v[k].end); maxEnd.push_back(m); }
	}
	void holding(const std::vector<Segment>& v, long pos, std::vector<size_t>& out) const {
		out.clear();
		for (long i = (long)(std::upper_bound(start.begin(), start.end(), pos) - start.begin()) - 1; i >= 0 && maxEnd[(size_t)i] >= pos; i--)
			if (v[order[(size_t)i]].end >= pos) out.push_back(order[(size_t)i]);
		std::sort(out.begin(), out.end());
	}
};

bool write_all(FILE* fp, const std::string& s) { return fwrite(s.data(), 1, s.size(), fp) == s.size(); }

void format_eaf(std::string& s, double v) {
	char b[32];
	snprintf(b, sizeof(b), "%.6g", v);
	s += b;
}
}  // namespace

int Job::write_truth_vcf(int s, const std::string& path) {
	const double t0 = std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
	const int ploidy = cfg.num["ploidy"];
	const Sample& sm = samples[s];
	const size_t P = cfg.popu.size();
	// populations the sample's reads come from, and their weights per copy-base (Job::prepare_sample_multi: reads of a
	// population are proportional to props * ACN).  Without abundance rows that is the first population alone, and only its
	// segments have been phased: the columns of the others stay '.'.
	std::vector<double> props(P, 0.0);
	std::vector<char> used(P, 0);
	if (sm.props.empty()) { props[0] = 1.0; used[0] = 1; }
	else for (size_t p = 0; p < P; p++) { props[p] = sm.props[p]; used[p] = 1; }

	FILE* fp = fopen(path.c_str(), "w");
	if (!fp) return SSC_ERR_SINK;
	std::string out;
	out += "##fileformat=VCFv4.2\n##source=simuReads (simuscop_b200) haplotype truth\n";
	out += "##reference=" + cfg.str["ref"] + "\n";
	for (const FastaEntry& e : fasta.records) out += "##contig=<ID=" + e.name + ",length=" + std::to_string(e.length) + ">\n";
	out += "##ALT=<ID=CNV,Description=\"Copy-number segment\">\n"
	       "##INFO=<ID=EAF,Number=A,Type=Float,Description=\"Expected allele fraction in this sample before GC bias: sum of abundance x ALT copies over sum of abundance x copies, over the populations\">\n"
	       "##INFO=<ID=SVTYPE,Number=1,Type=String,Description=\"Type of the symbolic allele\">\n"
	       "##INFO=<ID=END,Number=1,Type=Integer,Description=\"Last position of the copy-number segment\">\n"
	       "##FORMAT=<ID=GT,Number=1,Type=String,Description=\"Allele of every copy: haplotype index by haplotype index, each index's tandem copies in order\">\n"
	       "##FORMAT=<ID=HCN,Number=.,Type=Integer,Description=\"Tandem copies of each haplotype index, of every segment of the population that holds the first changed base\">\n"
	       "##FORMAT=<ID=CN,Number=1,Type=Integer,Description=\"Copy number of the segment\">\n"
	       "##FORMAT=<ID=MCN,Number=1,Type=Integer,Description=\"Major copy number of the segment\">\n"
	       "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT";
	for (auto& p : cfg.popu) out += "\t" + p;
	out += "\n";
	bool ok = write_all(fp, out);
	long nRec = 0;
	for (size_t ri = 0; ri < fasta.records.size(); ri++) {
		// fasta.names[ri] is the record's chr-stripped name, which the variation files and the segments use
		const std::string& name = fasta.names[ri];
		const std::string& contig = fasta.records[ri].name;
		if (std::find(chroms.begin(), chroms.end(), name) == chroms.end() || fasta.entry(name)->offset != fasta.records[ri].offset) continue;
		const std::string& chr = fasta.chromosome(name);
		std::map<VarKey, std::vector<VarSite>> sites;             // record -> per population
		struct Line { long pos; std::string ref, alt, rest; };
		std::vector<Line> cnvLines;
		std::vector<std::vector<std::vector<int>>> repsOf(P);     // [population][segment] copies per haplotype index
		for (size_t pi = 0; pi < P; pi++) {
			if (!used[pi]) continue;
			const std::string& popu = cfg.popu[pi];
			std::vector<Segment>& v = segs[popu][name];
			repsOf[pi].resize(v.size());
			for (size_t k = 0; k < v.size(); k++) {
				Segment& sg = v[k];
				const size_t refOff = (size_t)(sg.start - 1);
				const long refLen = (long)std::min((size_t)sg.refSize(), chr.size() > refOff ? chr.size() - refOff : 0);
				std::vector<int>& reps = repsOf[pi][k];
				std::vector<Poke> pokes;
				phased_copies_and_pokes(sg, popu, reps, pokes);
				if (sg.fromCnv) {
					std::string hcn;
					for (int j = 0; j < ploidy; j++) hcn += (j ? "," : "") + std::to_string(reps[j]);
					std::string rest = ".\tPASS\tSVTYPE=CNV;END=" + std::to_string(sg.end) + "\tCN:MCN:HCN";
					for (size_t q = 0; q < P; q++)
						rest += q == pi ? "\t" + std::to_string(sg.CN) + ":" + std::to_string(sg.mCN) + ":" + hcn : std::string("\t.");
					cnvLines.push_back(Line{sg.start, chr.substr(refOff, 1), "<CNV>", rest});
				}
				if (refLen <= 0) continue;
				std::vector<std::vector<Piece>> ropes;
				segment_splices(sg, popu, (size_t)refLen, reps, ropes);
				int copy0 = 0;                                     // allele index of the first copy of haplotype index j
				for (int j = 0; j < ploidy; j++) {
					std::map<long, char> sub;                      // later substitutions of the same base win (SNP, then SNV)
					for (const Poke& pk : pokes) if (pk.hap == j && pk.off < refLen) sub[pk.off] = pk.c;
					// the runs and literals of every copy; a literal belongs to the copy of the run before it
					std::vector<std::vector<const Piece*>> byCopy(reps[j]);
					int cur = -1;
					std::vector<const Piece*> lead;                // literals in front of the first run
					for (const Piece& pc : ropes[j]) {
						if (pc.copy >= 0) { cur = pc.copy; byCopy[cur].insert(byCopy[cur].end(), lead.begin(), lead.end()); lead.clear(); }
						if (pc.copy >= 0 || cur >= 0) byCopy[cur].push_back(&pc);
						else lead.push_back(&pc);
					}
					for (int t = 0; t < reps[j]; t++) {
						CopyWalk w{chr, sg.start, refLen, {}};
						long prev = -1;
						std::string lit;
						for (const Piece* pc : byCopy[t]) {
							if (pc->copy < 0) { lit += pc->lit; continue; }
							if (pc->b <= pc->a) continue;
							w.gap(prev, pc->a, lit);
							lit.clear();
							for (auto it = sub.lower_bound(pc->a); it != sub.end() && it->first < pc->b; ++it) w.snv(it->first, it->second);
							prev = pc->b - 1;
						}
						w.gap(prev, refLen, lit);
						for (auto& r : w.out) {
							std::vector<VarSite>& vs = sites[r.first];
							if (vs.empty()) vs.resize(P);
							VarSite& site = vs[pi];
							site.locus = r.second;
							std::vector<char>& al = site.copies[(int)k];
							if ((int)al.size() < copy0 + t + 1) al.resize((size_t)(copy0 + t + 1), 0);
							al[(size_t)(copy0 + t)] = 1;
						}
					}
					copy0 += reps[j];
				}
			}
		}
		std::vector<SegIndex> index;
		for (size_t pi = 0; pi < P; pi++) index.emplace_back(segs[cfg.popu[pi]][name]);
		std::vector<size_t> hold;
		std::vector<Line> lines;
		for (auto& kv : sites) {
			long locus = 0;
			for (auto& site : kv.second) if (!site.copies.empty()) { locus = site.locus; break; }
			std::string rest = ".\tPASS\tEAF=";
			std::string cols;
			double num = 0, den = 0;
			for (size_t pi = 0; pi < P; pi++) {
				if (!used[pi]) { cols += "\t."; continue; }
				const std::vector<Segment>& v = segs[cfg.popu[pi]][name];
				std::string gt, hcn;
				int alt = 0, n = 0;
				index[pi].holding(v, locus, hold);
				for (size_t k : hold) {
					const std::vector<int>& reps = repsOf[pi][k];
					auto it = kv.second[pi].copies.find((int)k);
					int c = 0;
					for (int j = 0; j < ploidy; j++) {
						hcn += (hcn.empty() ? "" : ",") + std::to_string(reps[j]);
						for (int t = 0; t < reps[j]; t++, c++) {
							const bool a = it != kv.second[pi].copies.end() && c < (int)it->second.size() && it->second[(size_t)c];
							gt += (gt.empty() ? "" : "|") + std::string(a ? "1" : "0");
							alt += a; n++;
						}
					}
				}
				cols += "\t" + (gt.empty() ? std::string(".") : gt + ":" + hcn);
				num += props[pi] * alt; den += props[pi] * n;
			}
			format_eaf(rest, den > 0 ? num / den : 0.0);
			rest += "\tGT:HCN" + cols;
			lines.push_back(Line{std::get<0>(kv.first), std::get<1>(kv.first), std::get<2>(kv.first), rest});
		}
		lines.insert(lines.end(), cnvLines.begin(), cnvLines.end());
		std::stable_sort(lines.begin(), lines.end(), [](const Line& a, const Line& b) { return std::tie(a.pos, a.ref, a.alt) < std::tie(b.pos, b.ref, b.alt); });
		out.clear();
		for (const Line& l : lines) out += contig + "\t" + std::to_string(l.pos) + "\t.\t" + l.ref + "\t" + l.alt + "\t" + l.rest + "\n";
		ok = ok && write_all(fp, out);
		nRec += (long)lines.size();
	}
	if (fclose(fp) != 0 || !ok) return SSC_ERR_SINK;
	if (getenv("SIMUSCOP_TIMING")) {
		const double t1 = std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
		fprintf(stderr, "[simuscop timing] truth VCF %.3f s (%ld records)\n", t1 - t0, nRec);
	}
	return 0;
}

}  // namespace sschost
