// host_plan.cpp -- segmentation, haplotype construction, GC-weighted read plan, and streaming of
// one output sample into the device handle (haplotype store + bins) through the C ABI.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <atomic>
#include <chrono>
#include <thread>
#include <cstring>
#include <iostream>
#include <stdexcept>

#include "host.h"

namespace sschost {

// randomInteger, lib/mydefine/MyDefine.cpp:192-194 (libc rand(), seeded in begin_plan)
long Job::rand_int(long start, long end) {
	return (long)(start + (end - start) * (rand() / (RAND_MAX + 1.0)));
}

// Genome::divideSegment, lib/genome/Genome.cpp:741-763
void Job::divide_segment(const std::string& popu, const std::string& chr, long s, long e, int CN, int mCN, int& idx, bool fromCnv) {
	const unsigned int segMax = 1000000;
	std::vector<Segment>& v = segs[popu][chr];
	auto make = [&](long a, long b) {
		Segment g;
		g.idx = idx++; g.chr = chr; g.start = a; g.end = b; g.CN = CN; g.mCN = mCN; g.fromCnv = fromCnv;
		auto it = targets.find(chr);                         // Segment::initTargets, Segment.cpp:67-79
		if (!targets.empty() && it != targets.end())
			for (size_t i = 0; i < it->second.size(); i++) {
				long ts = it->second[i].spos, te = it->second[i].epos;
				if ((ts >= a && ts <= b) || (te >= a && te <= b) || (ts < a && te > b)) g.targetIdx.push_back((int)i);
			}
		v.push_back(g);
	};
	long size = e - s + 1;
	int n = (int)(size / segMax);
	unsigned int m = (unsigned int)(size - (long)n * segMax);
	for (int i = 0; i < n; i++) {
		if (i == n - 1 && m < segMax / 2) { make(s, e); s = e + 1; }
		else { make(s, s + segMax - 1); s += segMax; }
	}
	if (s <= e) make(s, e);
}

// Genome::generateSegments, lib/genome/Genome.cpp:634-682
void Job::generate_segments() {
	int ploidy = cfg.num["ploidy"];
	int mCN = (int)ceil((float)ploidy / 2);
	if (!targets.empty()) {
		chroms.clear();
		for (auto& kv : targets) chroms.push_back(kv.first);
	}
	for (auto& popu : cfg.popu) {
		for (auto& chr : chroms) {
			int idx = 0;
			std::vector<Cnv>& cv = cnvs[popu][chr];
			long segStart = 1;
			long chrLen = chrom_len(chr);
			segs[popu][chr];
			for (auto c : cv) {
				if (segStart > chrLen) break;
				c.epos = std::min(c.epos, chrLen);
				if (segStart < c.spos) divide_segment(popu, chr, segStart, c.spos - 1, ploidy, mCN, idx, false);
				divide_segment(popu, chr, c.spos, c.epos, (int)c.cn, (int)c.mcn, idx, true);
				segStart = c.epos + 1;
			}
			if (segStart <= chrLen) divide_segment(popu, chr, segStart, chrLen, ploidy, mCN, idx, false);
		}
	}
}

// Segment::generateSegSequences, lib/segment/Segment.cpp:124-460
// Copy-number phasing of a segment, the rand()-driven head of Segment::generateSegSequences (Segment.cpp:140-215):
// which haplotype indices exist (CN < ploidy) or how many copies each carries, and which of them form the "major" set.
// Runs once per segment (the first time its haplotypes are needed), in segment order: it consumes rand().
void Job::phase_segment(Segment& seg) {
	const int ploidy = cfg.num["ploidy"];
	const int CN = seg.CN, mCN = seg.mCN;
	if (seg.mIndx.empty()) {
		if (CN < ploidy) {
			for (int i = 0; i < CN; i++)
				while (true) {
					int j = (int)rand_int(0, ploidy);
					if (std::find(seg.seqReps.begin(), seg.seqReps.end(), j) == seg.seqReps.end()) { seg.seqReps.push_back(j); break; }
				}
			for (int i = 0; i < mCN; i++) seg.mIndx.push_back(seg.seqReps[i]);
		} else {
			for (int i = 0; i < ploidy; i++) seg.seqReps.push_back(1);
			int n = CN - ploidy;
			int k = (int)rand_int(0, ploidy);
			int i;
			for (i = n; i >= 0; i--) {
				if (seg.seqReps[k] + i == mCN) { seg.seqReps[k] += i; seg.mIndx.push_back(k); break; }
				else if (seg.seqReps[k] + i == CN - mCN) {
					seg.seqReps[k] += i;
					for (int j = 0; j < ploidy; j++) if (j != k) seg.mIndx.push_back(j);
					break;
				}
			}
			if (i >= 0) {
				n -= i;
				// the remaining copies go to the other haplotype indices; a haploid genome has none and the reference spins
				// forever in this loop (Segment.cpp:183-189) -- reject instead of hanging
				if (n > 0 && ploidy < 2)
					die(1, "ERROR: copy number " + std::to_string(CN) + " with major copy number " + std::to_string(mCN) + " cannot be phased with ploidy " +
					           std::to_string(ploidy) + " (" + seg.chr + ":" + std::to_string(seg.start) + ")");
				while (n > 0) { int j = (int)rand_int(0, ploidy); if (j != k) { seg.seqReps[j]++; n--; } }
			} else {
				while (n > 0) { int j = (int)rand_int(0, ploidy); seg.seqReps[j]++; n--; }
				for (int j = 0; j < ploidy; j++) seg.mIndx.push_back(j);
			}
		}
	}
}

void Job::build_haplotypes(Segment& seg, const std::string& popu, std::vector<std::string>& haps) {
	const int ploidy = cfg.num["ploidy"];
	haps.assign(ploidy, std::string());
	if (seg.CN == 0) die(1, "ERROR: copy number 0 segments are not supported (" + popu + " " + seg.chr + ":" + std::to_string(seg.start) + ")");
	const std::string& chrSeq = fasta.chromosome(seg.chr);
	const size_t refOff = (size_t)(seg.start - 1);
	const size_t refLen = std::min((size_t)seg.refSize(), chrSeq.size() > refOff ? chrSeq.size() - refOff : 0);
	const char* ref = chrSeq.data() + refOff;
	const unsigned int refSize = (unsigned int)refLen;
	const int CN = seg.CN;
	auto inM = [&](int j) { return std::find(seg.mIndx.begin(), seg.mIndx.end(), j) != seg.mIndx.end(); };
	phase_segment(seg);
	if (CN < ploidy) {
		for (int i = 0; i < ploidy; i++)
			if (std::find(seg.seqReps.begin(), seg.seqReps.end(), i) != seg.seqReps.end()) haps[i].assign(ref, refLen);
	} else {
		for (int i = 0; i < ploidy; i++) {
			haps[i].reserve((size_t)refSize * seg.seqReps[i] + 64);
			for (int j = 0; j < seg.seqReps[i]; j++) haps[i].append(ref, refLen);
		}
	}
	bool touched = false;   // the reference is already upper case: the final toupper only matters after a variant was applied
	auto poke = [&](std::string& h, int sindx, char c) {
		unsigned int len = (unsigned int)h.length();
		touched = true;
		for (unsigned int t = 0; t < len / refSize; t++) h[sindx + t * refSize] = c;
	};
	// SNPs: heterozygous, alternating between the major set and its complement (Segment.cpp:233-265)
	int k = 0;
	auto sit = snps.find(seg.chr);
	if (sit != snps.end())
		for (const Snp& s : sit->second) {
			if (s.pos >= seg.start && s.pos <= seg.end) {
				int sindx = (int)(s.pos - seg.start);
				for (int j = 0; j < ploidy; j++) if ((k == 0) == inM(j)) poke(haps[j], sindx, s.nucleotide);
				k = (k + 1) % 2;
			}
		}
	// SNVs (Segment.cpp:267-311)
	k = 0;
	for (const Snv& s : snvs[popu][seg.chr]) {
		if (s.pos >= seg.start && s.pos <= seg.end) {
			int sindx = (int)(s.pos - seg.start);
			if (!s.het) for (int j = 0; j < ploidy; j++) poke(haps[j], sindx, s.alt);
			else {
				for (int j = 0; j < ploidy; j++) if ((k == 0) == inM(j)) poke(haps[j], sindx, s.alt);
				k = (k + 1) % 2;
			}
		}
	}
	// insertions (Segment.cpp:313-370)
	std::vector<std::map<int, int>> insMap(ploidy), delMap(ploidy);
	std::vector<int> insLens(ploidy, 0), delLens(ploidy, 0);
	k = 0;
	for (const Ins& in : inss[popu][seg.chr]) {
		if (in.pos >= seg.start && in.pos <= seg.end) {
			int sindx = (int)(in.pos + 1 - seg.start);
			int len = (int)in.seq.length();
			for (int j = 0; j < ploidy; j++) {
				if (in.het && ((k == 0 && !inM(j)) || (k == 1 && inM(j)))) continue;
				int offset = 0;
				touched = true;
				for (auto& kv : insMap[j]) if (kv.first <= sindx) offset += kv.second;
				std::string& h = haps[j];
				int n = (int)(h.length() / (refSize + insLens[j]));
				for (int t = 0; t < n; t++) h.insert((size_t)(sindx + offset + t * (refSize + insLens[j] + len)), in.seq);
				insLens[j] += len;
				insMap[j].insert(std::make_pair(sindx, len));
			}
			if (in.het) k = (k + 1) % 2;
		}
	}
	// deletions (Segment.cpp:372-444)
	k = 0;
	for (const Del& d : dels[popu][seg.chr]) {
		if (d.pos >= seg.start && d.pos <= seg.end) {
			int sindx = (int)(d.pos - seg.start);
			for (int j = 0; j < ploidy; j++) {
				if (d.het && ((k == 0 && !inM(j)) || (k == 1 && inM(j)))) continue;
				int offset = 0;
				for (auto& kv : insMap[j]) if (kv.first <= sindx) offset += kv.second;
				for (auto& kv : delMap[j]) if (kv.first <= sindx) offset -= kv.second;
				if (sindx + offset < 0) continue;
				std::string& h = haps[j];
				int n = (int)(h.length() / (refSize + insLens[j] - delLens[j]));
				for (int t = 0; t < n; t++) h.erase((size_t)(sindx + offset + t * (refSize + insLens[j] - delLens[j] - d.len)), (size_t)d.len);
				delLens[j] += d.len;
				delMap[j].insert(std::make_pair(sindx, d.len));
			}
			if (d.het) k = (k + 1) % 2;
		}
	}
	if (touched)
		for (auto& h : haps) std::transform(h.begin(), h.end(), h.begin(), [](unsigned char c) { return (char)toupper(c); });
}

// calculateGCPercent, lib/mydefine/MyDefine.cpp:279-303
static int gc_percent(const char* s, size_t n) {
	if (n == 0) return 0;
	int gc = 0, nn = 0;
	for (size_t i = 0; i < n; i++) {
		const char c = s[i];
		gc += (c == 'G') | (c == 'C');
		nn += (c == 'N');
	}
	if (nn > 0) return -1;
	return 100 * gc / (int)(n - nn);
}

// fn(lo, hi, r) over R contiguous ranges of [0, n), each on its own thread; the ranges ascend with r, so results that are
// concatenated in range order are in element order whatever R is
static unsigned plan_threads() { return std::max(1u, std::min(16u, std::thread::hardware_concurrency())); }
template <class F> static void parallel_ranges(size_t n, unsigned R, F fn) {
	if (R <= 1 || n < 2) { fn((size_t)0, n, 0u); return; }
	std::vector<std::thread> th;
	for (unsigned r = 1; r < R; r++) th.emplace_back(fn, n * r / R, n * (r + 1) / R, r);
	fn((size_t)0, n / R, 0u);
	for (auto& t : th) t.join();
}

static inline bool is_acgtn(char ch) { const char c = (char)(ch & 0xDF); return c == 'A' || c == 'C' || c == 'G' || c == 'T' || c == 'N'; }   // either case: haplotypes are upper-cased last (Segment.cpp:448-458)

namespace {
// phase timers of the plan construction (printed when SIMUSCOP_TIMING is set)
struct PhaseTimers {
	double build = 0, gc = 0, upload = 0, counts = 0, census = 0, enumerate = 0, flatten = 0, setPlan = 0;
	static double now() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
} g_tm;
}  // namespace

// Segment::getWeightedLength, lib/segment/Segment.cpp:550-641
double Job::weighted_length(Segment& seg, const std::string& popu) {
	double wl = 0;
	if (seg.weighted) {
		for (auto& b : seg.bins) wl += b.weight;
		return wl;
	}
	std::vector<std::string> haps;
	double t0 = PhaseTimers::now();
	build_haplotypes(seg, popu, haps);
	double t1 = PhaseTimers::now();
	wl = weighted_length_from(seg, haps);
	g_tm.build += t1 - t0; g_tm.gc += PhaseTimers::now() - t1;
	// keep the strings for the materialisation pass when they fit the host budget (saves the second build)
	size_t bytes = 0;
	for (auto& h : haps) bytes += h.size();
	if ((long long)bytes <= hapCacheBudget) { hapCacheBudget -= (long long)bytes; seg.hapCache.swap(haps); }
	return wl;
}

// The bins of Segment::getWeightedLength (Segment.cpp:567-624) in the reference's order, without their weights:
// bin = (spos, epos, haplotype), GC interval = bases [gcStart, gcStart + gcLen) of that haplotype string, and the
// weight formula: kind 0: gcFactor / fragSize; kind 1: gcFactor * n / (fragSize * fragSize); kind 2: no draw, weight 0.
void Job::enumerate_bins(const Segment& seg, const std::vector<size_t>& hapLen, std::vector<BinSpec>& out) {
	const int ploidy = cfg.num["ploidy"];
	const unsigned int fragSize = 1000;
	out.clear();
	if (targets.empty()) {
		for (int i = 0; i < ploidy; i++) {
			const size_t len = hapLen[i];
			if (len == 0) continue;
			int k = (int)(len / fragSize);
			for (int j = 0; j < k; j++) {
				long spos = (long)j * fragSize, epos = (long)(j + 1) * fragSize - 1;
				out.push_back(BinSpec{spos, epos, i, 0, 0, spos, (long)fragSize});
			}
			if ((size_t)k * fragSize < len) {
				long spos = (long)k * fragSize;
				out.push_back(BinSpec{spos, (long)len - 1, i, 1, (long)(len - (size_t)spos), spos, (long)(len - (size_t)spos)});
			}
		}
	} else if (!seg.targetIdx.empty()) {
		const std::vector<Target>& tg = targets[seg.chr];
		for (int i = 0; i < ploidy; i++) {
			const size_t len = hapLen[i];
			if (len == 0) continue;
			int n = ((int)seg.seqReps.size() < ploidy) ? 1 : seg.seqReps[i];
			long refLen = (long)(len / n);
			for (int k = 0; k < n; k++)
				for (int m : seg.targetIdx) {
					long spos = std::max(tg[m].spos, seg.start) - seg.start;
					long epos = std::min(tg[m].epos, seg.start + refLen - 1) - seg.start;
					long sk = spos + (long)(k * len / n), ek = epos + (long)(k * len / n);
					out.push_back(BinSpec{sk, ek, i, 1, ek - sk + 1, sk, ek >= sk ? ek - sk + 1 : 0});
				}
		}
	} else {
		out.push_back(BinSpec{0, 0, 0, 2, 0, 0, 0});
	}
}

// weights of the enumerated bins from their GC percentages (one Profile::getGCFactor draw per bin, in bin order)
// factors (optional): the getGCFactor draw of every bin, made ahead in the same per-percentage order (device_weights)
double Job::weights_from_gc(Segment& seg, const std::vector<BinSpec>& specs, const int* gc, const double* factors) {
	const unsigned int fragSize = 1000;
	double wl = 0;
	seg.bins.reserve(seg.bins.size() + specs.size());
	for (size_t b = 0; b < specs.size(); b++) {
		const BinSpec& sp = specs[b];
		double w;
		if (sp.kind == 0) w = (factors ? factors[b] : prof.gc_factor(gc[b])) / fragSize;
		else if (sp.kind == 1) w = (factors ? factors[b] : prof.gc_factor(gc[b])) * sp.n / (fragSize * fragSize);
		else w = 0.0;
		seg.bins.push_back(Bin{sp.spos, sp.epos, sp.hap, w, 0});
		wl += w;
	}
	seg.weighted = !seg.bins.empty();
	return wl;
}

double Job::weighted_length_from(Segment& seg, const std::vector<std::string>& haps) {
	std::vector<size_t> hapLen(haps.size());
	for (size_t i = 0; i < haps.size(); i++) hapLen[i] = haps[i].length();
	std::vector<BinSpec> specs;
	enumerate_bins(seg, hapLen, specs);
	std::vector<int> gc(specs.size());
	for (size_t b = 0; b < specs.size(); b++)
		gc[b] = specs[b].kind == 2 ? 0 : gc_percent(haps[specs[b].hap].data() + specs[b].gcStart, (size_t)specs[b].gcLen);
	return weights_from_gc(seg, specs, gc.data());
}

// A segment none of whose variants is an insertion or deletion: every haplotype is the reference slice repeated once per
// copy with SNP / SNV alleles substituted (Segment.cpp:217-311), so the device can build it from the uploaded chromosome.
bool Job::segment_is_copy_only(const Segment& seg, const std::string& popu) {
	for (const Ins& in : inss[popu][seg.chr]) if (in.pos >= seg.start && in.pos <= seg.end) return false;
	for (const Del& d : dels[popu][seg.chr]) if (d.pos >= seg.start && d.pos <= seg.end) return false;
	return true;
}

// copies per haplotype index and the substitutions (haplotype, offset in the first copy, allele) in application order
void Job::segment_copies_and_pokes(Segment& seg, const std::string& popu, std::vector<int>& reps, std::vector<Poke>& pokes) {
	if (seg.CN == 0) die(1, "ERROR: copy number 0 segments are not supported (" + popu + " " + seg.chr + ":" + std::to_string(seg.start) + ")");
	phase_segment(seg);
	phased_copies_and_pokes(seg, popu, reps, pokes);
}

void Job::phased_copies_and_pokes(const Segment& seg, const std::string& popu, std::vector<int>& reps, std::vector<Poke>& pokes) {
	const int ploidy = cfg.num["ploidy"];
	reps.assign(ploidy, 0);
	for (int i = 0; i < ploidy; i++)
		reps[i] = seg.CN < ploidy ? (std::find(seg.seqReps.begin(), seg.seqReps.end(), i) != seg.seqReps.end() ? 1 : 0) : seg.seqReps[i];
	auto inM = [&](int j) { return std::find(seg.mIndx.begin(), seg.mIndx.end(), j) != seg.mIndx.end(); };
	pokes.clear();
	int k = 0;
	auto sit = snps.find(seg.chr);
	if (sit != snps.end())
		for (const Snp& sn : sit->second)
			if (sn.pos >= seg.start && sn.pos <= seg.end) {
				for (int j = 0; j < ploidy; j++) if ((k == 0) == inM(j)) pokes.push_back(Poke{j, (long)(sn.pos - seg.start), sn.nucleotide});
				k = (k + 1) % 2;
			}
	k = 0;
	for (const Snv& sv : snvs[popu][seg.chr])
		if (sv.pos >= seg.start && sv.pos <= seg.end) {
			if (!sv.het) for (int j = 0; j < ploidy; j++) pokes.push_back(Poke{j, (long)(sv.pos - seg.start), sv.alt});
			else {
				for (int j = 0; j < ploidy; j++) if ((k == 0) == inM(j)) pokes.push_back(Poke{j, (long)(sv.pos - seg.start), sv.alt});
				k = (k + 1) % 2;
			}
		}
}

namespace {
// std::string::insert / erase semantics on a splice list (including their out_of_range behaviour, which the string path has
// through the standard library)
long rope_len(const std::vector<Piece>& r) { long n = 0; for (const Piece& p : r) n += p.len(); return n; }

// index of the piece that starts exactly at pos after splitting (pos <= length)
size_t rope_split(std::vector<Piece>& r, long pos) {
	long at = 0;
	for (size_t i = 0; i < r.size(); i++) {
		const long n = r[i].len();
		if (pos == at) return i;
		if (pos < at + n) {
			Piece left = r[i], right = r[i];
			const long cut = pos - at;
			if (left.copy >= 0) { left.b = left.a + cut; right.a = left.b; }
			else { left.lit = r[i].lit.substr(0, (size_t)cut); right.lit = r[i].lit.substr((size_t)cut); }
			r[i] = left;
			r.insert(r.begin() + (long)i + 1, right);
			return i + 1;
		}
		at += n;
	}
	return r.size();
}

void rope_insert(std::vector<Piece>& r, long pos, const std::string& seq) {
	if (pos < 0 || pos > rope_len(r)) throw std::out_of_range("basic_string::insert");
	const size_t i = rope_split(r, pos);
	Piece p; p.copy = -1; p.a = p.b = 0; p.lit = seq;
	r.insert(r.begin() + (long)i, p);
}

void rope_erase(std::vector<Piece>& r, long pos, long n) {
	const long total = rope_len(r);
	if (pos < 0 || pos > total) throw std::out_of_range("basic_string::erase");
	if (n < 0) n = total - pos;                       // (size_t)len of a negative length: to the end, as the string path
	n = std::min(n, total - pos);
	if (n <= 0) return;
	const size_t i = rope_split(r, pos);
	const size_t j = rope_split(r, pos + n);
	r.erase(r.begin() + (long)i, r.begin() + (long)j);
}
}  // namespace

// Insertions and deletions of a segment applied to splice lists: the same order, positions and offset bookkeeping as
// Job::build_haplotypes (Segment.cpp:313-444), with string insert / erase replaced by their splice-list forms.  The SNP / SNV
// substitutions, which the reference applies first, do not move any base: they are mapped onto the final layout afterwards
// (device_weights).
void Job::segment_splices(Segment& seg, const std::string& popu, size_t refLen, const std::vector<int>& reps, std::vector<std::vector<Piece>>& ropes) {
	const int ploidy = cfg.num["ploidy"];
	const unsigned int refSize = (unsigned int)refLen;
	auto inM = [&](int j) { return std::find(seg.mIndx.begin(), seg.mIndx.end(), j) != seg.mIndx.end(); };
	ropes.assign(ploidy, std::vector<Piece>());
	for (int i = 0; i < ploidy; i++)
		for (int t = 0; t < reps[i]; t++) { Piece p; p.copy = t; p.a = 0; p.b = (long)refLen; ropes[i].push_back(p); }
	std::vector<std::map<int, int>> insMap(ploidy), delMap(ploidy);
	std::vector<int> insLens(ploidy, 0), delLens(ploidy, 0);
	int k = 0;
	for (const Ins& in : inss[popu][seg.chr]) {
		if (in.pos >= seg.start && in.pos <= seg.end) {
			int sindx = (int)(in.pos + 1 - seg.start);
			int len = (int)in.seq.length();
			for (int j = 0; j < ploidy; j++) {
				if (in.het && ((k == 0 && !inM(j)) || (k == 1 && inM(j)))) continue;
				int offset = 0;
				for (auto& kv : insMap[j]) if (kv.first <= sindx) offset += kv.second;
				std::vector<Piece>& h = ropes[j];
				int n = (int)(rope_len(h) / (refSize + insLens[j]));
				for (int t = 0; t < n; t++) rope_insert(h, (long)(sindx + offset + t * (refSize + insLens[j] + len)), in.seq);
				insLens[j] += len;
				insMap[j].insert(std::make_pair(sindx, len));
			}
			if (in.het) k = (k + 1) % 2;
		}
	}
	k = 0;
	for (const Del& d : dels[popu][seg.chr]) {
		if (d.pos >= seg.start && d.pos <= seg.end) {
			int sindx = (int)(d.pos - seg.start);
			for (int j = 0; j < ploidy; j++) {
				if (d.het && ((k == 0 && !inM(j)) || (k == 1 && inM(j)))) continue;
				int offset = 0;
				for (auto& kv : insMap[j]) if (kv.first <= sindx) offset += kv.second;
				for (auto& kv : delMap[j]) if (kv.first <= sindx) offset -= kv.second;
				if (sindx + offset < 0) continue;
				std::vector<Piece>& h = ropes[j];
				int n = (int)(rope_len(h) / (refSize + insLens[j] - delLens[j]));
				for (int t = 0; t < n; t++) rope_erase(h, (long)(sindx + offset + t * (refSize + insLens[j] - delLens[j] - d.len)), (long)d.len);
				delLens[j] += d.len;
				delMap[j].insert(std::make_pair(sindx, d.len));
			}
			if (d.het) k = (k + 1) % 2;
		}
	}
	for (auto& h : ropes)
		for (Piece& p : h)
			if (p.copy < 0) std::transform(p.lit.begin(), p.lit.end(), p.lit.begin(), [](unsigned char c) { return (char)toupper(c); });
}

// Device mode of the weights pass: the haplotype strings of one population are built chromosome by chromosome, appended
// to the haplotype store(s) in contig order (for every haplotype index, the segments' strings in order) and dropped; the
// GC percentages of all bins of the chromosome come from ssc_gc_census on the packed store.  Same bins, same draws in
// the same order, hence the same weights as weighted_length_from() -- and no haplotype string outlives its chromosome.
int Job::device_weights(const std::string& popu, const std::vector<ssc_handle*>& devs, uint64_t& localSize,
                        std::map<std::string, ChrLayout>& layout) {
	const int ploidy = cfg.num["ploidy"];
	const bool useRefBuild = !getenv("SIMUSCOP_HOST_HAPLOTYPES");   // debugging: build every haplotype string on the host
	int rc = 0;
	// .fai geometry of a record as ssc_reference_upload_fasta wants it; false: not usable for the device path
	struct Geom { uint64_t off, rawLen, n; uint32_t lb, lw; };
	auto geom_of = [&](const std::string& c, Geom& g) -> bool {
		const FastaEntry* e = fasta.entry(c);
		if (!useRefBuild || !e || e->line_blen <= 0 || e->length <= 0) return false;
		const uint64_t lines = (uint64_t)((e->length - 1) / e->line_blen);                 // full lines in front of the last one
		g.off = (uint64_t)e->offset; g.n = (uint64_t)e->length; g.lb = (uint32_t)e->line_blen; g.lw = (uint32_t)e->line_len;
		g.rawLen = g.n + lines * (uint64_t)(e->line_len - e->line_blen);
		return true;
	};
	bool prefetched = false;                     // the record of the chromosome about to be processed is being read in the background
	for (size_t ci = 0; ci < chroms.size(); ci++) {
		const std::string& chr = chroms[ci];
		std::vector<Segment>& v = segs[popu][chr];
		ChrLayout& L = layout[chr];
		L.base.assign(v.size(), std::vector<int64_t>(ploidy, -1));
		L.hapLen.assign(v.size(), std::vector<size_t>(ploidy, 0));
		L.contigEnd.assign(ploidy, 0);
		double t0 = PhaseTimers::now();
		// The chromosome goes to the device straight from the FASTA file (raw lines -> pinned staging -> unfold kernel) and every
		// haplotype is assembled there: copies of the segment's reference slice per copy-number phasing, for segments with
		// insertion / deletion variants as a splice list of slice runs and inserted literals (Segment::generateSegSequences'
		// insert / erase arithmetic runs on the list instead of on strings), SNP / SNV alleles poked in afterwards.  The host
		// reads and upper-cases the chromosome only when it needs the string itself: IUPAC codes in the record (the count
		// comes back from the unfold kernel), in an inserted sequence or in an allele.  While this chromosome is processed, the
		// record of the next one is read and unfolded in the background (ssc_reference_prefetch_fasta).
		const FastaEntry* fe = fasta.entry(chr);
		const size_t chrLen = fe ? (size_t)fe->length : 0;
		bool needHost = !useRefBuild || !fe || fe->line_blen <= 0;
		bool devRef = false;
		Geom g;
		if (geom_of(chr, g)) {
			uint64_t nOther = 0;
			for (ssc_handle* dev : devs) {
				rc = prefetched ? ssc_reference_adopt_prefetched(dev, &nOther)
				                : ssc_reference_upload_fasta(dev, fasta.fd(), g.off, g.rawLen, g.n, g.lb, g.lw, &nOther);
				if (rc) return rc;
			}
			devRef = true;
			if (nOther > 0) needHost = true;
		}
		prefetched = false;
		Geom gn;
		if (ci + 1 < chroms.size() && geom_of(chroms[ci + 1], gn)) {
			for (ssc_handle* dev : devs) { rc = ssc_reference_prefetch_fasta(dev, fasta.fd(), gn.off, gn.rawLen, gn.n, gn.lb, gn.lw); if (rc) return rc; }
			prefetched = true;
		}
		static const std::string noSeq;
		const std::string& chrSeq = needHost ? fasta.chromosome(chr) : noSeq;
		std::vector<std::vector<std::string>> haps(v.size());
		std::vector<std::vector<int>> reps(v.size());
		std::vector<std::vector<Poke>> pokes(v.size());
		std::vector<std::vector<std::vector<Piece>>> ropes(v.size());      // [segment][haplotype]: splice lists of the segments with indel variants
		std::vector<char> onDev(v.size(), 0), hostGc(v.size(), 0);
		std::vector<size_t> refOffs(v.size(), 0), refLens(v.size(), 0);
		bool anyDev = false;
		for (size_t k = 0; k < v.size(); k++) {
			const size_t refOff = (size_t)(v[k].start - 1);
			const size_t refLen = std::min((size_t)v[k].refSize(), chrLen > refOff ? chrLen - refOff : 0);
			refOffs[k] = refOff; refLens[k] = refLen;
			// The device census counts every non-ACGT character as unknown; the reference only a literal 'N'
			// (calculateGCPercent, MyDefine.cpp:279-303).  A segment whose haplotypes can hold any other character (IUPAC
			// codes in the FASTA, in an inserted sequence or in an allele) keeps its strings on the host and gets its GC
			// percentages from gc_percent() below.
			bool exotic = needHost && fasta.other_in(refOff, refOff + refLen);
			if (!exotic && useRefBuild && refLen > 0) {
				segment_copies_and_pokes(v[k], popu, reps[k], pokes[k]);
				for (const Poke& pk : pokes[k]) exotic |= !is_acgtn(pk.c);
				if (!exotic && !segment_is_copy_only(v[k], popu)) {
					segment_splices(v[k], popu, refLen, reps[k], ropes[k]);
					for (auto& r : ropes[k]) for (const Piece& p : r) if (p.copy < 0) for (char c : p.lit) exotic |= !is_acgtn(c);
				}
				if (!exotic) {
					for (int h = 0; h < ploidy; h++) {
						if (ropes[k].empty()) L.hapLen[k][h] = refLen * (size_t)reps[k][h];
						else { size_t n = 0; for (const Piece& p : ropes[k][h]) n += (size_t)p.len(); L.hapLen[k][h] = n; }
					}
					onDev[k] = 1; anyDev = true;
					continue;
				}
				ropes[k].clear();
			}
			if (!needHost) fasta.chromosome(chr);          // (an exotic allele on a chromosome that was not needed on the host so far)
			build_haplotypes(v[k], popu, haps[k]);
			for (int h = 0; h < ploidy; h++) {
				L.hapLen[k][h] = haps[k][h].size();
				if (!exotic) for (char c : haps[k][h]) if (!is_acgtn(c)) { exotic = true; break; }
			}
			hostGc[k] = exotic ? 1 : 0;
		}
		double t1 = PhaseTimers::now();
		if (anyDev && !devRef)
			for (ssc_handle* dev : devs) { rc = ssc_reference_upload(dev, chrSeq.data(), chrSeq.size()); if (rc) return rc; }
		std::vector<int64_t> pokePos; std::vector<char> pokeChr;
		for (int h = 0; h < ploidy; h++) {
			for (size_t k = 0; k < v.size(); k++) {
				if (L.hapLen[k][h] == 0) continue;
				uint64_t first = localSize;
				if (onDev[k] && ropes[k].empty()) {
					for (ssc_handle* dev : devs) { rc = ssc_genome_append_ref(dev, refOffs[k], refLens[k], reps[k][h], &first); if (rc) return rc; }
					for (const Poke& pk : pokes[k])
						if (pk.hap == h && (size_t)pk.off < refLens[k])
							for (int t = 0; t < reps[k][h]; t++) { pokePos.push_back((int64_t)(first + (uint64_t)pk.off + (uint64_t)t * refLens[k])); pokeChr.push_back(pk.c); }
				} else if (onDev[k]) {
					// splice list: slice runs from the uploaded chromosome, literal runs from the host; a substitution lands on
					// every surviving run of the slice that holds its base (one per copy unless a deletion took it)
					uint64_t at = localSize;
					for (const Piece& p : ropes[k][h]) {
						const uint64_t n = (uint64_t)p.len();
						if (n == 0) continue;
						uint64_t f = at;
						for (ssc_handle* dev : devs) {
							rc = p.copy >= 0 ? ssc_genome_append_ref(dev, refOffs[k] + (uint64_t)p.a, n, 1, &f) : ssc_genome_append(dev, p.lit.data(), n, &f);
							if (rc) return rc;
						}
						if (p.copy >= 0)
							for (const Poke& pk : pokes[k])
								if (pk.hap == h && pk.off >= p.a && pk.off < p.b) { pokePos.push_back((int64_t)(f + (uint64_t)(pk.off - p.a))); pokeChr.push_back(pk.c); }
						at = f + n;
					}
				} else {
					for (ssc_handle* dev : devs) { rc = ssc_genome_append(dev, haps[k][h].data(), haps[k][h].size(), &first); if (rc) return rc; }
				}
				L.base[k][h] = (int64_t)first;
				localSize = first + L.hapLen[k][h];
			}
			L.contigEnd[h] = (int64_t)localSize;
		}
		if (!pokePos.empty()) {
			// later substitutions of the same base win (SNP, then SNV): keep the last one per store index
			std::map<int64_t, char> last;
			for (size_t i = 0; i < pokePos.size(); i++) last[pokePos[i]] = pokeChr[i];
			pokePos.clear(); pokeChr.clear();
			for (auto& kv : last) { pokePos.push_back(kv.first); pokeChr.push_back(kv.second); }
			for (ssc_handle* dev : devs) { rc = ssc_genome_poke(dev, pokePos.data(), pokeChr.data(), (int64_t)pokePos.size()); if (rc) return rc; }
		}
		for (size_t k = 0; k < v.size(); k++) if (!hostGc[k]) { haps[k].clear(); haps[k].shrink_to_fit(); }
		double t2 = PhaseTimers::now();
		// census of every bin of the chromosome in one call.  The per-bin passes of this block (bin enumeration, census intervals,
		// GC percentages, weights) run over contiguous segment ranges on a few host threads; everything they produce is
		// position-determined, only the getGCFactor draws are ordered (see below).
		const unsigned R = v.size() >= 8 ? std::min<unsigned>(plan_threads(), (unsigned)v.size()) : 1u;
		std::vector<std::vector<BinSpec>> specs(v.size());
		std::vector<size_t> cenOff(v.size() + 1, 0);          // census intervals of segment k: [cenOff[k], cenOff[k+1])
		parallel_ranges(v.size(), R, [&](size_t lo, size_t hi, unsigned) {
			for (size_t k = lo; k < hi; k++) {
				if (v[k].weighted) continue;
				enumerate_bins(v[k], L.hapLen[k], specs[k]);
				size_t n = 0;
				if (!hostGc[k]) for (auto& sp : specs[k]) n += sp.kind != 2;
				cenOff[k + 1] = n;
			}
		});
		for (size_t k = 0; k < v.size(); k++) cenOff[k + 1] += cenOff[k];
		std::vector<int64_t> starts(cenOff[v.size()]); std::vector<int32_t> lens(cenOff[v.size()]);
		parallel_ranges(v.size(), R, [&](size_t lo, size_t hi, unsigned) {
			for (size_t k = lo; k < hi; k++) {
				if (v[k].weighted || hostGc[k]) continue;
				size_t o = cenOff[k];
				for (auto& sp : specs[k]) {
					if (sp.kind == 2) continue;
					starts[o] = L.base[k][sp.hap] + sp.gcStart;
					lens[o] = (int32_t)sp.gcLen;
					o++;
				}
			}
		});
		std::vector<int32_t> cgc(starts.size()), cnn(starts.size());
		g_tm.enumerate += PhaseTimers::now() - t2;
		rc = ssc_gc_census(devs[0], starts.data(), lens.data(), (int64_t)starts.size(), cgc.data(), cnn.data());
		if (rc) return rc;
		double t3 = PhaseTimers::now();
		// GC percentage of every bin of the chromosome, then the getGCFactor draws.  Every percentage has its own engine
		// (Profile.cpp:1409-1415), so the draws of one percentage only depend on the order of the bins with that percentage:
		// the 101 streams are independent and are advanced by several threads, each stream in bin order -- the values are
		// the ones a single pass over the bins would draw.
		size_t flat = 0;
		std::vector<std::vector<int>> gcs(v.size());
		std::vector<size_t> flatOff(v.size(), 0);
		for (size_t k = 0; k < v.size(); k++) { if (v[k].weighted) continue; flatOff[k] = flat; flat += specs[k].size(); }
		// per range and percentage: how many draws (counting sort, so that byGc[g] lists its bins in bin order)
		std::vector<std::vector<uint32_t>> cnt(R, std::vector<uint32_t>(101, 0));
		parallel_ranges(v.size(), R, [&](size_t lo, size_t hi, unsigned r) {
			for (size_t k = lo; k < hi; k++) {
				if (v[k].weighted) continue;
				std::vector<int>& gc = gcs[k];
				gc.assign(specs[k].size(), 0);
				size_t q = cenOff[k];
				for (size_t b = 0; b < specs[k].size(); b++) {
					if (specs[k][b].kind == 2) continue;
					if (hostGc[k]) gc[b] = gc_percent(haps[k][specs[k][b].hap].data() + specs[k][b].gcStart, (size_t)specs[k][b].gcLen);
					else {
						// calculateGCPercent, lib/mydefine/MyDefine.cpp:279-303: empty -> 0, any N -> -1, else 100*gc/n (integer)
						const int32_t n = lens[q];
						gc[b] = n == 0 ? 0 : (cnn[q] > 0 ? -1 : 100 * cgc[q] / n);
						q++;
					}
					if (gc[b] >= 0 && gc[b] <= 100) cnt[r][gc[b]]++;
				}
			}
		});
		std::vector<double> factors(flat, 0.0);
		{
			std::vector<std::vector<uint32_t>> byGc(101);
			std::vector<std::vector<size_t>> at(R, std::vector<size_t>(101, 0));
			for (int g = 0; g <= 100; g++) {
				size_t tot = 0;
				for (unsigned r = 0; r < R; r++) { at[r][g] = tot; tot += cnt[r][g]; }
				byGc[g].resize(tot);
			}
			parallel_ranges(v.size(), R, [&](size_t lo, size_t hi, unsigned r) {
				std::vector<size_t> o = at[r];
				for (size_t k = lo; k < hi; k++) {
					if (v[k].weighted) continue;
					for (size_t b = 0; b < specs[k].size(); b++) {
						const int g = gcs[k][b];
						if (specs[k][b].kind != 2 && g >= 0 && g <= 100) byGc[g][o[g]++] = (uint32_t)(flatOff[k] + b);
					}
				}
			});
			const unsigned T = plan_threads();
			std::atomic<int> next(0);
			auto run = [&]() {
				for (int g = next.fetch_add(1); g <= 100; g = next.fetch_add(1)) {
					if (byGc[g].empty()) continue;
					// engine and distribution of this percentage on the thread's own stack while it draws: the 101 engines
					// are 8 bytes apart in memory, neighbouring percentages would fight over the same cache line
					std::default_random_engine eng = prof.gcEng[g];
					std::normal_distribution<double> dist = prof.gcDist[g];
					std::vector<double> out(byGc[g].size());               // drawn into private memory, scattered in one go
					for (size_t k = 0; k < out.size(); k++) {
						double x = dist(eng);
						while (x < 0) x = dist(eng);                     // Profile::getGCFactor, Profile.cpp:1507-1517
						out[k] = x;
					}
					for (size_t k = 0; k < out.size(); k++) factors[byGc[g][k]] = out[k];
					prof.gcEng[g] = eng; prof.gcDist[g] = dist;
				}
			};
			if (flat < 20000 || T == 1) run();
			else {
				std::vector<std::thread> th;
				for (unsigned t = 1; t < T; t++) th.emplace_back(run);
				run();
				for (auto& t : th) t.join();
			}
		}
		parallel_ranges(v.size(), R, [&](size_t lo, size_t hi, unsigned) {
			for (size_t k = lo; k < hi; k++) {
				if (v[k].weighted) continue;
				weights_from_gc(v[k], specs[k], gcs[k].data(), factors.data() + flatOff[k]);
			}
		});
		g_tm.build += t1 - t0; g_tm.upload += t2 - t1; g_tm.census += t3 - t2; g_tm.gc += PhaseTimers::now() - t3;
	}
	return 0;
}

// Genome::setReadCounts + Segment::setReadCount, lib/genome/Genome.cpp:783-825, lib/segment/Segment.cpp:462-476
void Job::set_read_counts(const std::string& popu, long nreads) {
	std::map<std::string, double> chrWL;
	double WL = 0;
	for (auto& chr : chroms) {
		double w = 0;
		for (auto& sg : segs[popu][chr]) w += weighted_length(sg, popu);
		WL += w;
		chrWL[chr] = w;
	}
	long cur = 0;
	for (size_t i = 0; i < chroms.size(); i++) {
		std::vector<Segment>& v = segs[popu][chroms[i]];
		double cw = chrWL[chroms[i]];
		long chrReads = (i + 1 < chroms.size()) ? (long)(nreads * (cw / WL)) : nreads - cur;
		long sum = 0;
		for (size_t j = 0; j < v.size(); j++) {
			long rc;
			if (j + 1 < v.size()) { rc = (long)((weighted_length(v[j], popu) / cw) * chrReads); sum += rc; }
			else rc = chrReads - sum;
			Segment& sg = v[j];
			double total = weighted_length(sg, popu) + 2.2204e-16;
			long acc = 0;
			for (auto& b : sg.bins) { long r = (long)(b.weight * rc / total); b.rc = (int)r; acc += r; }
			if (acc < rc && !sg.bins.empty()) sg.bins[0].rc += (int)(rc - acc);
			sg.readCount = rc;
		}
		cur += chrReads;
	}
}

// head of Genome::yieldReads, lib/genome/Genome.cpp:827-852
void Job::begin_plan() {
	if (planSeeded) return;
	planSeeded = true;
	reads = target_length() * cfg.num["coverage"] / cfg.num["readLength"];
	if (cfg.verbose()) std::cerr << "\nNumber of reads to sample: " << reads << std::endl;
	for (auto& pk : segs) {
		long sum = 0;
		for (auto& ck : pk.second)
			for (auto& sg : ck.second) sum += (long)((unsigned int)(sg.CN * sg.refSize()));
		acn[pk.first] = (double)sum / genome_length();
	}
	if (cfg.verbose()) {
		std::cerr << (acn.size() > 1 ? "\nAverage copy number of populations: " : "\nAverage copy number: ") << std::endl;
		for (auto& kv : acn) std::cerr << kv.first << ": " << kv.second << std::endl;
	}
	std::cerr << "\n*****Generating samples*****" << std::endl;
	srand((unsigned)seed);
	prof.seed_gc(seed);
}

namespace {
struct PlanWriter {
	FILE* fp = nullptr;
	template <class T> static void app(std::string& s, T v) { s.append((const char*)&v, sizeof(T)); }
	void rec(int32_t tag, const std::string& body) {
		int64_t n = (int64_t)body.size();
		fwrite(&tag, 4, 1, fp); fwrite(&n, 8, 1, fp); fwrite(body.data(), 1, body.size(), fp);
	}
};
}  // namespace

int Job::prepare_sample(int s, ssc_handle* dev, const std::string& dumpPath, int64_t* planned, int64_t* emitted) {
	std::vector<ssc_handle*> devs;
	if (dev) devs.push_back(dev);
	return prepare_sample_multi(s, devs, dumpPath, planned, emitted);
}

int Job::prepare_sample_multi(int s, const std::vector<ssc_handle*>& devs, const std::string& dumpPath, int64_t* planned, int64_t* emitted) {
	begin_plan();
	const Sample& sm = samples[s];
	const int ploidy = cfg.num["ploidy"];
	const bool paired = cfg.paired();
	// dev == nullptr: plan-only mode (no GPU needed): store offsets are tracked locally, the plan is only dumped
	ssc_profile_tables pt;
	prof.fill(&pt, cfg);
	int rc = 0;
	for (ssc_handle* dev : devs) { rc = ssc_set_profile(dev, &pt); if (rc) return rc; }
	uint64_t localSize = 0;

	// populations of this sample and their read budgets (Genome.cpp:868, 931-936)
	std::vector<std::pair<std::string, long>> pops;
	if (sm.props.empty()) pops.push_back({cfg.popu[0], reads});
	else {
		double w_acn = 0;
		for (size_t i = 0; i < cfg.popu.size(); i++) w_acn += sm.props[i] * acn[cfg.popu[i]];
		for (size_t i = 0; i < cfg.popu.size(); i++) {
			long pr = (long)(reads * sm.props[i] * acn[cfg.popu[i]] / w_acn);   // long * float is a float product in the reference
			pops.push_back({cfg.popu[i], pr});
		}
	}

	PlanWriter pw;
	// "<path>.flat": profile tables + the flat bin / segment / name arrays handed to ssc_set_plan, no haplotype strings
	// (tags 5-7; a full dump of a 3 Gb diploid job would carry 6 GB of ASCII)
	const bool flatDump = dumpPath.size() > 5 && dumpPath.compare(dumpPath.size() - 5, 5, ".flat") == 0;
	if (!dumpPath.empty()) {
		pw.fp = fopen(dumpPath.c_str(), "wb");
		if (!pw.fp) die(3, "cannot open " + dumpPath);
		fwrite("SSCPLAN1", 1, 8, pw.fp);
		std::string p;
		int32_t hdr[16] = {prof.N, prof.K, prof.B, prof.Q, prof.minQ, prof.RL, paired ? 1 : 0, prof.useCdf2 ? 1 : 0,
		                   cfg.num["insertSize"], prof.isizeCdf.empty() ? 0 : prof.minIS, (int32_t)prof.isizeCdf.size(),
		                   (int32_t)prof.insCdf.size(), (int32_t)prof.delCdf.size(), prof.rows, ploidy, 0};
		p.append((const char*)hdr, sizeof(hdr));
		PlanWriter::app<double>(p, prof.insertRate); PlanWriter::app<double>(p, prof.delRate);
		char b8[8]; memset(b8, 0, 8); strncpy(b8, prof.bases.c_str(), 8); p.append(b8, 8);
		auto ad = [&](const std::vector<double>& v) { if (!v.empty()) p.append((const char*)v.data(), v.size() * 8); };
		ad(prof.isizeCdf); ad(prof.insCdf); ad(prof.delCdf); ad(prof.sub1); if (prof.useCdf2) ad(prof.sub2); ad(prof.qual);
		pw.rec(1, p);
	}

	// upper bound of the haplotype store of this sample
	uint64_t reserve = 0;
	for (auto& pp : pops)
		for (auto& chr : chroms) {
			uint64_t insTotal = 0;
			for (auto& in : inss[pp.first][chr]) insTotal += in.seq.length();
			for (auto& sg : segs[pp.first][chr]) reserve += (uint64_t)std::max(sg.CN, 1) * ((uint64_t)sg.refSize() + insTotal);
		}
	for (ssc_handle* dev : devs) { rc = ssc_genome_reserve(dev, reserve + 1024); if (rc) return rc; }

	std::vector<ssc_bin> bins;
	std::vector<ssc_segment> segments;
	std::string names;
	const bool onDevice = !devs.empty();
	for (auto& pp : pops) {
		const std::string& popu = pp.first;
		// device mode: weights pass = haplotype upload + GC census on the GPU; plan-only mode: host strings
		std::map<std::string, ChrLayout> layout;
		if (onDevice) { rc = device_weights(popu, devs, localSize, layout); if (rc) return rc; }
		double tc0 = PhaseTimers::now();
		set_read_counts(popu, pp.second);
		g_tm.counts += PhaseTimers::now() - tc0;
		const double tf0 = PhaseTimers::now();
		{
			size_t nb = bins.size(), ns = segments.size();
			for (auto& chr : chroms) { ns += segs[popu][chr].size(); for (auto& sg : segs[popu][chr]) nb += sg.bins.size(); }
			bins.reserve(nb); segments.reserve(ns);
		}
		for (auto& chr : chroms) {
			std::vector<Segment>& v = segs[popu][chr];
			const int32_t nameOff = (int32_t)names.size();
			const std::string nm = "@" + popu + "#" + chr + "#";
			names += nm;
			// the chromosome's haplotype strings (Genome.cpp:876-878): needed here in plan-only mode and for a plan dump
			std::vector<std::vector<std::string>> haps(v.size());
			if (!onDevice || (pw.fp && !flatDump)) {
				for (size_t k = 0; k < v.size(); k++) {
					if (!v[k].hapCache.empty()) {     // kept from the weights pass (same strings: generateSegSequences is deterministic once mIndx is set)
						size_t bb = 0;
						for (auto& h : v[k].hapCache) bb += h.size();
						haps[k].swap(v[k].hapCache);
						v[k].hapCache.clear(); v[k].hapCache.shrink_to_fit();
						hapCacheBudget += (long long)bb;
					} else build_haplotypes(v[k], popu, haps[k]);
				}
			}
			if (pw.fp && !flatDump) {
				std::string u;
				PlanWriter::app<int32_t>(u, (int32_t)popu.size()); PlanWriter::app<int32_t>(u, (int32_t)chr.size());
				u += popu; u += chr;
				pw.rec(2, u);
			}
			// contig layout: for every haplotype index, the segments' strings in order
			ChrLayout hostLayout;
			if (!onDevice) {
				hostLayout.base.assign(v.size(), std::vector<int64_t>(ploidy, -1));
				hostLayout.hapLen.assign(v.size(), std::vector<size_t>(ploidy, 0));
				hostLayout.contigEnd.assign(ploidy, 0);
				for (int h = 0; h < ploidy; h++) {
					for (size_t k = 0; k < v.size(); k++) {
						hostLayout.hapLen[k][h] = haps[k][h].size();
						if (haps[k][h].empty()) continue;
						hostLayout.base[k][h] = (int64_t)localSize;
						localSize += haps[k][h].size();
					}
					hostLayout.contigEnd[h] = (int64_t)localSize;
				}
			}
			const ChrLayout& L = onDevice ? layout[chr] : hostLayout;
			// flat ssc_bin records of the chromosome: offsets first, then the segments filled side by side on host threads
			std::vector<size_t> binOff(v.size() + 1, bins.size());
			std::vector<uint32_t> segsizes(v.size(), 0);
			const int32_t segId0 = (int32_t)segments.size();
			for (size_t k = 0; k < v.size(); k++) {
				Segment& sg = v[k];
				uint64_t seqSize = 0;
				for (int h = 0; h < ploidy; h++) seqSize += L.hapLen[k][h];
				segsizes[k] = (uint32_t)((unsigned int)seqSize / (unsigned int)sg.CN);   // Segment.cpp:712-714
				binOff[k + 1] = binOff[k] + sg.bins.size();
				ssc_segment ss;
				ss.first_bin = (int64_t)binOff[k]; ss.n_bins = (int64_t)sg.bins.size();
				ss.name_offset = nameOff; ss.name_len = (int32_t)nm.size();
				segments.push_back(ss);
			}
			bins.resize(binOff[v.size()]);
			parallel_ranges(v.size(), v.size() >= 8 ? std::min<unsigned>(plan_threads(), (unsigned)v.size()) : 1u, [&](size_t lo, size_t hi, unsigned) {
				for (size_t k = lo; k < hi; k++) {
					const Segment& sg = v[k];
					ssc_bin* out = bins.data() + binOff[k];
					for (const Bin& b : sg.bins) {
						ssc_bin sb;
						memset(&sb, 0, sizeof(sb));
						const bool present = b.hap >= 0 && b.hap < ploidy && L.base[k][b.hap] >= 0;
						sb.hap_base = present ? L.base[k][b.hap] : 0;
						sb.contig_end = present ? L.contigEnd[b.hap] : 0;
						sb.spos = (int32_t)b.spos; sb.epos = (int32_t)b.epos;
						sb.segsize = segsizes[k];
						sb.read_count = (present && sg.readCount != 0) ? b.rc : 0;   // Segment::yieldReads early return, Segment.cpp:675-677
						sb.segment = segId0 + (int32_t)k;
						*out++ = sb;
					}
				}
			});
			for (size_t k = 0; k < v.size(); k++) {
				Segment& sg = v[k];
				const uint32_t segsize = segsizes[k];
				if (pw.fp && !flatDump) {
					std::string r;
					PlanWriter::app<int32_t>(r, sg.idx); PlanWriter::app<int32_t>(r, sg.CN);
					PlanWriter::app<int64_t>(r, sg.start); PlanWriter::app<int64_t>(r, sg.end);
					PlanWriter::app<int64_t>(r, (int64_t)segsize); PlanWriter::app<int64_t>(r, sg.readCount);
					PlanWriter::app<int32_t>(r, (int32_t)sg.bins.size()); PlanWriter::app<int32_t>(r, ploidy);
					for (int h = 0; h < ploidy; h++) PlanWriter::app<int64_t>(r, (int64_t)haps[k][h].size());
					for (int h = 0; h < ploidy; h++) r += haps[k][h];
					for (auto& b : sg.bins) PlanWriter::app<int64_t>(r, b.spos);
					for (auto& b : sg.bins) PlanWriter::app<int64_t>(r, b.epos);
					for (auto& b : sg.bins) PlanWriter::app<int32_t>(r, b.hap);
					for (auto& b : sg.bins) PlanWriter::app<int32_t>(r, b.rc);
					pw.rec(3, r);
				}
			}
		}
		g_tm.flatten += PhaseTimers::now() - tf0;
	}
	if (pw.fp && flatDump) {
		pw.rec(5, std::string((const char*)bins.data(), bins.size() * sizeof(ssc_bin)));
		pw.rec(6, std::string((const char*)segments.data(), segments.size() * sizeof(ssc_segment)));
		pw.rec(7, names);
	}
	if (pw.fp) { pw.rec(9, std::string()); fclose(pw.fp); }
	if (devs.empty()) { if (planned) *planned = 0; if (emitted) *emitted = 0; lastPrepared = s; return 0; }
	const double ts0 = PhaseTimers::now();
	for (ssc_handle* dev : devs) {
		rc = ssc_set_plan(dev, seed, bins.data(), (int64_t)bins.size(), segments.data(), (int64_t)segments.size(),
		                  names.data(), (int64_t)names.size(), planned, emitted);
		if (rc) return rc;
	}
	lastPrepared = s;
	g_tm.setPlan += PhaseTimers::now() - ts0;
	if (getenv("SIMUSCOP_TIMING"))
		fprintf(stderr, "[simuscop timing] reference upload / haplotype strings %.2f s, append+pack %.2f s, gc census (device, incl. bin enumeration %.2f s) %.2f s, "
		                "gc weights (host) %.2f s, read counts %.2f s, flat bins %.2f s, ssc_set_plan %.2f s (%lld bins)\n",
		        g_tm.build, g_tm.upload, g_tm.enumerate, g_tm.census, g_tm.gc, g_tm.counts, g_tm.flatten, g_tm.setPlan, (long long)bins.size());
	return 0;
}

}  // namespace sschost
