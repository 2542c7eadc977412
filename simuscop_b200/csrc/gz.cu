// gz.cu -- on-GPU gzip of the FASTQ blobs (SURVEY 8f rank 3: the step after the path is 197 GB of text over
// PCIe and disk).  Every ticket blob (32 records, ~10.6 KB per file) becomes one gzip member (RFC 1952) holding a
// single final DEFLATE block (RFC 1951) of literals only, coded with one dynamic Huffman table per plan: FASTQ has no
// long-range structure worth an LZ77 search on this path, and four bases + a handful of quality symbols code to
// ~2 bits per character.  The table is fitted on the host to a sample of the first batch and shared by all
// members, so the per-member cost is a ~60-byte block header.  Concatenated members are a valid .gz file
// (SeqWriter's plain files, lib/seqwriter/SeqWriter.cpp:41-54, remain the default output).
// Bytes absent from the sample still get codes, of 14-15 bits: a later blob full of them (a 64-byte name that is not in
// the sample, N-run qualities) can code to nearly twice its size.  So, as zlib does, a member whose coded form would be
// longer than its raw bytes + 23 is written as one stored block instead (gzip header, 0x01, LEN, NLEN, the raw bytes,
// CRC-32, ISIZE): no member exceeds its blob + 23 bytes.  The blobs come from either generation kernel, one per ticket of 32
// pairs: the fast kernel's are at most 32 x 612 = 19 584 bytes in a scratch pitch of 20 480 (interleaved, both mates: 39 168 in
// 40 960); the generic kernel's (gzip mode, RL up to 320) at most 32 worst-case records of the plan, 29 568 bytes at RL 320 with
// 64-byte names (interleaved 59 136), in a pitch of that + 31 rounded to 16 (api.cu, ticket_bytes): still within the 16-bit LEN
// of one stored block.  The member pitch is the blob pitch.
// BGZF (the "bgzf" option, DESIGN 13): the same member with FLG = FEXTRA and the 8-byte BC field after the 10-byte header, so
// the tables carry an 18-byte header in the prefix and the DEFLATE bits follow 64 bits later; the warp writes BSIZE (member
// length - 1) once the length is known.  A stored member is then raw + 31 bytes, and no block exceeds the 65 536 bytes BGZF
// allows (39 199 from the fast kernel, 59 167 from the generic kernel).
//
// Kernel: one warp per (ticket, file); interleaved output is one file (the second file's jobs have length 0).  A round takes 256 bytes (two 32-bit words per lane): LUT -> up to 2 x 60 bits
// per lane, warp scan of the bit counts, OR into a shared-memory round buffer (two buffers in turn: the one just
// written out is zeroed word by word as it is stored), coalesced store of the completed words.  CRC-32 (the gzip
// trailer) is computed on the fly without a second pass: lane l keeps the pure remainder of its strided word pairs
// (slice-by-4 tables), advanced by 256 bytes of zeros per round through four 256-entry tables of the linear map
// x^2048 mod P; the lanes are combined at the end with one GF(2) multiplication each.  Coded words past the scratch pitch
// are counted but not stored: such a member is always rewritten in the stored form.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdint>
#include <cstring>
#include <queue>
#include <vector>

#include "gz.h"

namespace ssc {

// ------------------------------------------------------------------------------------------------
// host: CRC-32 arithmetic (reflected, polynomial 0xEDB88320) and the Huffman table
// ------------------------------------------------------------------------------------------------
static const uint32_t GZ_POLY = 0xEDB88320u;

// a(x) * b(x) mod P, reflected representation (bit 31 = x^0), as zlib's multmodp
static uint32_t h_multmodp(uint32_t a, uint32_t b) {
	uint32_t m = 1u << 31, p = 0;
	for (;;) {
		if (a & m) {
			p ^= b;
			if ((a & (m - 1)) == 0) break;
		}
		m >>= 1;
		b = (b & 1) ? (b >> 1) ^ GZ_POLY : b >> 1;
	}
	return p;
}

// x^(8n) mod P
static uint32_t h_xpow8(uint64_t n) {
	uint32_t p = 1u << 31;              // x^0
	uint32_t sq = 1u << 23;             // x^8
	while (n) {
		if (n & 1) p = h_multmodp(sq, p);
		sq = h_multmodp(sq, sq);
		n >>= 1;
	}
	return p;
}

uint32_t gz_crc32_host(const uint8_t* p, size_t n) {
	static uint32_t T[256];
	static bool init = false;
	if (!init) {
		for (uint32_t i = 0; i < 256; i++) { uint32_t c = i; for (int k = 0; k < 8; k++) c = (c & 1) ? (c >> 1) ^ GZ_POLY : c >> 1; T[i] = c; }
		init = true;
	}
	uint32_t c = 0xFFFFFFFFu;
	for (size_t i = 0; i < n; i++) c = T[(c ^ p[i]) & 0xff] ^ (c >> 8);
	return c ^ 0xFFFFFFFFu;
}

namespace {

// length-limited Huffman code lengths (<= maxLen) for n symbols with freq > 0; classic heap Huffman, frequencies are
// flattened (f -> f/2 + 1) until the tree is shallow enough
void huff_lengths(const std::vector<uint64_t>& freq, int maxLen, std::vector<int>& len) {
	const int n = (int)freq.size();
	std::vector<uint64_t> f(freq);
	len.assign(n, 0);
	for (;;) {
		struct Node { uint64_t w; int id; };
		auto cmp = [](const Node& a, const Node& b) { return a.w > b.w || (a.w == b.w && a.id > b.id); };
		std::priority_queue<Node, std::vector<Node>, decltype(cmp)> pq(cmp);
		std::vector<int> parent(2 * n, -1);
		int used = 0;
		for (int i = 0; i < n; i++) if (f[i] > 0) { pq.push({f[i], i}); used++; }
		if (used == 1) { for (int i = 0; i < n; i++) len[i] = f[i] > 0 ? 1 : 0; return; }
		int next = n;
		while (pq.size() > 1) {
			Node a = pq.top(); pq.pop();
			Node b = pq.top(); pq.pop();
			parent[a.id] = next; parent[b.id] = next;
			pq.push({a.w + b.w, next});
			next++;
		}
		int deepest = 0;
		for (int i = 0; i < n; i++) {
			if (f[i] == 0) { len[i] = 0; continue; }
			int d = 0;
			for (int v = i; parent[v] >= 0; v = parent[v]) d++;
			len[i] = d;
			deepest = std::max(deepest, d);
		}
		if (deepest <= maxLen) return;
		for (int i = 0; i < n; i++) if (f[i] > 0) f[i] = f[i] / 2 + 1;
	}
}

// canonical DEFLATE codes (RFC 1951 3.2.2), returned bit-reversed (the stream is filled from the least significant bit)
void canonical_codes(const std::vector<int>& len, std::vector<uint32_t>& code) {
	int maxLen = 0;
	for (int l : len) maxLen = std::max(maxLen, l);
	std::vector<int> blCount(maxLen + 2, 0), nextCode(maxLen + 2, 0);
	for (int l : len) if (l) blCount[l]++;
	int c = 0;
	for (int b = 1; b <= maxLen; b++) { c = (c + blCount[b - 1]) << 1; nextCode[b] = c; }
	code.assign(len.size(), 0);
	for (size_t i = 0; i < len.size(); i++) {
		if (!len[i]) continue;
		uint32_t v = (uint32_t)nextCode[len[i]]++, r = 0;
		for (int k = 0; k < len[i]; k++) r |= ((v >> k) & 1u) << (len[i] - 1 - k);
		code[i] = r;
	}
}

struct BitWriter {
	std::vector<uint32_t> w;
	uint32_t bits = 0;
	void put(uint32_t v, int n) {          // n <= 24, LSB first
		for (int i = 0; i < n; i++) {
			if ((bits >> 5) >= w.size()) w.push_back(0);
			w[bits >> 5] |= ((v >> i) & 1u) << (bits & 31);
			bits++;
		}
	}
};

}  // namespace

const char* gz_build_tables(const uint64_t hist[256], GzTables* t, bool bgzf) {
	memset(t, 0, sizeof(*t));
	// ---- literal/length code: all 256 byte values stay encodable (a population name may hold any byte), + end of block
	std::vector<uint64_t> freq(257);
	for (int i = 0; i < 256; i++) freq[i] = hist[i] * 16 + 1;
	freq[256] = 1;
	std::vector<int> len;
	huff_lengths(freq, 15, len);
	std::vector<uint32_t> code;
	canonical_codes(len, code);
	for (int i = 0; i < 257; i++) t->lut[i] = code[i] | ((uint32_t)len[i] << 16);

	// ---- gzip member header (RFC 1952) + dynamic block header (RFC 1951 3.2.7)
	BitWriter bw;
	// BGZF: FLG = FEXTRA and the 8-byte extra field (XLEN 6, SI1 'B', SI2 'C', SLEN 2, BSIZE) after the 10 bytes; the encoder
	// writes BSIZE (block length - 1) once it knows the length
	const uint8_t gzh[18] = {0x1f, 0x8b, 8, (uint8_t)(bgzf ? 4 : 0), 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0, 0, 0};
	t->headerBytes = bgzf ? 18 : 10;
	for (uint32_t i = 0; i < t->headerBytes; i++) bw.put(gzh[i], 8);
	bw.put(1, 1);                          // BFINAL
	bw.put(2, 2);                          // BTYPE = dynamic Huffman
	// code length sequence: 257 literal/length lengths + 2 distance lengths of 1 (never used: the block is all literals;
	// two one-bit codes are what zlib itself sends in that case, the form every inflater accepts)
	std::vector<int> seq(len.begin(), len.end());
	seq.push_back(1); seq.push_back(1);
	// run-length encode with symbols 16 (repeat previous 3..6), 17 (zeros 3..10), 18 (zeros 11..138)
	std::vector<std::pair<int, int>> rle;   // (symbol, extra value)
	for (size_t i = 0; i < seq.size();) {
		size_t j = i;
		while (j < seq.size() && seq[j] == seq[i]) j++;
		size_t run = j - i;
		if (seq[i] == 0) {
			while (run >= 11) { size_t r = std::min<size_t>(run, 138); rle.push_back({18, (int)r - 11}); run -= r; }
			if (run >= 3) { rle.push_back({17, (int)run - 3}); run = 0; }
			while (run--) rle.push_back({0, 0});
		} else {
			rle.push_back({seq[i], 0}); run--;
			while (run >= 3) { size_t r = std::min<size_t>(run, 6); rle.push_back({16, (int)r - 3}); run -= r; }
			while (run--) rle.push_back({seq[i], 0});
		}
		i = j;
	}
	std::vector<uint64_t> clFreq(19, 0);
	for (auto& p : rle) clFreq[p.first]++;
	std::vector<int> clLen;
	huff_lengths(clFreq, 7, clLen);
	std::vector<uint32_t> clCode;
	canonical_codes(clLen, clCode);
	static const int order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
	int hclen = 19;
	while (hclen > 4 && clLen[order[hclen - 1]] == 0) hclen--;
	bw.put(257 - 257, 5);                  // HLIT
	bw.put(2 - 1, 5);                      // HDIST
	bw.put((uint32_t)(hclen - 4), 4);      // HCLEN
	for (int i = 0; i < hclen; i++) bw.put((uint32_t)clLen[order[i]], 3);
	for (auto& p : rle) {
		bw.put(clCode[p.first], clLen[p.first]);
		if (p.first == 16) bw.put((uint32_t)p.second, 2);
		else if (p.first == 17) bw.put((uint32_t)p.second, 3);
		else if (p.first == 18) bw.put((uint32_t)p.second, 7);
	}
	if (bw.w.size() > GZ_PREFIX_WORDS) return "gzip block header too long";
	for (size_t i = 0; i < bw.w.size(); i++) t->prefix[i] = bw.w[i];
	t->prefixBits = bw.bits;

	// ---- CRC tables
	for (uint32_t i = 0; i < 256; i++) { uint32_t c = i; for (int k = 0; k < 8; k++) c = (c & 1) ? (c >> 1) ^ GZ_POLY : c >> 1; t->crcT[0][i] = c; }
	for (int k = 1; k < 4; k++)
		for (uint32_t i = 0; i < 256; i++) t->crcT[k][i] = t->crcT[0][t->crcT[k - 1][i] & 0xff] ^ (t->crcT[k - 1][i] >> 8);
	const uint32_t x2048 = h_xpow8(256);                 // advance a remainder by 256 zero bytes
	for (int k = 0; k < 4; k++)
		for (uint32_t i = 0; i < 256; i++) t->crcS[k][i] = h_multmodp(x2048, i << (8 * k));
	for (uint32_t n = 0; n < 256; n++) t->xp[n] = h_xpow8(n);
	return "";
}

// Host mirror of deflate_blobs_kernel for one blob (same tables, same lane-strided CRC arithmetic, same bit packing, same
// choice between the coded and the stored form): lets the table construction and the CRC algebra be checked against zlib
// without a GPU, and the kernel's members byte for byte.  Returns the member size, or 0 when it does not fit cap.
size_t gz_member_host(const GzTables* t, const uint8_t* src, uint32_t len, uint8_t* dst, size_t cap) {
	if (len == 0 || len > 0xFFFFu) return 0;
	const uint32_t hb = t->headerBytes;                   // 10, or 18 for a BGZF block
	const size_t storedExtra = hb + 13;                   // GZ_STORED_EXTRA or GZ_BGZF_STORED_EXTRA
	if (hb > 10 && (size_t)len + storedExtra > (size_t)GZ_BGZF_MAX_BLOCK) return 0;   // a block might not fit its 16-bit BSIZE
	std::vector<uint32_t> out(t->prefix, t->prefix + ((t->prefixBits + 31) >> 5));
	uint64_t bits = t->prefixBits;
	auto put = [&](uint64_t v, uint32_t n) {
		for (uint32_t i = 0; i < n; i++, bits++) {
			if ((bits >> 5) >= out.size()) out.push_back(0);
			out[bits >> 5] |= (uint32_t)((v >> i) & 1u) << (bits & 31);
		}
	};
	if (t->prefixBits & 31u) out.back() &= (1u << (t->prefixBits & 31u)) - 1u;
	const uint32_t W = len >> 2, P2 = W >> 1;          // full word pairs; an odd last word goes with the tail bytes
	uint32_t A[32], last[32];
	for (int l = 0; l < 32; l++) { A[l] = 0; last[l] = 0xFFFFFFFFu; }
	auto step = [&](uint32_t c) { return t->crcT[3][c & 0xff] ^ t->crcT[2][(c >> 8) & 0xff] ^ t->crcT[1][(c >> 16) & 0xff] ^ t->crcT[0][c >> 24]; };
	for (uint32_t pi = 0; pi < P2; pi++) {
		uint32_t w0, w1; memcpy(&w0, src + 8 * (size_t)pi, 4); memcpy(&w1, src + 8 * (size_t)pi + 4, 4);
		const int l = pi & 31;
		uint32_t c = A[l];
		c = t->crcS[0][c & 0xff] ^ t->crcS[1][(c >> 8) & 0xff] ^ t->crcS[2][(c >> 16) & 0xff] ^ t->crcS[3][c >> 24];
		A[l] = c ^ step(step(pi == 0 ? ~w0 : w0) ^ w1);
		last[l] = pi;
		for (int k = 0; k < 4; k++) { const uint32_t e = t->lut[(w0 >> (8 * k)) & 0xff]; put(e & 0xffffu, e >> 16); }
		for (int k = 0; k < 4; k++) { const uint32_t e = t->lut[(w1 >> (8 * k)) & 0xff]; put(e & 0xffffu, e >> 16); }
	}
	uint32_t crc = 0;
	for (int l = 0; l < 32; l++) if (last[l] != 0xFFFFFFFFu) crc ^= h_multmodp(t->xp[(P2 - 1 - last[l]) * 8], A[l]);
	if (P2 == 0) crc = 0xFFFFFFFFu;                      // fewer than 8 bytes: plain byte-wise CRC from the initial value
	for (uint32_t i = P2 * 8; i < len; i++) { crc = t->crcT[0][(crc ^ src[i]) & 0xff] ^ (crc >> 8); const uint32_t e = t->lut[src[i]]; put(e & 0xffffu, e >> 16); }
	crc = ~crc;
	put(t->lut[256] & 0xffffu, t->lut[256] >> 16);
	while (bits & 7) put(0, 1);
	put(crc, 32); put(len, 32);
	size_t n = (size_t)(bits >> 3);
	if (n > (size_t)len + storedExtra) {                  // coding would expand the blob: one stored block
		if ((size_t)len + storedExtra > cap) return 0;
		memcpy(dst, out.data(), hb);                      // the gzip header of the coded form
		const uint8_t blk[5] = {0x01, (uint8_t)len, (uint8_t)(len >> 8), (uint8_t)~len, (uint8_t)(~len >> 8)};
		memcpy(dst + hb, blk, 5);
		memcpy(dst + hb + 5, src, len);
		for (int k = 0; k < 4; k++) { dst[hb + 5 + len + k] = (uint8_t)(crc >> (8 * k)); dst[hb + 9 + len + k] = (uint8_t)(len >> (8 * k)); }
		n = (size_t)len + storedExtra;
	} else {
		if (n > cap) return 0;
		memcpy(dst, out.data(), n);
	}
	if (hb > 10) { dst[16] = (uint8_t)(n - 1); dst[17] = (uint8_t)((n - 1) >> 8); }   // BSIZE
	return n;
}

// ------------------------------------------------------------------------------------------------
// device
// ------------------------------------------------------------------------------------------------
static constexpr int GZ_WARPS = 8;
static constexpr int GZ_RB = 128;           // round buffer words: 31 carry bits + 32 lanes * 120 bits < 122 words (+ the trailer round)

__device__ __forceinline__ uint32_t d_multmodp(uint32_t a, uint32_t b) {
	uint32_t p = 0;
#pragma unroll 4
	for (int i = 31; i >= 0; i--) {
		if ((a >> i) & 1u) p ^= b;
		b = (b & 1u) ? (b >> 1) ^ 0xEDB88320u : b >> 1;
	}
	return p;
}

// OR the low n (<= 64) bits of v into the bit stream buf at bit offset off
__device__ __forceinline__ void put_bits(uint32_t* buf, uint32_t off, unsigned long long v, uint32_t n) {
	if (n == 0) return;
	const uint32_t w0 = off >> 5, s = off & 31u;
	const uint32_t lo = (uint32_t)v, hi = (uint32_t)(v >> 32);
	atomicOr(&buf[w0], lo << s);
	if (s + n > 32) atomicOr(&buf[w0 + 1], __funnelshift_l(lo, hi, s));
	if (s + n > 64) atomicOr(&buf[w0 + 2], s ? (hi >> (32 - s)) : 0u);
}

__global__ void __launch_bounds__(GZ_WARPS * 32) deflate_blobs_kernel(const uint8_t* __restrict__ raw1, const uint8_t* __restrict__ raw2,
                                                                      const unsigned long long* __restrict__ rawLens, int nTiles, uint32_t rawPitch,
                                                                      uint8_t* __restrict__ gz1, uint8_t* __restrict__ gz2,
                                                                      unsigned long long* __restrict__ gzLens, uint32_t gzPitch,
                                                                      const GzTables* __restrict__ tab) {
	__shared__ uint32_t s_lut[257];
	__shared__ uint32_t s_T[4][256];
	__shared__ uint32_t s_S[4][256];
	__shared__ uint32_t s_xp[256];
	__shared__ uint32_t s_prefix[GZ_PREFIX_WORDS];
	__shared__ uint32_t s_rb[GZ_WARPS][2][GZ_RB];
	for (int i = threadIdx.x; i < 257; i += blockDim.x) s_lut[i] = tab->lut[i];
	for (int i = threadIdx.x; i < 1024; i += blockDim.x) { (&s_T[0][0])[i] = (&tab->crcT[0][0])[i]; (&s_S[0][0])[i] = (&tab->crcS[0][0])[i]; }
	for (int i = threadIdx.x; i < 256; i += blockDim.x) s_xp[i] = tab->xp[i];
	for (int i = threadIdx.x; i < GZ_PREFIX_WORDS; i += blockDim.x) s_prefix[i] = tab->prefix[i];
	for (int i = threadIdx.x; i < GZ_WARPS * 2 * GZ_RB; i += blockDim.x) (&s_rb[0][0][0])[i] = 0u;
	__syncthreads();
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	uint32_t* rbA = s_rb[warp][0];              // buffer of the current round: all zero except its first word (the carry)
	uint32_t* rbB = s_rb[warp][1];              // all zero
	const uint32_t prefixBits = tab->prefixBits;
	const uint32_t hdrBytes = tab->headerBytes;          // 10, or 18 for a BGZF block
	const uint32_t storedExtra = hdrBytes + 13u;         // GZ_STORED_EXTRA or GZ_BGZF_STORED_EXTRA
	const int nWarps = gridDim.x * GZ_WARPS;
	auto crc_step = [&](uint32_t c) { return s_T[3][c & 0xff] ^ s_T[2][(c >> 8) & 0xff] ^ s_T[1][(c >> 16) & 0xff] ^ s_T[0][c >> 24]; };
	for (int job = blockIdx.x * GZ_WARPS + warp; job < 2 * nTiles; job += nWarps) {
		const int ticket = job >> 1, file = job & 1;
		const unsigned long long lens = rawLens[ticket];
		const uint32_t len = file ? (uint32_t)(lens & 0x7fffffffull) : (uint32_t)(lens >> 31);
		uint32_t outBytes = 0;
		if (len > 0) {
			const uint2* src64 = (const uint2*)((file ? raw2 : raw1) + (size_t)ticket * rawPitch);
			const uint8_t* src8 = (const uint8_t*)src64;
			uint32_t* dst32 = (uint32_t*)((file ? gz2 : gz1) + (size_t)ticket * gzPitch);
			const uint32_t pitchWords = gzPitch >> 2;     // coded words past it are counted, not stored (the member goes stored)
			// ---- member header + block header
			uint32_t outWords = prefixBits >> 5, carryBits = prefixBits & 31u;
			for (uint32_t i = lane; i < outWords; i += 32) dst32[i] = s_prefix[i];
			if (lane == 0) rbA[0] = carryBits ? (s_prefix[outWords] & ((1u << carryBits) - 1u)) : 0u;
			__syncwarp();
			// ---- the word pairs of the blob
			const uint32_t P2 = len >> 3;
			uint32_t A = 0, lastIdx = 0xFFFFFFFFu;
			for (uint32_t base = 0; base < P2; base += 32) {
				const uint32_t idx = base + lane;
				const bool valid = idx < P2;
				unsigned long long acc0 = 0, acc1 = 0;
				uint32_t n0 = 0, n1 = 0;
				if (valid) {
					const uint2 wv = src64[idx];
					// CRC: pure remainder of this lane's strided word pairs; the 0xFFFFFFFF initial value = inverting the first word
					uint32_t c = A;
					c = s_S[0][c & 0xff] ^ s_S[1][(c >> 8) & 0xff] ^ s_S[2][(c >> 16) & 0xff] ^ s_S[3][c >> 24];
					A = c ^ crc_step(crc_step(idx == 0 ? ~wv.x : wv.x) ^ wv.y);
					lastIdx = idx;
#pragma unroll
					for (int k = 0; k < 4; k++) {
						const uint32_t e = s_lut[(wv.x >> (8 * k)) & 0xffu];
						acc0 |= (unsigned long long)(e & 0xffffu) << n0;
						n0 += e >> 16;
					}
#pragma unroll
					for (int k = 0; k < 4; k++) {
						const uint32_t e = s_lut[(wv.y >> (8 * k)) & 0xffu];
						acc1 |= (unsigned long long)(e & 0xffffu) << n1;
						n1 += e >> 16;
					}
				}
				const uint32_t n = n0 + n1;
				uint32_t incl = n;
#pragma unroll
				for (int d = 1; d < 32; d <<= 1) { const uint32_t o = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += o; }
				const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
				const uint32_t off = carryBits + incl - n;
				put_bits(rbA, off, acc0, n0);
				put_bits(rbA, off + n0, acc1, n1);
				__syncwarp();
				const uint32_t totalBits = carryBits + total, nw = totalBits >> 5;
				// store the completed words, zero them, and move the partial last word to the other (all zero) buffer
				for (uint32_t i = lane; i <= nw; i += 32) {
					const uint32_t v = rbA[i];
					rbA[i] = 0u;
					if (i < nw) { if (outWords + i < pitchWords) dst32[outWords + i] = v; } else rbB[0] = v;
				}
				__syncwarp();
				{ uint32_t* tswap = rbA; rbA = rbB; rbB = tswap; }
				carryBits = totalBits & 31u;
				outWords += nw;
			}
			// ---- CRC of the whole blob
			uint32_t part = lastIdx != 0xFFFFFFFFu ? d_multmodp(s_xp[(P2 - 1u - lastIdx) * 8u], A) : 0u;   // advance to the last pair
#pragma unroll
			for (int d = 16; d > 0; d >>= 1) part ^= __shfl_xor_sync(0xffffffffu, part, d);
			uint32_t crc = P2 ? part : 0xFFFFFFFFu;       // fewer than 8 bytes: plain byte-wise CRC from the initial value
			for (uint32_t i = P2 * 8u; i < len; i++) crc = s_T[0][(crc ^ src8[i]) & 0xff] ^ (crc >> 8);
			crc = ~crc;
			// ---- tail bytes (< 8), end of block, byte alignment, trailer (CRC32, ISIZE)
			unsigned long long accA = 0, accB = 0;
			uint32_t nA = 0, nB = 0;
			for (uint32_t i = P2 * 8u; i < len; i++) {
				const uint32_t e = s_lut[src8[i]];
				if (i < P2 * 8u + 4u) { accA |= (unsigned long long)(e & 0xffffu) << nA; nA += e >> 16; }
				else { accB |= (unsigned long long)(e & 0xffffu) << nB; nB += e >> 16; }
			}
			{ const uint32_t e = s_lut[256]; accB |= (unsigned long long)(e & 0xffffu) << nB; nB += e >> 16; }   // <= 3 literals + end of block
			const uint32_t dataEnd = carryBits + nA + nB;
			const uint32_t trailerAt = (dataEnd + 7u) & ~7u;
			if (lane == 0) { put_bits(rbA, carryBits, accA, nA); put_bits(rbA, carryBits + nA, accB, nB); }
			if (lane == 1) put_bits(rbA, trailerAt, (unsigned long long)crc | ((unsigned long long)len << 32), 64);
			__syncwarp();
			const uint32_t totalBits = trailerAt + 64u;
			const uint32_t nw = (totalBits + 31u) >> 5;
			for (uint32_t i = lane; i < nw; i += 32) { if (outWords + i < pitchWords) dst32[outWords + i] = rbA[i]; rbA[i] = 0u; }
			outBytes = outWords * 4u + (totalBits >> 3);
			__syncwarp();
			if (outBytes > len + storedExtra) {
				// coding would expand the blob (bytes the table was not fitted to): one stored block, as gz_member_host
				uint8_t* dst8 = (uint8_t*)dst32;
				const uint32_t h = hdrBytes;
				for (uint32_t i = lane; i < len + storedExtra; i += 32) {
					uint32_t b;
					if (i < h) b = s_prefix[i >> 2] >> (8u * (i & 3u));                              // the gzip header of the coded form
					else if (i == h) b = 1u;                                                      // BFINAL, BTYPE = stored
					else if (i < h + 5u) b = (i < h + 3u ? len : ~len) >> (8u * ((i - h - 1u) & 1u));   // LEN, NLEN
					else if (i < h + 5u + len) b = src8[i - h - 5u];
					else b = (i < h + 9u + len ? crc : len) >> (8u * ((i - h - 5u - len) & 3u));  // CRC-32, ISIZE
					dst8[i] = (uint8_t)b;
				}
				outBytes = len + storedExtra;
				__syncwarp();
			}
			if (hdrBytes > 10u && lane == 0) {
				// BGZF: BSIZE = block length - 1, over the 0 of the prefix (its word was stored before the last __syncwarp)
				uint8_t* dst8 = (uint8_t*)dst32;
				dst8[16] = (uint8_t)(outBytes - 1u);
				dst8[17] = (uint8_t)((outBytes - 1u) >> 8);
			}
		}
		if (lane == 0) {
			// the two files of a ticket are different jobs: each adds its own half of the packed length (zeroed by the host)
			atomicAdd(gzLens + ticket, file ? (unsigned long long)outBytes : ((unsigned long long)outBytes << 31));
		}
	}
}

cudaError_t launch_deflate_blobs(const uint8_t* raw1, const uint8_t* raw2, const unsigned long long* rawLens, int nTiles, uint32_t rawPitch,
                                 uint8_t* gz1, uint8_t* gz2, unsigned long long* gzLens, uint32_t gzPitch, const GzTables* tab,
                                 int smCount, cudaStream_t stream) {
	if (nTiles <= 0) return cudaSuccess;
	int grid = smCount * 6;
	const int need = (2 * nTiles + GZ_WARPS - 1) / GZ_WARPS;
	if (grid > need) grid = need;
	deflate_blobs_kernel<<<grid, GZ_WARPS * 32, 0, stream>>>(raw1, raw2, rawLens, nTiles, rawPitch, gz1, gz2, gzLens, gzPitch, tab);
	return cudaGetLastError();
}

}  // namespace ssc
