// bz_decode.cu -- bzip2 block decoder for sm_100a.
//
// Replaces BZ2_bzBuffToBuffDecompress(dst,&n,src,len,0,0) as called per KLB block by
// klb_imageIO::blockUncompressor{,ImageFull} (src/klb_imageIO.cpp:627, :1034) plus the scatter of the block into
// the image (:673-746, :1080-1125):
//   k_decode      stream/block header, coding tables, Huffman decode, inverse MTF, RUNA/RUNB expansion
//                 (decompress.c:196-487, huffman.c:170-205)            -> last column L + symbol counts
//   k_inv_bwt     inverse BWT: stable counting sort = LF mapping (decompress.c:494-573), then the n-step walk is
//                 cut at splitters and walked by 1024 threads in parallel (list ranking by sampling)
//   k_unrle       inverse of the initial run-length coding + CRC check (bzlib.c:561-728) fused with the scatter
//                 of the block into the symbol image
#include "lfm_radix.cuh"
#include "bz_randtable.h"
#include "bz_rle1.cuh"
#include <algorithm>
#include <cstdlib>

namespace lfm {

__device__ const uint16_t kRNums[512] = BZ_RNUMS_INIT;

// =====================================================================================================
// k_huff_decode : one warp per KLB block stream -- ONLY the inherently sequential part.
//   * the compressed stream is staged through a shared-memory ring of big-endian words (coalesced copies by the warp);
//   * every lane runs the same (uniform) parser, so nothing has to be broadcast;
//   * a 64-bit bit buffer lives in registers; symbols of <= DEC_LB bits come out of a per-table lookup (one shared
//     load per symbol on the critical path); longer ones use bzip2's limit/base/perm walk (decompress.c GET_MTF_VAL);
//   * a group of 50 symbols (RUNA/RUNB/rank+1/EOB) is decoded straight through -- three symbols per refill, no branch per
//     symbol -- staged in shared memory and stored with two coalesced stores (details at the symbol loop below).
// Inverse move-to-front and run expansion are done in parallel by k_imtf.
// =====================================================================================================
// lookup bits of the per-table code table: 10 when every stream is resident at once (a lone stream decodes 16-22 % faster with 10
// bits: fewer codes take the long-code walk), 9 when the streams outnumber the warp slots that shared memory leaves (12 KB -> 6 KB
// of tables per warp: 10 -> 15 warps per SM at 147 KB blocks); chosen per launch, launch_decode()

template <int DEC_LB>
struct DecWarpSmemT {
	uint16_t lut[kGroups][1 << DEC_LB];              // len | sym << 5   (0: longer than DEC_LB bits)
	int32_t  limit[kGroups][24];
	int32_t  base[kGroups][24];
	uint16_t perm[kGroups][kMaxAlpha + 2];
	uint8_t  len[kGroups][kMaxAlpha + 2];
	int32_t  minlen[kGroups];
};

constexpr uint32_t DEC_RING = 256;               // staged stream words per warp (power of two)
constexpr uint32_t DEC_OUT = 128;                // staged output symbols per warp (power of two)
// selectors are kept as nibbles: shared memory per warp decides how many streams an SM decodes at once (the decoder is
// pure latency: ~100 cycles per symbol and warp): ~21 KB per warp for 147 KB blocks -> 10 warps per SM
__host__ __device__ inline size_t dec_sel_bytes(uint32_t selcap) { return (((size_t)selcap + 1) / 2 + 15) & ~(size_t)15; }

extern __shared__ __align__(16) uint8_t dec_smem[];

// SINGLE (standalone streams, bz_stream.cu): job = ONE bzip2 block that starts at bit begin[job] of the payload (its block magic),
// no stream header; the level bound comes from job_level[job] (9 when NULL); end[0] = payload bytes.  The bit after the block's
// last symbol goes to endbit[job] (~0 when the block does not decode), its stored CRC to crc_out[job].
template <int DEC_LB, bool SINGLE>
__global__ void __launch_bounds__(256)
k_huff_decode(const uint8_t* __restrict__ payload, const uint64_t* __restrict__ begin, const uint64_t* __restrict__ end,
              uint32_t njobs, DecJob* __restrict__ jobs, uint16_t* __restrict__ mtfv_all, uint32_t mcap, uint32_t cap,
              uint32_t selcap, uint32_t nsub, uint64_t* __restrict__ endbit, uint32_t* __restrict__ crc_out,
              const uint32_t* __restrict__ job_level)
{
	const uint32_t lane = lane_id(), w = warp_id(), nw = blockDim.x >> 5;
	const uint32_t job = blockIdx.x * nw + w;
	if (job >= njobs) return;
	using DecWarpSmem = DecWarpSmemT<DEC_LB>;
	constexpr int DEC_LUT = 1 << DEC_LB;
	const size_t per_warp = sizeof(DecWarpSmem) + dec_sel_bytes(selcap) + (size_t)DEC_RING * 4 + (size_t)DEC_OUT * 2;
	DecWarpSmem& S = *reinterpret_cast<DecWarpSmem*>(dec_smem + (size_t)w * per_warp);
	uint8_t* selector = dec_smem + (size_t)w * per_warp + sizeof(DecWarpSmem);
	uint32_t* sw = reinterpret_cast<uint32_t*>(selector + dec_sel_bytes(selcap));
	uint16_t* so = reinterpret_cast<uint16_t*>(sw + DEC_RING);           // decoded symbols, flushed 32 at a time
	// the stream's bzip2 blocks go to records job * nsub + kb (kb = 0, 1, ...); errors are reported in record 0
	DecJob& J0 = jobs[(size_t)job * nsub];
	const uint64_t beg = SINGLE ? (begin[job] >> 3) : begin[job];
	const uint8_t* src = payload + beg;
	const uint64_t nbytes = end[SINGLE ? 0 : job] - beg;
	#define FAIL(code) do { if (lane == 0) { J0.status = (code); J0.n = 0; J0.n_mtf = 0; if (SINGLE) endbit[job] = ~0ull; } return; } while (0)
	for (uint32_t k = lane; k < nsub; k += 32) {
		DecJob& Jk = jobs[(size_t)job * nsub + k];
		Jk.n = 0; Jk.n_mtf = 0; Jk.out_bytes = 0; Jk.orig_ptr = 0; Jk.stored_crc = 0; Jk.status = 0; Jk.flags = kSubUnused; Jk.level = 0; Jk.max_block = 0;
	}
	__syncwarp();

	// ---- the stream is staged through a ring of big-endian words: word i = bytes 4i..4i+3, zero past the end
	const uint32_t nwords = (uint32_t)((nbytes + 3) / 4);
	const uint32_t mis = (uint32_t)((uintptr_t)src & 3);
	const uint32_t* a32 = reinterpret_cast<const uint32_t*>(src - mis);       // payload base is 256-byte aligned: never below it
	auto load_word = [&](uint32_t i) -> uint32_t {
		const uint64_t b0 = (uint64_t)i * 4;
		uint32_t v = 0;
		if (b0 + 8 <= nbytes) {                           // bulk: two aligned words cover stream bytes 4i .. 4i+3
			uint32_t lo = a32[i], hi = a32[i + 1];
			v = mis ? __funnelshift_r(lo, hi, mis * 8) : lo;
			v = __byte_perm(v, 0, 0x0123);
		} else if (b0 < nbytes) {                         // tail: byte by byte
			#pragma unroll
			for (int k = 0; k < 4; k++) v = (v << 8) | (b0 + k < nbytes ? (uint32_t)src[b0 + k] : 0u);
		}
		return v;
	};
	uint32_t staged_end = 0, wi = 0;                       // words [wi, staged_end) are in the ring, not yet consumed
	auto top_up = [&]() {                                  // uniform; never overwrites an unconsumed word
		while (staged_end + 32 <= wi + DEC_RING) { sw[(staged_end + lane) & (DEC_RING - 1)] = load_word(staged_end + lane); staged_end += 32; }
		__syncwarp();
	};
	top_up();

	// ---- uniform bit reader: bb holds bc >= 32 valid bits, left aligned (zeros below them); nxt = ring word wi, already
	// in a register, so a refill is two shifts and an OR on the critical path and the shared load of the following word
	// overlaps the next symbols
	uint64_t bb = ((uint64_t)sw[0] << 32) | sw[1];
	uint32_t bc = 64; wi = 2;
	uint32_t nxt = sw[2];
	const uint32_t wi_limit = nwords + 4;                  // a well-formed stream never needs words beyond this
	auto drop = [&](uint32_t nb) {                         // nb <= 32
		bb <<= nb; bc -= nb;
		if (bc < 32) { bb |= (uint64_t)nxt << (32 - bc); bc += 32; wi++; nxt = sw[wi & (DEC_RING - 1)]; }
	};
	auto peek = [&](uint32_t nb) -> uint32_t { return (uint32_t)(bb >> (64 - nb)); };
	auto get = [&](uint32_t nb) -> uint32_t { uint32_t v = peek(nb); drop(nb); return v; };

	int level;
	if (SINGLE) {
		drop((uint32_t)(begin[job] & 7u));
		level = job_level ? (int)job_level[job] : 9;
	} else {
		if (get(8) != 'B' || get(8) != 'Z' || get(8) != 'h') FAIL(1);
		level = (int)get(8) - '0';
		if (level < 1 || level > 9) FAIL(1);
	}
	const uint32_t max_block = min((uint32_t)(100000 * level), cap);
	uint32_t m1 = get(24), m2 = get(24);
	uint32_t combined = 0, kb = 0;
	for (;; kb++) {                                        // one bzip2 block per iteration (decompress.c:196-487)
	if (SINGLE && (m1 != 0x314159 || m2 != 0x265359)) FAIL(1);
	if (m1 == 0x177245 && m2 == 0x385090) break;           // end of stream
	if (m1 != 0x314159 || m2 != 0x265359) FAIL(2);
	if (kb >= nsub) FAIL(4);                               // more blocks than this block geometry can produce
	DecJob& J = jobs[(size_t)job * nsub + kb];
	uint16_t* mtfv = mtfv_all + ((size_t)job * nsub + kb) * mcap;
	const uint32_t stored_crc = get(32);
	const uint32_t randomised = get(1);                    // never produced since bzip2 0.9.5 (compress.c:629), still legal to read
	const uint32_t orig_ptr = get(24);
	uint32_t iu[8] = { 0, 0, 0, 0, 0, 0, 0, 0 };
	uint32_t n_in_use = 0;
	{
		uint32_t used16 = get(16);
		for (int i = 0; i < 16; i++) if (used16 & (0x8000u >> i)) {
			uint32_t bits = get(16);
			uint32_t rev = __brev(bits) >> 16;             // bit j <-> byte value 16 i + j
			#pragma unroll
			for (int k = 0; k < 8; k++) if ((i >> 1) == k) iu[k] |= rev << ((i & 1) * 16);
			n_in_use += __popc(bits);
		}
	}
	if (n_in_use == 0) FAIL(2);
	const int alpha = (int)n_in_use + 2;
	const int n_groups = (int)get(3);
	const int n_sel = (int)get(15);
	if (n_groups < 2 || n_groups > 6 || n_sel < 1) FAIL(2);
	// all n_sel (<= 32767) selectors are read, as libbz2 1.0.8 does; only the first selcap are kept (more than any block of this
	// slot geometry can use: other encoders may round the count up), and a group past them is corrupt (decompress.c:287-300)
	const int n_sel_kept = min(n_sel, (int)selcap);
	{
		uint32_t pos = 0x543210u;                          // 6 nibbles: move-to-front list of table ids
		for (int i = 0; i < n_sel; i++) {
			if ((i & 63) == 0) { top_up(); if (wi > wi_limit) FAIL(2); }
			uint32_t v = peek(6);                          // unary: count leading ones (at most n_groups-1)
			int j = __clz(~(v << 26));
			if (j >= n_groups) FAIL(2);
			drop((uint32_t)j + 1);
			uint32_t t = (pos >> (4 * j)) & 15u;
			uint32_t lowmask = (1u << (4 * j)) - 1u;
			pos = (pos & ~((lowmask << 4) | 15u)) | ((pos & lowmask) << 4) | t;
			if (lane == 0 && i < n_sel_kept) selector[i >> 1] = (i & 1) ? (uint8_t)((selector[i >> 1] & 15u) | (t << 4)) : (uint8_t)t;
		}
	}
	// code lengths (decompress.c:314-331): per symbol a run of (1, d) bit pairs -- d = 0: +1, d = 1: -1 -- closed by a 0 bit.  The
	// whole record is read from one 32-bit window without a loop: the closing bit is the first 0 at an even position, the deltas
	// are the odd bits before it.  The encoder only writes runs of equal deltas (compress.c:574-581), for which checking the length
	// before and after the run is bzip2's per-step range check; anything else (mixed deltas, more than 15 pairs) takes the
	// bit-by-bit loop.  Failures are collected and reported per table: no branch per symbol besides the loop itself.
	for (int t = 0; t < n_groups; t++) {
		int curr = (int)get(5);
		bool badlen = false;
		for (int i0 = 0; i0 < alpha; i0 += 16) {
			top_up(); if (wi > wi_limit) FAIL(2);
			const int i1 = min(alpha, i0 + 16);
			#pragma unroll 1
			for (int i = i0; i < i1; i++) {
				const uint32_t w = (uint32_t)(bb >> 32);
				const uint32_t z = ~w & 0xAAAAAAAAu;
				const uint32_t lz = (uint32_t)__clz((int)z);      // 2 * (number of pairs); 32: no closing bit in the window
				const uint32_t k = lz >> 1;
				const uint32_t ones = (uint32_t)__popc(w & 0x55555555u & ~__funnelshift_rc(0xFFFFFFFFu, 0u, lz));
				if (z == 0u || (ones != 0u && ones != k)) {          // rare: the reference loop
					for (;;) {
						if (curr < 1 || curr > 20) FAIL(2);
						uint32_t two = peek(2);
						if (!(two & 2)) { drop(1); break; }
						drop(2);
						curr += (two & 1) ? -1 : 1;
					}
				} else {
					badlen = badlen | (curr < 1) | (curr > 20);
					curr += (int)k - 2 * (int)ones;
					badlen = badlen | (curr < 1) | (curr > 20);
					const uint32_t nb = lz + 1u;                     // <= 31
					bb <<= nb; bc -= nb;
					const bool fill = bc < 32u;
					bb |= fill ? ((uint64_t)nxt << ((32u - bc) & 31u)) : 0ull;
					bc += fill ? 32u : 0u; wi += fill ? 1u : 0u;
					nxt = sw[wi & (DEC_RING - 1)];
				}
				if (lane == 0) S.len[t][i] = (uint8_t)curr;
			}
		}
		if (badlen) FAIL(2);
	}
	__syncwarp();
	// ---- decode tables: lane t builds table t (huffman.c:170-205 + the lookup)
	if ((int)lane < n_groups) {
		const int t = (int)lane;
		int mn = 32, mx = 0;
		int32_t* base = S.base[t]; int32_t* limit = S.limit[t];
		for (int i = 0; i < 24; i++) { base[i] = 0; limit[i] = 0; }
		for (int i = 0; i < alpha; i++) { int l = S.len[t][i]; mx = l > mx ? l : mx; mn = l < mn ? l : mn; base[l + 1]++; }
		for (int i = 1; i < 23; i++) base[i] += base[i - 1];
		{   // counting sort by length; the running positions live in limit[] (shared memory, filled in below) instead of a
			// thread-local array indexed by the length (local memory, or a chain of 24 selects per access)
			for (int i = 0; i < 24; i++) limit[i] = base[i];
			for (int i = 0; i < alpha; i++) { int l = S.len[t][i]; S.perm[t][limit[l]++] = (uint16_t)i; }
			for (int i = 0; i < 24; i++) limit[i] = 0;
		}
		// lookup: symbols in (length, symbol) order own consecutive, left-to-right ranges of the DEC_LB-bit code space
		{
			uint32_t fill = 0;
			for (int p = 0; p < alpha; p++) {
				int sym = S.perm[t][p], l = S.len[t][sym];
				if (l > DEC_LB) break;
				uint32_t span = 1u << (DEC_LB - l);
				uint16_t e = (uint16_t)(l | (sym << 5));
				for (uint32_t q = 0; q < span && fill + q < (uint32_t)DEC_LUT; q++) S.lut[t][fill + q] = e;
				fill += span;
			}
			for (; fill < (uint32_t)DEC_LUT; fill++) S.lut[t][fill] = 0;
		}
		int vec = 0;
		for (int i = mn; i <= mx; i++) { vec += base[i + 1] - base[i]; limit[i] = vec - 1; vec <<= 1; }
		for (int i = mn + 1; i <= mx; i++) base[i] = ((limit[i - 1] + 1) << 1) - base[i];
		S.minlen[t] = mn;
	}
	__syncwarp();
	top_up();

	// ---- symbols (decompress.c:349-487 without the MTF): append until EOB.  A lone warp is bound by the instructions it issues
	// (~4 cycles each), not by the lookup -> shift -> lookup chain, so the loop is written for the fewest instructions per symbol:
	//   * a group of 50 symbols is decoded straight through, six symbols per loop trip; the 64-bit bit buffer is refilled once
	//     per THREE symbols (>= 33 valid bits after a refill, a table code takes <= DEC_LB = 10);
	//   * no per-symbol end test: EOB is looked for once per group among the 50 staged symbols; the group that holds it (and a
	//     group with an invalid code) is decoded again from the saved reader state by the careful one-symbol-at-a-time loop,
	//     which stops at EOB and fails on invalid codes -- whatever the fast path decoded beyond EOB is discarded;
	//   * every lane stores the (uniform) symbol to the staging row: one STS with an immediate offset, no predicate;
	//   * a code longer than DEC_LB bits (table entry 0, ~1 % of the symbols) takes bzip2's limit/base/perm walk in line.
	const uint32_t EOB = n_in_use + 1;
	uint32_t nsym = 0;
	bool done = false;
	uint32_t hi = (uint32_t)(bb >> 32), lo = (uint32_t)bb;
	auto refill = [&]() {                                    // predicated: adds the next word when <= 32 bits are left (then lo is empty)
		const bool fill = bc <= 32u;
		const uint32_t add_hi = __funnelshift_rc(nxt, 0u, bc);             // nxt >> bc, 0 for bc == 32 (clamped shift)
		const uint32_t add_lo = nxt << ((32u - bc) & 31u);
		hi |= fill ? add_hi : 0u;
		lo = fill ? add_lo : lo;
		bc += fill ? 32u : 0u;
		wi += fill ? 1u : 0u;
		nxt = sw[wi & (DEC_RING - 1)];
	};
	for (int grp = 0; !done; grp++) {
		if (grp >= n_sel_kept) FAIL(2);
		const int t = (selector[grp >> 1] >> ((grp & 1) * 4)) & 15;
		if (t >= n_groups) FAIL(2);
		const uint16_t* lut = S.lut[t];
		const uint32_t hi0 = hi, lo0 = lo, bc0 = bc, wi0 = wi, nxt0 = nxt;          // reader state at the start of the group
		bool bad = false;
		// bzip2's limit/base/perm walk for ONE symbol (decompress.c GET_MTF_VAL); an invalid code only raises `bad` here
		auto long_symbol = [&]() -> uint32_t {
			refill();                                            // >= 33 bits: the walk looks at 20
			const uint32_t window = hi >> 12;
			const int32_t* limit = S.limit[t]; const int32_t* base = S.base[t];
			int zn = S.minlen[t];
			while (zn < 20 && (int32_t)(window >> (20 - zn)) > limit[zn]) zn++;
			const int32_t idx = (int32_t)(window >> (20 - zn)) - base[zn];
			bad = bad | ((int32_t)(window >> (20 - zn)) > limit[zn]) | (idx < 0) | (idx >= kMaxAlpha);
			const uint32_t sym = S.perm[t][bad ? 0 : idx];
			hi = __funnelshift_l(lo, hi, (uint32_t)zn); lo <<= zn; bc -= (uint32_t)zn;
			refill();                                            // the symbols after it in this run of three find >= 33 bits again
			return sym;
		};
		// a run of N <= 3 symbols after one refill, WITHOUT a branch per symbol: consuming table entry 0 (a long code) is a no-op,
		// so the run is decoded blindly and, if one of its entries was 0, decoded again with the long codes walked in line
		auto run = [&](uint16_t* dst, auto NC) {
			constexpr int N = decltype(NC)::value;
			refill();
			const uint32_t h0 = hi, l0 = lo, b0 = bc;
			uint32_t lowest = 0xffffffffu;
			#pragma unroll
			for (int i = 0; i < N; i++) {
				const uint32_t e = lut[hi >> (32 - DEC_LB)];      // len | sym << 5   (0: longer than DEC_LB bits)
				hi = __funnelshift_l(lo, hi, e); lo = __funnelshift_l(0u, lo, e); bc -= e & 31u;     // funnel shifts take their count modulo 32
				dst[i] = (uint16_t)(e >> 5);
				lowest = min(lowest, e);
			}
			if (lowest == 0u) {
				hi = h0; lo = l0; bc = b0;
				#pragma unroll 1
				for (int i = 0; i < N; i++) {
					const uint32_t e = lut[hi >> (32 - DEC_LB)];
					uint32_t sym = e >> 5;
					if (e == 0u) sym = long_symbol();
					else { hi = __funnelshift_l(lo, hi, e); lo = __funnelshift_l(0u, lo, e); bc -= e & 31u; }
					dst[i] = (uint16_t)sym;
				}
			}
		};
		uint16_t* sg = so;
		#pragma unroll 1
		for (int c = 0; c < kGSize / 6; c++, sg += 6) {
			run(sg, std::integral_constant<int, 3>()); run(sg + 3, std::integral_constant<int, 3>());
			if (bad) break;
		}
		if (!bad) run(sg, std::integral_constant<int, 2>());
		static_assert(kGSize == 50 && kGSize % 6 == 2 && DEC_OUT >= 64, "group layout of the fast path");
		__syncwarp();
		uint32_t v0 = so[lane], v1 = so[32 + (lane & 31)];
		uint32_t cnt = (uint32_t)kGSize;
		const uint32_t eobm0 = __ballot_sync(0xffffffffu, v0 == EOB), eobm1 = __ballot_sync(0xffffffffu, v1 == EOB && lane < (uint32_t)kGSize - 32u);
		__syncwarp();
		if (bad | ((eobm0 | eobm1) != 0u)) {                   // uniform: the last group of the block (or an invalid code)
			hi = hi0; lo = lo0; bc = bc0; wi = wi0; nxt = nxt0;
			uint32_t k = 0;
			bool stop = false;
			while (!stop && k < (uint32_t)kGSize) {
				refill();
				const uint32_t e = lut[hi >> (32 - DEC_LB)];
				uint32_t sym;
				if (e != 0u) { hi = __funnelshift_l(lo, hi, e); lo = __funnelshift_l(0u, lo, e); bc -= e & 31u; sym = e >> 5; }
				else {
					bb = ((uint64_t)hi << 32) | lo;
					const uint32_t window = peek(20);
					const int32_t* limit = S.limit[t]; const int32_t* base = S.base[t];
					int zn = S.minlen[t]; int32_t zvec = (int32_t)(window >> (20 - zn));
					for (;;) {
						if (zn > 20) FAIL(2);
						if (zvec <= limit[zn]) break;
						zn++;
						if (zn <= 20) zvec = (int32_t)(window >> (20 - zn));
					}
					const int32_t idx = zvec - base[zn];
					if (idx < 0 || idx >= kMaxAlpha) FAIL(2);
					sym = S.perm[t][idx];
					drop((uint32_t)zn);
					hi = (uint32_t)(bb >> 32); lo = (uint32_t)bb;
				}
				so[k] = (uint16_t)sym;
				k++;
				stop = (sym == EOB);
			}
			done = stop; cnt = k;
			__syncwarp();
			v0 = so[lane]; v1 = so[32 + (lane & 31)];
			__syncwarp();
		}
		if (lane < cnt && nsym + lane < mcap) mtfv[nsym + lane] = (uint16_t)v0;
		if (32u + lane < cnt && nsym + 32u + lane < mcap) mtfv[nsym + 32u + lane] = (uint16_t)v1;
		nsym += cnt;
		if (nsym > mcap || wi > wi_limit) FAIL(2);               // more symbols than any block of this geometry can hold
		top_up();
	}
	bb = ((uint64_t)hi << 32) | lo;
	if (bc <= 32u) { bb |= (uint64_t)nxt << (32u - bc); bc += 32u; wi++; nxt = sw[wi & (DEC_RING - 1)]; }      // back to the header reader's invariant
	if (wi > wi_limit) FAIL(2);
	if (lane == 0) {
		J.n_mtf = nsym; J.n_in_use = n_in_use; J.orig_ptr = orig_ptr; J.stored_crc = stored_crc; J.level = (uint32_t)level; J.status = 0;
		J.max_block = max_block; J.flags = (kb == 0 ? kSubFirst : 0u) | (randomised ? kSubRand : 0u);
		for (int k = 0; k < 8; k++) J.in_use[k] = iu[k];
	}
	if (SINGLE) {                                          // the block ends here: what follows is the chain walk's business
		if (lane == 0) { J.flags |= kSubLast; endbit[job] = beg * 8 + (uint64_t)wi * 32 - bc; crc_out[job] = stored_crc; }
		return;
	}
	combined = ((combined << 1) | (combined >> 31)) ^ stored_crc;         // bzlib.c / decompress.c: calculatedCombinedCRC
	m1 = get(24); m2 = get(24);                            // next block header or end-of-stream magic
	}
	// end of stream: combined CRC of all blocks (single block: == block CRC)
	if (get(32) != combined) FAIL(3);
	if (wi > wi_limit) FAIL(2);
	__syncwarp();
	if (lane == 0) {
		if (kb == 0) { J0.level = (uint32_t)level; J0.flags = kSubFirst | kSubLast; }      // empty stream
		else jobs[(size_t)job * nsub + kb - 1].flags |= kSubLast;
	}
	#undef FAIL
}

// Sequential per-thread readers over global arrays: a thread that walks its chunk element by element pays one memory
// latency per element (ncu: 77-97 % long-scoreboard stalls on those lines); these fetch 16 bytes at a time with one block of
// lookahead, the element comes out of registers.  Bases are 16-byte aligned (job slots), `lim` = first element never needed.
struct HalfReader {
	const uint4* base; uint32_t blk, lim; uint4 cur, nxt;
	__device__ __forceinline__ void init(const uint16_t* p, uint32_t i, uint32_t lim_) {
		base = reinterpret_cast<const uint4*>(p); lim = lim_; blk = i >> 3; cur = base[blk];
		nxt = ((blk + 1) << 3) < lim ? base[blk + 1] : make_uint4(0, 0, 0, 0);
	}
	__device__ __forceinline__ uint32_t get(uint32_t i) {
		const uint32_t b = i >> 3;
		if (b != blk) {
			cur = (b == blk + 1) ? nxt : base[b];
			blk = b;
			nxt = ((b + 1) << 3) < lim ? base[b + 1] : make_uint4(0, 0, 0, 0);
		}
		const uint32_t w = (i >> 1) & 3u;
		const uint32_t v = w == 0 ? cur.x : w == 1 ? cur.y : w == 2 ? cur.z : cur.w;
		return (v >> ((i & 1u) * 16u)) & 0xffffu;
	}
};

// =====================================================================================================
// k_imtf : one CTA per block -- run expansion + inverse move-to-front, in parallel over chunks of symbols.
// A chunk's effect on the list is a permutation that does not depend on the list it starts from, so
//   A. thread t runs the inverse MTF over its symbols on an IDENTITY list: each symbol yields an index q into the
//      (unknown) list at the chunk start; the final list is the chunk's permutation P(t);
//   B. the chunk-start lists follow by composition   start(t+1)[j] = start(t)[P(t)[j]]   (128 cheap CTA-wide steps);
//   C. thread t replays its symbols: output byte = seqToUnseq[start(t)[q]], RUNA/RUNB runs repeat the front symbol.
// Output offsets come from a block scan of the per-chunk output counts. (decompress.c:349-487)
// =====================================================================================================
constexpr int IM_NT = 128;
constexpr int IM_STS = IM_NT + 1;         // word row stride of the packed per-thread lists

extern __shared__ __align__(16) uint8_t im_smem[];

__global__ void __launch_bounds__(IM_NT)
k_imtf(const uint16_t* __restrict__ mtfv_all, uint32_t mcap, DecJob* __restrict__ jobs, uint32_t njobs,
       uint8_t* __restrict__ q_all /* scratch slot per block (the text slot, free until the inverse BWT) */,
       uint8_t* __restrict__ bwt_all, uint32_t cap)
{
	uint32_t* st = reinterpret_cast<uint32_t*>(im_smem);                               // [64][STS] packed lists
	// the chunk-start lists reuse the same bytes: element (pos, t) of the permutation P(t) is read into a register just
	// before element (pos, t) of start(t) is stored (phase B)
	uint32_t* red = reinterpret_cast<uint32_t*>(im_smem + 64 * IM_STS * 4);             // [64]
	uint32_t* s_start = red + 64;                                                       // [NT + 1] chunk boundaries (symbol index)
	uint8_t* unseq = reinterpret_cast<uint8_t*>(s_start + IM_NT + 4);                   // [256]
	uint8_t* st8 = reinterpret_cast<uint8_t*>(st);
	#define ST_BYTE(pos, t) st8[(((pos) >> 2) * IM_STS + (t)) * 4 + ((pos) & 3)]

	const uint32_t tid = threadIdx.x;
	const uint32_t job = blockIdx.x;
	if (job >= njobs) return;
	DecJob& J = jobs[job];
	if (J.status != 0) return;
	const uint32_t n_mtf = J.n_mtf;
	if (n_mtf == 0) return;                                                             // empty stream
	const uint16_t* mtfv = mtfv_all + (size_t)job * mcap;
	uint8_t* qs = q_all + (size_t)job * cap;
	uint8_t* L = bwt_all + (size_t)job * cap;
	const uint32_t EOB = J.n_in_use + 1, max_block = J.max_block;
	const uint32_t nsym = n_mtf - 1;                                                    // without EOB
	if (nsym > cap) { if (tid == 0) J.status = 2; return; }                            // every symbol yields >= 1 byte

	// seqToUnseq from the inUse map
	{
		uint32_t below = 0, acc = 0;
		for (int v = 0; v < 2; v++) {
			const uint32_t val = tid + v * IM_NT;
			acc = 0; below = 0;
			for (int k = 0; k < 8; k++) {
				uint32_t wv = J.in_use[k];
				if ((val >> 5) == (uint32_t)k) below = acc + __popc(wv & ((1u << (val & 31)) - 1u));
				acc += __popc(wv);
			}
			if ((J.in_use[val >> 5] >> (val & 31)) & 1u) unseq[below] = (uint8_t)val;
		}
	}
	// chunk boundaries: never inside a RUNA/RUNB run
	const uint32_t CS = (nsym + IM_NT - 1) / IM_NT;
	{
		uint32_t a = min(nsym, tid * CS);
		if (a > 0) while (a < nsym && mtfv[a] <= 1 && mtfv[a - 1] <= 1) a++;
		s_start[tid] = a;
		if (tid == 0) s_start[IM_NT] = nsym;
	}
	// identity list
	#pragma unroll 4
	for (int wv = 0; wv < 64; wv++) st[wv * IM_STS + tid] = (uint32_t)(4 * wv) * 0x01010101u + 0x03020100u;
	__syncthreads();
	const uint32_t a0 = s_start[tid], a1 = max(a0, s_start[tid + 1]);

	// ---- A. inverse MTF on the identity list; q per symbol, output count per chunk
	uint32_t outc = 0;
	bool bad = false;
	{
		uint32_t* my = st + tid;
		uint32_t i = a0;
		HalfReader rd;
		if (a0 < a1) rd.init(mtfv, a0, a1);
		while (i < a1) {
			uint32_t sym = rd.get(i);
			if (sym <= 1) {                                   // a whole run: bijective base 2
				uint32_t run = 0, wgt = 1;
				for (;;) {
					run += (sym + 1u) * wgt; wgt <<= 1; i++;
					if (run > max_block) { bad = true; break; }
					if (i >= a1) break;
					sym = rd.get(i);
					if (sym > 1) break;
				}
				if (bad) break;
				outc += run;
				if (outc > max_block) { bad = true; break; }       // keeps the CTA-wide sum below 128 * max_block: no uint32 wrap
				continue;
			}
			if (sym >= EOB) { bad = true; break; }
			const uint32_t r = sym - 1, wj = r >> 2, j = r & 3;
			uint32_t carry = 0;
			// words below wj shift up by one byte; the entry at (wj, j) goes to the front
			const uint32_t target = my[wj * IM_STS];
			const uint32_t v = (target >> (8 * j)) & 255u;
			carry = v;
			for (uint32_t ww = 0; ww < wj; ww++) {
				const uint32_t word = my[ww * IM_STS];
				my[ww * IM_STS] = (word << 8) | carry;
				carry = word >> 24;
			}
			{
				const uint32_t low = j ? (target & (0xFFFFFFFFu >> (32 - 8 * j))) : 0u;
				const uint32_t keep = (j == 3) ? 0u : (target & (0xFFFFFFFFu << (8 * (j + 1))));
				my[wj * IM_STS] = keep | (low << 8) | carry;
			}
			qs[i] = (uint8_t)v;
			outc++;
			i++;
		}
		if (outc > max_block) bad = true;
	}
	uint32_t total; const uint32_t inc = block_scan_add<IM_NT>(outc, red, &total);
	if (__syncthreads_or(bad || total > max_block || total > cap)) { if (tid == 0) J.status = 2; return; }

	// ---- B. chunk-start lists by composition; thread j owns positions j and j + NT
	{
		uint32_t cur0 = tid, cur1 = tid + IM_NT;              // start(0) = identity
		for (uint32_t t = 0; t < IM_NT; t++) {
			const uint32_t p0 = ST_BYTE(tid, t), p1 = ST_BYTE(tid + IM_NT, t);      // P(t), before its bytes become start(t)
			ST_BYTE(tid, t) = (uint8_t)cur0; ST_BYTE(tid + IM_NT, t) = (uint8_t)cur1;
			__syncthreads();
			cur0 = ST_BYTE(p0, t); cur1 = ST_BYTE(p1, t);                 // column t is not written again: no second barrier
		}
		__syncthreads();
	}

	// ---- C. replay: bytes out
	{
		uint32_t o = inc - outc;
		uint32_t front = unseq[ST_BYTE(0, tid)];
		uint32_t i = a0;
		HalfReader rd;
		if (a0 < a1) rd.init(mtfv, a0, a1);
		while (i < a1) {
			uint32_t sym = rd.get(i);
			if (sym <= 1) {
				uint32_t run = 0, wgt = 1;
				for (;;) {
					run += (sym + 1u) * wgt; wgt <<= 1; i++;
					if (i >= a1) break;
					sym = rd.get(i);
					if (sym > 1) break;
				}
				for (uint32_t k = 0; k < run; k++) L[o + k] = (uint8_t)front;
				o += run;
				continue;
			}
			front = unseq[ST_BYTE((uint32_t)qs[i], tid)];
			L[o++] = (uint8_t)front;
			i++;
		}
	}
	#undef ST_BYTE
	if (tid == 0) { J.n = total; if (J.orig_ptr >= total) J.status = 2; }
}

size_t imtf_smem_bytes() { return (size_t)64 * IM_STS * 4 + 64 * 4 + (IM_NT + 4) * 4 + 256 + 64; }

// =====================================================================================================
// k_inv_bwt : one persistent CTA per block.
//   1. LF mapping = one stable counting-sort pass over the last column (decompress.c:494-510 cftab + tt);
//   2. the n-step walk through tt (decompress.c:511-573 / bzlib.c unRLE) is a linked list.  It is cut at every K-th array
//      position (+ the start): ~n/32 sublists.  Every thread measures four sublists at a time (four independent pointer
//      chases in flight), the sublists are ranked by pointer jumping in shared memory (ceil(log2) rounds), and then
//      written, again four at a time per thread.
//   A block whose rotations are not all distinct (exactly periodic text, u repeated r times) walks a cycle of c = n / r
//   steps r times.  The path from the start is then one lap: it is written as above, and the rest of the text repeats it.
// =====================================================================================================
constexpr int IB_MAXS = 6144;     // max number of regular splitters
constexpr int IB_ILP  = 4;        // sublists walked concurrently by one thread
constexpr uint32_t IB_NIL = 0xFFFFu;

extern __shared__ __align__(16) uint8_t ib_smem[];

// NT = 1024: one CTA per SM; NT = 256 (fewer, longer sublists: maxs <= 3072): four CTAs per SM for small blocks, so that the 484
// blocks of a 2048^2 frame are all resident at once instead of four waves of 148 CTAs (the same split as k_bwt)
template <int NT>
__global__ void __launch_bounds__(NT, NT == 1024 ? 1 : 4)
k_inv_bwt(const uint8_t* __restrict__ bwt_all, uint32_t cap, DecJob* __restrict__ jobs, uint32_t njobs,
          uint32_t* __restrict__ tt_all, uint8_t* __restrict__ txt_all, uint32_t maxs)
{
	constexpr int BWT_NT = NT;                       // shadows the namespace constant inside this kernel
	__shared__ uint32_t wcnt[(NT / 32) * BWT_WS];
	__shared__ uint32_t run[256];
	__shared__ uint32_t red[64];
	uint32_t* s_dist = reinterpret_cast<uint32_t*>(ib_smem);                         // [2][maxs + 2]
	uint16_t* s_nxt = reinterpret_cast<uint16_t*>(s_dist + 2 * (maxs + 2));         // [2][maxs + 2]
	const uint32_t tid = threadIdx.x;
	uint32_t* tt = tt_all + (size_t)blockIdx.x * cap;          // per-CTA scratch

	for (uint32_t job = blockIdx.x; job < njobs; job += gridDim.x) {
		DecJob& J = jobs[job];
		const uint32_t n = J.n;
		if (J.status != 0 || n == 0) continue;
		const uint8_t* L = bwt_all + (size_t)job * cap;
		uint8_t* txt = txt_all + (size_t)job * cap;

		// ---- LF mapping: T[pos] = i for the i-th occurrence ... stable counting sort of positions by byte
		digit_starts<NT>(n, run, wcnt, red, [&](uint32_t e) { return (uint32_t)L[e]; });     // cftab (decompress.c:494-510)
		radix_scatter<BWT_R, uint32_t, NT>(n, run, wcnt,
			[&](uint32_t e) { return (e << 8) | (uint32_t)L[e]; },
			[&](uint32_t p) { return p & 255u; },
			[&](uint32_t pos, uint32_t p) { tt[pos] = p >> 8; });
		__syncthreads();
		for (uint32_t j = tid; j < n; j += BWT_NT) tt[j] = (tt[j] << 8) | (uint32_t)L[j];    // bzip2's tt layout
		__syncthreads();

		// ---- splitters: every K-th position, plus the start of the walk
		uint32_t kshift = 2;                               // sublists of ~4 .. 32 steps: as many as the ranking arrays hold
		while (((n + (1u << kshift) - 1) >> kshift) > maxs) kshift++;
		const uint32_t K = 1u << kshift, S = (n + K - 1) >> kshift;
		const uint32_t p0 = tt[J.orig_ptr] >> 8;
		const bool p0_regular = (p0 & (K - 1)) == 0;
		const uint32_t nspl = S + (p0_regular ? 0 : 1);
		const uint32_t start_id = p0_regular ? (p0 >> kshift) : S;
		{   // ---- measure: length of every sublist and the sublist it runs into
			for (uint32_t q0 = tid; q0 < nspl; q0 += BWT_NT * IB_ILP) {
				uint32_t p[IB_ILP], len[IB_ILP]; bool act[IB_ILP];
				#pragma unroll
				for (int j = 0; j < IB_ILP; j++) { const uint32_t q = q0 + j * BWT_NT; act[j] = q < nspl; p[j] = q < S ? (q << kshift) : p0; len[j] = 0; }
				bool any = true;
				while (any) {
					any = false;
					#pragma unroll
					for (int j = 0; j < IB_ILP; j++) if (act[j]) p[j] = tt[p[j]] >> 8;
					#pragma unroll
					for (int j = 0; j < IB_ILP; j++) if (act[j]) {
						len[j]++;
						if ((p[j] & (K - 1)) == 0 || p[j] == p0 || len[j] >= n) act[j] = false; else any = true;
					}
				}
				#pragma unroll
				for (int j = 0; j < IB_ILP; j++) {
					const uint32_t q = q0 + j * BWT_NT;
					if (q < nspl) {
						uint32_t id = (p[j] == p0) ? start_id : (p[j] >> kshift);
						if (id == start_id) id = IB_NIL;                         // open the cycle at the start: a path
						s_dist[q] = len[j]; s_nxt[q] = (uint16_t)id;
					}
				}
			}
		}
		__syncthreads();
		// ---- rank the sublists: distance to the end of the path by pointer jumping (double buffered)
		uint32_t cur = 0;
		for (uint32_t span = 1; span < nspl; span <<= 1) {
			const uint32_t* di = s_dist + cur * (maxs + 2); const uint16_t* ni = s_nxt + cur * (maxs + 2);
			uint32_t* dq = s_dist + (cur ^ 1) * (maxs + 2); uint16_t* nq = s_nxt + (cur ^ 1) * (maxs + 2);
			for (uint32_t q = tid; q < nspl; q += BWT_NT) {
				const uint32_t nx = ni[q];
				uint32_t d = di[q], n2 = nx;
				if (nx != IB_NIL) { d += di[nx]; n2 = ni[nx]; }
				dq[q] = d; nq[q] = (uint16_t)n2;
			}
			cur ^= 1;
			__syncthreads();
		}
		const uint32_t* dfin = s_dist + cur * (maxs + 2);
		const uint16_t* nfin = s_nxt + cur * (maxs + 2);
		// the path from the start is one lap of the walk's cycle: c = n steps, or n / r for a text that is some u repeated r times;
		// the sublists off the path lie on other cycles and never reach the end of the path
		const uint32_t c = dfin[start_id];
		const bool lap = nfin[start_id] == IB_NIL && c >= 1 && c <= n;              // always (tt is a permutation)
		__syncthreads();
		if (!lap) { if (tid == 0) J.status = 2; continue; }                         // uniform
		{
			// ---- write the lap: sublist q on the path starts at output offset c - dist_to_end(q)
			for (uint32_t q0 = tid; q0 < nspl; q0 += BWT_NT * IB_ILP) {
				// 147 KB blocks: the bytes of a sublist leave as aligned 32-bit words (byte stores only for the ragged first and last word: a
				// word shared with the neighbouring sublist): a quarter of the store instructions (16-frame slice: 5.43 -> 4.99 ms)
				uint32_t p[IB_ILP], off[IB_ILP], end[IB_ILP], acc[IB_ILP], beg[IB_ILP];
				#pragma unroll
				for (int j = 0; j < IB_ILP; j++) {
					const uint32_t q = q0 + j * BWT_NT;
					p[j] = q < S ? (q << kshift) : p0; off[j] = 0; end[j] = 0; acc[j] = 0;
					if (q < nspl && nfin[q] == IB_NIL) { off[j] = c - dfin[q]; end[j] = c; }     // end: upper bound, the walk stops at the next splitter
					beg[j] = off[j];
				}
				bool any = true;
				while (any) {
					any = false;
					uint32_t e[IB_ILP];
					#pragma unroll
					for (int j = 0; j < IB_ILP; j++) if (off[j] < end[j]) e[j] = tt[p[j]];
					#pragma unroll
					for (int j = 0; j < IB_ILP; j++) if (off[j] < end[j]) {
						const uint32_t o = off[j];
						acc[j] |= (e[j] & 255u) << (8u * (o & 3u));
						p[j] = e[j] >> 8; off[j] = o + 1;
						const bool stop = (p[j] & (K - 1)) == 0 || p[j] == p0;
						if (stop) end[j] = off[j]; else any = true;
						if (NT != 1024) txt[o] = (uint8_t)e[j];              // small blocks (four CTAs per SM): plain byte stores measured faster
						else if ((o & 3u) == 3u || stop) {
							if (o + 1 - beg[j] == 4u) *reinterpret_cast<uint32_t*>(txt + (o & ~3u)) = acc[j];      // slots are 16-byte aligned
							else for (uint32_t bpos = beg[j]; bpos <= o; bpos++) txt[bpos] = (uint8_t)(acc[j] >> (8u * (bpos & 3u)));
							acc[j] = 0; beg[j] = o + 1;
						}
					}
				}
			}
		}
		__syncthreads();
		// ---- exactly periodic block: bzip2's n-step walk laps the cycle, so the rest of the text repeats the first lap (when c does
		// not divide n, which only corrupt data gives, this is still what the walk gives; the block CRC decides)
		for (uint32_t k = c + tid; k < n; k += BWT_NT) txt[k] = txt[k % c];
		__syncthreads();
		// de-randomisation (decompress.c BZ_RAND_INIT_MASK / BZ_RAND_UPD_MASK / BZ_RAND_MASK, bzlib.c:577-640): byte j of the block is
		// XORed with 1 when j + 2 is a partial sum of the cyclic BZ2_rNums sequence -- a few hundred bytes per block, walked by one
		// thread (only streams of bzip2 <= 0.9.0 carry the bit)
		if ((J.flags & kSubRand) && tid == 0) {
			uint32_t sum = 0;
			for (uint32_t k = 0;; k++) {
				sum += kRNums[k & 511u];
				if (sum - 2u >= n) break;
				txt[sum - 2u] ^= 1u;
			}
		}
		__syncthreads();
	}
}

// =====================================================================================================
// k_unrle : one CTA per block -- inverse of bzip2's initial run-length coding, CRC check, scatter into the image.
// The decoder is a 5-state machine (state = equal bytes seen in a row, 4 = "next byte is a repeat count",
// 0 = fresh start; bzlib.c:561-728).  Parallel form:
//   1. thread t runs the machine over its chunk of the text for all 5 possible entry states -> (exit state, bytes out);
//   2. the entry state and output offset of every chunk follow from composing those maps in chunk order;
//   3. thread t replays its chunk from the now known entry state, writing into a staging copy of the block
//      (shared memory; the block's dead BWT slot when it does not fit);
//   4. CRC-32 of the staged block: per-chunk table CRC + binary tree of carry-less multiplications (as in k_rle1);
//   5. rows are copied to the symbol image, one warp per row.
// =====================================================================================================
constexpr int UR_NT = 256;

extern __shared__ __align__(16) uint8_t ur_smem[];

// shared state of the run-length machine of one block (phases 1-2)
template <int NT>
struct UrShared {
	uint32_t fn[NT];          // packed transition map of each chunk: 5 x 3 bits (then the CRC level multipliers)
	uint32_t cnt[NT][5];      // bytes produced by each chunk for each entry state
	uint32_t in[NT], off[NT];
	uint32_t crc[NT];
	uint32_t total;
	uint32_t red[64];
};

// ---- 1 + 2. chunk maps, entry state and output offset of every chunk; returns the block's output length (all threads)
template <int NT>
__device__ __forceinline__ uint32_t ur_lengths(const uint8_t* txt, uint32_t n, uint32_t a0, uint32_t a1, UrShared<NT>& U)
{
	const uint32_t tid = threadIdx.x, lane = lane_id(), wid = warp_id();
	{
		// all five entry states in one pass over the chunk (each byte is loaded once)
		uint32_t st[5] = { 0, 1, 2, 3, 4 }, cn[5] = { 0, 0, 0, 0, 0 };
		uint32_t prev = a0 > 0 ? txt[a0 - 1] : 0x100u;
		ByteReader rd;
		if (a0 < a1) rd.init(txt, a0, a1);
		// the five machines fall into step at the first run break that none of them reads as a count byte (a handful of
		// bytes into the chunk): from there on ONE machine is simulated and its byte count added to all five
		uint32_t i = a0;
		bool same = false;
		for (; i < a1 && !same; i++) {
			const uint32_t ch = rd.get(i);
			const bool eq = (ch == prev);
			#pragma unroll
			for (int m = 0; m < 5; m++) {
				if (st[m] == 4) { cn[m] += ch; st[m] = 0; }
				else { st[m] = (st[m] >= 1 && eq) ? st[m] + 1 : 1; cn[m]++; }
			}
			prev = ch;
			same = (st[0] == st[1]) & (st[1] == st[2]) & (st[2] == st[3]) & (st[3] == st[4]);
		}
		if (same) {
			uint32_t s1 = st[0], c1 = 0;
			for (; i < a1; i++) {
				const uint32_t ch = rd.get(i);
				if (s1 == 4) { c1 += ch; s1 = 0; }
				else { s1 = (s1 >= 1 && ch == prev) ? s1 + 1 : 1; c1++; }
				prev = ch;
			}
			#pragma unroll
			for (int m = 0; m < 5; m++) { st[m] = s1; cn[m] += c1; }
		}
		uint32_t fn = 0;
		#pragma unroll
		for (int m = 0; m < 5; m++) { fn |= st[m] << (3 * m); U.cnt[tid][m] = cn[m]; }
		U.fn[tid] = fn;
	}
	__syncthreads();
	// entry state / output offset of every chunk: inclusive scan of the composed transition maps (composition is associative),
	// applied to the start state 0; then a block scan of the byte counts for those entry states
	{
		auto compose = [](uint32_t f, uint32_t g2) -> uint32_t {                      // first f, then g2
			uint32_t h = 0;
			#pragma unroll
			for (int m = 0; m < 5; m++) { const uint32_t mid = (f >> (3 * m)) & 7u; h |= ((g2 >> (3 * mid)) & 7u) << (3 * m); }
			return h;
		};
		const uint32_t ident = 0u | (1u << 3) | (2u << 6) | (3u << 9) | (4u << 12);
		uint32_t f = U.fn[tid];
		#pragma unroll
		for (int o = 1; o < 32; o <<= 1) { const uint32_t pf = __shfl_up_sync(0xffffffffu, f, o); if (lane >= (uint32_t)o) f = compose(pf, f); }
		if (lane == 31) U.in[wid] = f;                                                // U.in doubles as the warp totals for a moment
		__syncthreads();
		uint32_t before = ident;
		for (uint32_t ww = 0; ww < wid; ww++) before = compose(before, U.in[ww]);
		uint32_t ef = __shfl_up_sync(0xffffffffu, f, 1);
		if (lane == 0) ef = ident;
		const uint32_t excl = compose(before, ef);                                    // map of everything before my chunk
		const uint32_t st_in = excl & 7u;                                              // applied to state 0
		__syncthreads();
		U.in[tid] = st_in;
		uint32_t tot; const uint32_t incs = block_scan_add<NT>(U.cnt[tid][st_in], U.red, &tot);
		U.off[tid] = incs - U.cnt[tid][st_in];
		if (tid == 0) U.total = tot;
	}
	__syncthreads();
	return U.total;
}

// ---- 3. replay my chunk from its entry state into out[obase + my offset ..]
template <int NT>
__device__ __forceinline__ void ur_replay(const uint8_t* txt, uint32_t a0, uint32_t a1, const UrShared<NT>& U, uint8_t* out, uint64_t obase)
{
	uint32_t st = U.in[threadIdx.x];
	uint8_t* o = out + obase + U.off[threadIdx.x];
	uint32_t pv = a0 > 0 ? txt[a0 - 1] : 0x100u;             // the byte before (never equal to a byte at the block start)
	ByteReader rd;
	if (a0 < a1) rd.init(txt, a0, a1);
	for (uint32_t i = a0; i < a1; i++) {
		const uint32_t ch = rd.get(i);
		if (st == 4) { for (uint32_t k = 0; k < ch; k++) o[k] = (uint8_t)pv; o += ch; st = 0; }
		else { st = (st >= 1 && ch == pv) ? st + 1 : 1; *o++ = (uint8_t)ch; }
		pv = ch;
	}
}

// =====================================================================================================
// k_unrle : one CTA per block -- inverse of bzip2's initial run-length coding, CRC check, scatter into the image.
// The decoder is a 5-state machine (state = equal bytes seen in a row, 4 = "next byte is a repeat count",
// 0 = fresh start; bzlib.c:561-728).  Parallel form:
//   1. thread t runs the machine over its chunk of the text for all 5 possible entry states -> (exit state, bytes out);
//   2. the entry state and output offset of every chunk follow from composing those maps in chunk order;
//   3. thread t replays its chunk from the now known entry state, writing into a staging copy of the block
//      (shared memory; the block's dead BWT slot when it does not fit);
//   4. CRC-32 of the staged block: per-chunk table CRC + binary tree of carry-less multiplications (rle1_crc, bz_rle1.cuh);
//   5. rows are copied to the symbol image, one warp per row.
// k_unrle_len / k_unrle_flat (standalone streams) run phases 1-2, and 1-4 into a flat output at the block's global offset.
// =====================================================================================================
template <int NT>
__global__ void __launch_bounds__(NT)
k_unrle(const uint8_t* __restrict__ txt_all, uint8_t* __restrict__ stage_all /* = BWT slots, dead by now */, uint32_t cap /* sub-slot */,
        uint32_t nsub, DecJob* __restrict__ jobs, uint32_t njobs, uint16_t* __restrict__ sym, Geom g, const uint64_t* __restrict__ block_ids,
        int stage_in_smem)
{
	__shared__ uint32_t crc_tab[256];
	__shared__ UrShared<NT> U;
	const uint32_t tid = threadIdx.x, lane = lane_id(), wid = warp_id();
	const uint32_t job = blockIdx.x;                                    // KLB block; its bzip2 blocks are records job * nsub + k
	if (job >= njobs) return;
	DecJob& J0 = jobs[(size_t)job * nsub];
	for (uint32_t k = 0; k < nsub; k++) if (jobs[(size_t)job * nsub + k].status != 0) return;
	if (tid < 256) crc_tab[tid] = crc_table_entry(tid);
	uint32_t c0[5], ext[5];
	block_box(g, block_ids[job], c0, ext);
	const uint32_t rows = ext[1] * ext[2] * ext[3] * ext[4], rowpx = ext[0];
	const uint32_t gcount = rows * rowpx * 2;
	uint8_t* stage = stage_in_smem ? ur_smem : stage_all + (size_t)job * nsub * cap;

	uint32_t obase = 0;                                                 // bytes of the KLB block decoded by the blocks before this one
	for (uint32_t kb = 0; kb < nsub; kb++) {
		DecJob& J = jobs[(size_t)job * nsub + kb];
		if (J.flags & kSubUnused) break;
		const uint8_t* txt = txt_all + ((size_t)job * nsub + kb) * cap;
		const uint32_t n = J.n;
		__syncthreads();
		const uint32_t CH = (n + NT - 1) / NT;
		const uint32_t a0 = min(n, tid * CH), a1 = min(n, a0 + CH);
		const uint32_t len = ur_lengths<NT>(txt, n, a0, a1, U);
		if (len > gcount - obase) { if (tid == 0) { J0.status = 2; J0.out_bytes = obase + len; } return; }     // more than the KLB block holds
		ur_replay<NT>(txt, a0, a1, U, stage, obase);
		__syncthreads();
		if (rle1_crc<NT>(stage, obase, len, crc_tab, U.crc, U.fn) != J.stored_crc) { if (tid == 0) J0.status = 3; return; }
		if (tid == 0) J.out_bytes = len;
		obase += len;
	}
	if (obase != gcount) { if (tid == 0) { J0.status = 2; J0.out_bytes = obase; } return; }
	__syncthreads();
	// ---- 5. scatter rows into the image
	for (uint32_t r = wid; r < rows; r += NT / 32) {
		uint32_t y = r % ext[1], q = r / ext[1];
		uint32_t z = q % ext[2]; q /= ext[2];
		uint32_t c = q % ext[3], t = q / ext[3];
		uint16_t* row = sym + (c0[0] + (uint64_t)(c0[1] + y) * g.stride[1] + (uint64_t)(c0[2] + z) * g.stride[2]
		                       + (uint64_t)(c0[3] + c) * g.stride[3] + (uint64_t)(c0[4] + t) * g.stride[4]);
		const uint16_t* srcrow = reinterpret_cast<const uint16_t*>(stage) + (size_t)r * rowpx;
		for (uint32_t x = lane; x < rowpx; x += 32) row[x] = srcrow[x];
	}
	(void)lane;
}

// lens[j] = output bytes of block j (0 when it failed an earlier stage: its status says why)
__global__ void __launch_bounds__(UR_NT)
k_unrle_len(const uint8_t* __restrict__ txt_all, uint32_t cap, const DecJob* __restrict__ jobs, uint32_t* __restrict__ lens)
{
	__shared__ UrShared<UR_NT> U;
	const DecJob& J = jobs[blockIdx.x];
	if (J.status != 0) { if (threadIdx.x == 0) lens[blockIdx.x] = 0; return; }
	const uint8_t* txt = txt_all + (size_t)blockIdx.x * cap;
	const uint32_t n = J.n, CH = (n + UR_NT - 1) / UR_NT;
	const uint32_t a0 = min(n, threadIdx.x * CH), a1 = min(n, a0 + CH);
	const uint32_t len = ur_lengths<UR_NT>(txt, n, a0, a1, U);
	if (threadIdx.x == 0) lens[blockIdx.x] = len;
}

// block j replayed into out[boff[j] ..], CRC checked against the stored one (status 3)
__global__ void __launch_bounds__(UR_NT)
k_unrle_flat(const uint8_t* __restrict__ txt_all, uint32_t cap, DecJob* __restrict__ jobs, const uint64_t* __restrict__ boff, uint8_t* __restrict__ out)
{
	__shared__ uint32_t crc_tab[256];
	__shared__ UrShared<UR_NT> U;
	DecJob& J = jobs[blockIdx.x];
	if (J.status != 0) return;
	if (threadIdx.x < 256) crc_tab[threadIdx.x] = crc_table_entry(threadIdx.x);
	const uint8_t* txt = txt_all + (size_t)blockIdx.x * cap;
	const uint32_t n = J.n, CH = (n + UR_NT - 1) / UR_NT;
	const uint32_t a0 = min(n, threadIdx.x * CH), a1 = min(n, a0 + CH);
	const uint32_t len = ur_lengths<UR_NT>(txt, n, a0, a1, U);
	if ((uint64_t)len != boff[blockIdx.x + 1] - boff[blockIdx.x]) { if (threadIdx.x == 0) J.status = 2; return; }
	uint8_t* o = out + boff[blockIdx.x];
	ur_replay<UR_NT>(txt, a0, a1, U, o, 0);
	__syncthreads();
	if (rle1_crc<UR_NT>(o, 0, len, crc_tab, U.crc, U.fn) != J.stored_crc && threadIdx.x == 0) J.status = 3;
}

// ------------------------------------------------------------------------------------------------ launchers
int launch_decode(const uint8_t* payload, const uint64_t* begin, const uint64_t* end, uint32_t njobs, uint32_t nsub, DecJob* jobs,
                  uint16_t* mtfv, uint32_t mcap, uint8_t* q_scratch, uint8_t* bwt, uint32_t cap, uint32_t selcap, cudaStream_t st,
                  cudaEvent_t between, uint64_t* endbit, uint32_t* crc_out, const uint32_t* job_level, bool imtf)
{
	static const int lb_forced = getenv("LFM_B200_DEC_LB") ? atoi(getenv("LFM_B200_DEC_LB")) : 0;
	int dev = 0, sms = 148; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
	auto plan = [&](size_t table_bytes, int& nw, size_t& per_warp) -> size_t {      // warps per CTA for the most streams per SM; returns streams per SM
		per_warp = table_bytes + dec_sel_bytes(selcap) + (size_t)DEC_RING * 4 + (size_t)DEC_OUT * 2;
		nw = 0; size_t best = 0;
		for (int c = 1; c <= 8; c++) {
			const size_t cta = per_warp * c + 1024;                                    // 227 KB of shared memory, 1 KB reserved per CTA
			if (cta > 200 * 1024) break;
			const size_t warps = std::min<size_t>(32, (227 * 1024) / cta) * c;
			if (warps >= best) { best = warps; nw = c; }
		}
		return best;
	};
	int nw = 0; size_t per_warp = 0;
	const size_t resident10 = plan(sizeof(DecWarpSmemT<10>), nw, per_warp) * (size_t)sms;
	const bool nine = lb_forced == 9 || (lb_forced != 10 && (size_t)njobs > resident10);
	if (nine) plan(sizeof(DecWarpSmemT<9>), nw, per_warp);
	if (nw < 1) return 1;
	const size_t smem = per_warp * nw;
	auto go = [&](auto kern) {
		cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
		kern<<<(njobs + nw - 1) / nw, nw * 32, smem, st>>>(payload, begin, end, njobs, jobs, mtfv, mcap, cap, selcap, nsub, endbit, crc_out, job_level);
	};
	if (endbit) { if (nine) go(k_huff_decode<9, true>); else go(k_huff_decode<10, true>); }
	else { if (nine) go(k_huff_decode<9, false>); else go(k_huff_decode<10, false>); }
	if (between) cudaEventRecord(between, st);               // stage timing: Huffman decode | inverse MTF
	if (!imtf) return 0;
	const size_t smem2 = imtf_smem_bytes();
	cudaFuncSetAttribute(k_imtf, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2);
	k_imtf<<<njobs * nsub, IM_NT, smem2, st>>>(mtfv, mcap, jobs, njobs * nsub, q_scratch, bwt, cap);
	return 0;
}
size_t inv_bwt_scratch_elems(int grid, uint32_t cap) { return (size_t)grid * cap; }
constexpr uint32_t IB_MAXS_SMALL = 3072;
// resident CTAs per SM of the variant launch_inv_bwt picks: 4 (256 threads) for slots of up to 48 KB
int inv_bwt_ctas_per_sm(uint32_t cap)
{
	static const int forced = getenv("LFM_B200_IBWT_NT") ? atoi(getenv("LFM_B200_IBWT_NT")) : 0;
	if (forced == 1024) return 1;
	return cap <= 48 * 1024 ? 4 : 1;
}
void launch_inv_bwt(const uint8_t* bwt, uint32_t cap, DecJob* jobs, uint32_t njobs, uint32_t* tt_scratch, uint8_t* txt,
                    int grid, cudaStream_t st)
{
	if (inv_bwt_ctas_per_sm(cap) == 4) {
		const size_t smem = (size_t)2 * (IB_MAXS_SMALL + 2) * (4 + 2);
		cudaFuncSetAttribute(k_inv_bwt<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
		k_inv_bwt<256><<<grid, 256, smem, st>>>(bwt, cap, jobs, njobs, tt_scratch, txt, IB_MAXS_SMALL);
		return;
	}
	const size_t smem = (size_t)2 * (IB_MAXS + 2) * (4 + 2);
	cudaFuncSetAttribute(k_inv_bwt<1024>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
	k_inv_bwt<1024><<<grid, 1024, smem, st>>>(bwt, cap, jobs, njobs, tt_scratch, txt, (uint32_t)IB_MAXS);
}
void launch_unrle_len(const uint8_t* txt, uint32_t cap, const DecJob* jobs, uint32_t njobs, uint32_t* lens, cudaStream_t st)
{
	k_unrle_len<<<njobs, UR_NT, 0, st>>>(txt, cap, jobs, lens);
}
void launch_unrle_flat(const uint8_t* txt, uint32_t cap, DecJob* jobs, uint32_t njobs, const uint64_t* boff, uint8_t* out, cudaStream_t st)
{
	k_unrle_flat<<<njobs, UR_NT, 0, st>>>(txt, cap, jobs, boff, out);
}
void launch_unrle(const uint8_t* txt, uint8_t* stage_scratch, uint32_t cap, uint32_t nsub, uint32_t max_raw_bytes, DecJob* jobs, uint32_t njobs,
                  uint16_t* sym, const Geom& g, const uint64_t* block_ids, cudaStream_t st)
{
	const int in_smem = max_raw_bytes + 16 <= 200 * 1024;
	const size_t smem = in_smem ? (size_t)max_raw_bytes + 16 : 0;
	// (a 1024-thread variant for the 147 KB blocks was measured slower: 2.08 ms against 1.67 ms on the 16-frame stack)
	cudaFuncSetAttribute(k_unrle<UR_NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
	k_unrle<UR_NT><<<njobs, UR_NT, smem, st>>>(txt, stage_scratch, cap, nsub, jobs, njobs, sym, g, block_ids, in_smem);
}

}  // namespace lfm
