// bz_encode.cu -- bzip2 block encoder stages around the BWT, for sm_100a.
//
// Replaces, bit-exactly, what BZ2_bzBuffToBuffCompress(dst,&len,src,n,level,0,30) does for one KLB block
// (src/klb_imageIO.cpp:217):
//   k_rle1      gather of the block from the symbol image (klb_imageIO.cpp:133-183) + initial run-length coding +
//               block CRC + inUse map                      (bzlib.c:216-354 ADD_CHAR_TO_BLOCK / add_pair_to_block)
//   k_mtf       move-to-front + RUNA/RUNB zero-run coding   (compress.c:121-232 generateMTFValues)
//   k_huff_pack coding-table selection, 4 refinement passes, exact bzip2 Huffman code lengths, canonical codes,
//               MSB-first bit packing and stream framing     (compress.c:240-600 sendMTFValues, huffman.c:63-166,
//               compress.c:603-676 BZ2_compressBlock header/trailer)
#include <cstdio>
#include "bz_rle1.cuh"

#include <cstdlib>
namespace lfm {

// =====================================================================================================
// k_rle1 : one CTA per KLB block.
//   A. gather the block's rows from the symbol image into shared memory (into the block's still unused BWT
//      slot in global memory when it does not fit);
//   B. thread t owns a contiguous chunk (chunks right-aligned: only the first non-empty one is short);
//      run heads (byte != previous byte) are located per chunk, a forward max-scan / backward min-scan over
//      the threads tells every chunk where the run it starts in began and where the run it ends in stops;
//   C. bzip2's run rule in closed form: a run of length R (positions r = 0..R-1) emits byte r when r % 255 < 4
//      and a count byte after every r % 255 == 3  -> outputs(r0..r1) = g(r1) - g(r0), g(x) = 5 (x / 255) + h(x % 255);
//      block scan of the chunk totals gives the output offsets, then every thread writes its part;
//   D. CRC-32: per-chunk table CRC, combined in a binary tree with carry-less multiplications by x^(8 len) mod P.
// (bzlib.c:216-354 ADD_CHAR_TO_BLOCK / add_pair_to_block / flush_RL; bzlib_private.h:157-171)
// =====================================================================================================
constexpr int RLE_NT = 256;                 // small blocks; blocks above 48 KB run with 1024 threads (one CTA per SM: occupancy)

extern __shared__ __align__(16) uint8_t rle_smem[];

template <int NT>
__global__ void __launch_bounds__(NT)
k_rle1(const uint16_t* __restrict__ sym, Geom g, uint64_t first_block, uint32_t njobs,
       uint8_t* __restrict__ txt_all, uint8_t* __restrict__ raw_all /* = BWT slots, free at this point */, uint32_t cap /* sub-slot */,
       uint32_t nsub, EncJob* __restrict__ jobs, int stage_in_smem, uint32_t nblock_max)
{
	__shared__ uint32_t crc_tab[256];
	__shared__ uint32_t red[64];
	__shared__ uint32_t s_a[NT], s_b[NT];
	__shared__ uint32_t s_bout[kMaxSub + 1], s_bin[kMaxSub + 1];      // bzip2 block boundaries: output (post-RLE1) / input byte offsets
	__shared__ uint32_t s_min;
	const uint32_t tid = threadIdx.x, lane = lane_id(), wid = warp_id();
	const uint32_t job = blockIdx.x;
	if (job >= njobs) return;
	if (tid < 256) crc_tab[tid] = crc_table_entry(tid);

	uint32_t c0[5], ext[5];
	block_box(g, first_block + job, c0, ext);
	const uint32_t rows = ext[1] * ext[2] * ext[3] * ext[4], rowpx = ext[0];
	const uint32_t gcount = rows * rowpx * 2;
	uint8_t* out0 = txt_all + (size_t)job * nsub * cap;                 // bzip2 block k of this KLB block goes to out0 + k * cap
	uint8_t* stage = stage_in_smem ? rle_smem : raw_all + (size_t)job * nsub * cap;

	// ---- A. gather (one row per warp at a time)
	for (uint32_t r = wid; r < rows; r += NT / 32) {
		uint32_t y = r % ext[1], q = r / ext[1];
		uint32_t z = q % ext[2]; q /= ext[2];
		uint32_t c = q % ext[3], t = q / ext[3];
		const uint16_t* row = sym + (c0[0] + (uint64_t)(c0[1] + y) * g.stride[1] + (uint64_t)(c0[2] + z) * g.stride[2]
		                             + (uint64_t)(c0[3] + c) * g.stride[3] + (uint64_t)(c0[4] + t) * g.stride[4]);
		uint16_t* dst = reinterpret_cast<uint16_t*>(stage) + (size_t)r * rowpx;
		for (uint32_t x = lane; x < rowpx; x += 32) dst[x] = __ldg(row + x);
	}
	__syncthreads();
	const uint8_t* b = stage;

	// ---- B. chunks (right aligned) and run boundaries (bz_rle1.cuh)
	const uint32_t NONE = 0xFFFFFFFFu;
	const Rle1Chunk ck = rle1_chunk<NT>(b, 0, gcount, true, 0, gcount, red, s_a, s_b);

	// ---- C. count, scan, [block boundaries], write
	const uint32_t outc = rle1_count(b, ck);
	uint32_t total; const uint32_t incs = block_scan_add<NT>(outc, red, &total);
	const uint32_t n = total;
	auto walk = [&](auto emit, auto rec_end) { rle1_walk(b, ck, incs - outc, emit, rec_end); };

	// bzip2 closes a block after the record that brings it to nblockMAX bytes or more -- records are flushed when the first
	// byte of the NEXT record is consumed (ADD_CHAR_TO_BLOCK, bzlib.c:216-258), the test sits before every input byte
	// (copy_input_until_stop, :300-340), and the end of the input flushes whatever is pending into the current block
	// (flush_RL, :263): boundary = first record end b >= start + nblockMAX, unless only ONE more output byte follows
	// (then that byte was the last input byte and joined this block).
	uint32_t nb = 1;
	if (tid == 0) { s_bout[0] = 0; s_bin[0] = 0; }
	if (n > nblock_max + 1) {                                    // uniform
		const uint32_t o_first = incs - outc, o_last = incs;
		uint32_t start = 0;                                      // output offset where the open block starts (same in every thread)
		// at most nsub - 1 boundaries fit the records; one more round detects a stream that needs more than that
		for (uint32_t round = 0; round < nsub && round + 1 < (uint32_t)kMaxSub; round++) {
			const uint32_t T = start + nblock_max;
			if (tid == 0) s_min = NONE;
			__syncthreads();
			uint32_t cand = NONE, cand_in = 0;
			if (T + 1 < n && outc != 0 && o_last >= T && o_first <= T + 4)        // one of my output bytes has index in [T-1, T+4]
				walk([](uint32_t, uint8_t) {}, [&](uint32_t o, uint32_t in_end) { if (o >= T && cand == NONE) { cand = o; cand_in = in_end; } });
			if (cand != NONE) atomicMin(&s_min, cand);
			__syncthreads();
			const uint32_t bnd = s_min;
			const bool found = bnd != NONE && bnd + 1 < n;
			if (found && cand == bnd) { s_bout[nb] = bnd; s_bin[nb] = cand_in; }
			if (found) { nb++; start = bnd; }
			__syncthreads();                                         // s_min is reset by thread 0 in the next round
		}
	}
	if (tid == 0) { s_bout[nb] = n; s_bin[nb] = gcount; }
	__syncthreads();
	// does the stream fit the records reserved for it?  (the last block may still exceed nblockMAX when the loop stopped at kMaxSub)
	const bool too_big = nb > nsub || (s_bout[nb] - s_bout[nb - 1]) + 8 > cap;
	if (too_big) {
		if (tid < nsub) {
			EncJob& J = jobs[(size_t)job * nsub + tid];
			J.raw_bytes = gcount; J.n = 0; J.crc = 0; J.orig_ptr = 0; J.n_mtf = 0; J.n_in_use = 0; J.periodic = 0;
			J.status = tid == 0 ? 4u : 0u; J.flags = kSubUnused; J.total_bits = 0; J.out_bytes = 0; J.stream_crc = 0;
		}
		return;
	}
	{
		uint32_t kc = 0;
		const uint32_t o_first = incs - outc;
		while (kc + 1 < nb && o_first >= s_bout[kc + 1]) kc++;
		uint8_t* dst = out0 + (size_t)kc * cap - s_bout[kc];
		uint32_t lim = s_bout[kc + 1];
		walk([&](uint32_t o, uint8_t v) {
			if (o >= lim && kc + 1 < nb) { kc++; dst = out0 + (size_t)kc * cap - s_bout[kc]; lim = s_bout[kc + 1]; }
			dst[o] = v;
		}, [](uint32_t, uint32_t) {});
	}
	__syncthreads();
	// 8 wrap-around bytes after every block (the sort reads text[i + 0..7]) and zero padding to a multiple of 4
	for (uint32_t k = tid / 12; k < nb; k += NT / 12) {
		rle1_wrap(out0 + (size_t)k * cap, s_bout[k + 1] - s_bout[k], tid % 12);
	}
	// ---- D. CRC-32 of every block's input bytes (bz_rle1.cuh)
	uint32_t combined = 0;
	for (uint32_t k = 0; k < nb; k++) {
		const uint32_t bc = rle1_crc<NT>(b, s_bin[k], s_bin[k + 1] - s_bin[k], crc_tab, s_a, s_b);
		if (tid == 0) {
			EncJob& J = jobs[(size_t)job * nsub + k];
			combined = ((combined << 1) | (combined >> 31)) ^ bc;       // bzlib.c:  combinedCRC = (combinedCRC << 1 | >> 31) ^ blockCRC
			J.raw_bytes = gcount; J.n = s_bout[k + 1] - s_bout[k]; J.crc = bc; J.status = 0; J.periodic = 0; J.orig_ptr = 0;
			// the inUse map (bzlib.c:226, :243-258) is exactly "byte values with a non-zero count in the block": k_bwt derives
			// it from the byte histogram it needs anyway
			for (int q = 0; q < 8; q++) J.in_use[q] = 0;
			J.n_in_use = 0;
			J.flags = (k == 0 ? kSubFirst : 0u) | (k + 1 == nb ? kSubLast : 0u);
			J.stream_crc = combined; J.total_bits = 0; J.out_bytes = 0;
		}
	}
	if (tid >= nb && tid < nsub) {                               // records this stream does not need
		EncJob& J = jobs[(size_t)job * nsub + tid];
		J.raw_bytes = gcount; J.n = 0; J.crc = 0; J.orig_ptr = 0; J.n_mtf = 0; J.n_in_use = 0; J.periodic = 0; J.status = 0;
		J.flags = kSubUnused; J.total_bits = 0; J.out_bytes = 0; J.stream_crc = 0;
	}
}

// =====================================================================================================
// k_mtf : one CTA per block, move-to-front made parallel by chunking.
//   1. thread t scans its chunk of the BWT column backwards -> the chunk's recency list (distinct symbols, most
//      recent first) + membership bitmap;
//   2. the list state at the start of every chunk follows from   S(t+1) = recency(t) ++ (S(t) \ recency(t))
//      -- 256 cheap CTA-wide steps (one list entry per thread, a ballot-compaction per step);
//   3. thread t runs the ordinary sequential move-to-front over its chunk from S(t), lists interleaved in
//      shared memory ([position][thread], conflict-free), ranks go to a per-block scratch slot;
//   4. zero runs -> RUNA/RUNB (bijective base 2) with the run carried across chunk borders, output offsets by a
//      block scan, symbols written to mtfv.   (compress.c:121-232)
// =====================================================================================================
// Sequential per-thread reader of 32-bit words (forward or backward) through 16-byte register windows with one block of
// lookahead: a thread walking its chunk word by word pays one global-memory latency per word otherwise (ncu: 88-94 %
// long-scoreboard stalls on the re-reads of the rank scratch).  `lim` = number of words that may be touched (16-byte blocks
// that start below it are loaded whole: slots are 16-byte aligned and padded).
template <int DIR>
struct WordReader {
	const uint4* base; uint32_t blk, lim; uint4 cur, nxt;
	__device__ __forceinline__ uint4 fetch(uint32_t b) const { return (b << 2) < lim ? base[b] : make_uint4(0, 0, 0, 0); }
	__device__ __forceinline__ void init(const uint32_t* p, uint32_t w, uint32_t lim_) {
		base = reinterpret_cast<const uint4*>(p); lim = lim_; blk = w >> 2; cur = fetch(blk);
		nxt = (DIR > 0) ? fetch(blk + 1) : (blk ? fetch(blk - 1) : make_uint4(0, 0, 0, 0));
	}
	__device__ __forceinline__ uint32_t get(uint32_t w) {
		const uint32_t b = w >> 2;
		if (b != blk) {
			cur = (b == blk + (uint32_t)DIR) ? nxt : fetch(b);
			blk = b;
			nxt = (DIR > 0) ? fetch(b + 1) : (b ? fetch(b - 1) : make_uint4(0, 0, 0, 0));
		}
		const uint32_t k = w & 3u;
		return k == 0 ? cur.x : k == 1 ? cur.y : k == 2 ? cur.z : cur.w;
	}
};

constexpr int MTF_NT = 128;
constexpr int MTF_STS = MTF_NT + 1;        // word row stride of the packed start states

extern __shared__ __align__(16) uint8_t mtf_smem[];

__global__ void __launch_bounds__(MTF_NT)
k_mtf(const uint8_t* __restrict__ bwt_all, uint8_t* __restrict__ rank_all /* scratch, one slot per block */, uint32_t cap,
      EncJob* __restrict__ jobs, uint32_t njobs, uint16_t* __restrict__ mtfv_all, uint32_t mcap)
{
	// [32][STS] 64-bit words, 8 list positions per word (the rank search compares 8 entries per shared-memory load): first the chunks' recency lists, then -- column by column, as phase 2
	// consumes them -- the chunks' start states (element (pos, t) of both lives in the same byte)
	uint32_t* st = reinterpret_cast<uint32_t*>(mtf_smem);
	uint32_t* seen = st + 64 * MTF_STS;                                                     // [8][NT] membership bitmaps
	uint32_t* cnt = seen + 8 * MTF_NT;                                                      // [NT]
	uint32_t* zin = cnt + MTF_NT;                                                           // [NT]
	uint32_t* red = zin + MTF_NT;                                                           // [64]
	uint8_t* seqmap = reinterpret_cast<uint8_t*>(red + 64);                                 // [256]
	uint8_t* tmp = seqmap + 256;                                                            // [256]
	uint8_t* st8 = reinterpret_cast<uint8_t*>(st);
	#define ST_BYTE(pos, t) st8[(((pos) >> 3) * MTF_STS + (t)) * 8 + ((pos) & 7)]      // 8 list positions per 64-bit word, words of a thread MTF_STS apart

	const uint32_t tid = threadIdx.x, lane = lane_id(), wid = warp_id();
	const uint32_t job = blockIdx.x;
	if (job >= njobs) return;
	if (jobs[job].flags & kSubUnused) return;               // no bzip2 block in this record
	const uint32_t n = jobs[job].n;
	const uint8_t* bwt = bwt_all + (size_t)job * cap;
	uint8_t* rk = rank_all + (size_t)job * cap;
	uint16_t* mtfv = mtfv_all + (size_t)job * mcap;

	// unseqToSeq (compress.c:105-116); each thread fills two entries
	uint32_t n_in_use = 0;
	{
		uint32_t below0 = 0, below1 = 0;
		const uint32_t v0 = tid, v1 = tid + MTF_NT;
		for (int k = 0; k < 8; k++) {
			uint32_t wv = jobs[job].in_use[k];
			if ((v0 >> 5) == (uint32_t)k) below0 = n_in_use + __popc(wv & ((1u << (v0 & 31)) - 1u));
			if ((v1 >> 5) == (uint32_t)k) below1 = n_in_use + __popc(wv & ((1u << (v1 & 31)) - 1u));
			n_in_use += __popc(wv);
		}
		seqmap[v0] = (uint8_t)below0; seqmap[v1] = (uint8_t)below1;
	}
	__syncthreads();
	const uint32_t EOB = n_in_use + 1;
	const uint32_t CH = ((n + MTF_NT - 1) / MTF_NT + 3) & ~3u;      // whole words: chunks are read and written 4 bytes at a time
	const uint32_t c0 = min(n, tid * CH), c1 = min(n, c0 + CH);
	const uint32_t* bwt32 = reinterpret_cast<const uint32_t*>(bwt);    // slots are 16-byte aligned and padded past n
	uint32_t* rk32 = reinterpret_cast<uint32_t*>(rk);

	// ---- 1. recency list of the chunk
	#pragma unroll
	for (int k = 0; k < 8; k++) seen[k * MTF_NT + tid] = 0;
	uint32_t my_cnt = 0;
	const uint32_t nwords = (n + 3) >> 2;
	WordReader<-1> rb;
	if (c0 < c1) rb.init(bwt32, (((c1 + 3) & ~3u) - 4) >> 2, nwords);
	for (uint32_t i4 = (c0 < c1) ? ((c1 + 3) & ~3u) : c0; i4 > c0; i4 -= 4) {   // a non-empty chunk starts on a multiple of 4
		const uint32_t word = rb.get((i4 - 4) >> 2);
		#pragma unroll
		for (int k = 3; k >= 0; k--) {
			if (i4 - 4 + k < c1) {
				const uint32_t c = seqmap[(word >> (8 * k)) & 255u];
				const uint32_t wv = seen[(c >> 5) * MTF_NT + tid], bit = 1u << (c & 31);
				if (!(wv & bit)) { seen[(c >> 5) * MTF_NT + tid] = wv | bit; ST_BYTE(my_cnt, tid) = (uint8_t)c; my_cnt++; }
			}
		}
	}
	cnt[tid] = my_cnt;
	__syncthreads();

	// ---- 2. start state of every chunk; thread j owns list positions j and j + NT
	uint32_t mine0 = tid, mine1 = tid + MTF_NT;               // initial list: yy[i] = i
	for (uint32_t t = 0; t < MTF_NT; t++) {
		const uint32_t r0 = ST_BYTE(tid, t), r1 = ST_BYTE(tid + MTF_NT, t);       // recency list of chunk t, read before its bytes are reused
		ST_BYTE(tid, t) = (uint8_t)mine0; ST_BYTE(tid + MTF_NT, t) = (uint8_t)mine1;
		const uint32_t ct = cnt[t];
		if (ct == 0) continue;                                // empty chunk (only past the end of the block)
		const bool keep0 = !((seen[(mine0 >> 5) * MTF_NT + t] >> (mine0 & 31)) & 1u);
		const bool keep1 = !((seen[(mine1 >> 5) * MTF_NT + t] >> (mine1 & 31)) & 1u);
		const uint32_t bal0 = __ballot_sync(0xffffffffu, keep0), bal1 = __ballot_sync(0xffffffffu, keep1);
		if (lane == 0) { red[wid] = __popc(bal0); red[4 + wid] = __popc(bal1); }
		__syncthreads();
		uint32_t before0 = 0, before1 = 0;
		#pragma unroll
		for (int ww = 0; ww < 4; ww++) { uint32_t a0 = red[ww], a1 = red[4 + ww]; if ((uint32_t)ww < wid) { before0 += a0; before1 += a1; } before1 += a0; }
		const uint32_t lt = (1u << lane) - 1u;
		if (keep0) tmp[ct + before0 + __popc(bal0 & lt)] = (uint8_t)mine0;
		if (keep1) tmp[ct + before1 + __popc(bal1 & lt)] = (uint8_t)mine1;
		if (tid < ct) tmp[tid] = (uint8_t)r0;
		if (tid + MTF_NT < ct) tmp[tid + MTF_NT] = (uint8_t)r1;
		__syncthreads();
		mine0 = tmp[tid]; mine1 = tmp[tid + MTF_NT];
	}
	__syncthreads();

	// ---- 3. sequential move-to-front per chunk on the packed list (8 positions per 64-bit word)
	{
		uint64_t* my = reinterpret_cast<uint64_t*>(st) + tid;   // word w of my list (8 positions): my[w * STS]
		uint32_t front = (uint32_t)my[0] & 255u;
		WordReader<1> rf;
		if (c0 < c1) rf.init(bwt32, c0 >> 2, nwords);
		for (uint32_t i4 = c0; i4 < c1; i4 += 4) {
			const uint32_t inw = rf.get(i4 >> 2);
			uint32_t outw = 0;
			#pragma unroll
			for (int k = 0; k < 4; k++) {
				if (i4 + k < c1) {
					const uint32_t c = seqmap[(inw >> (8 * k)) & 255u];
					uint32_t r = 0;
					if (c != front) {
						const uint64_t pat = (uint64_t)c * 0x0101010101010101ull;
						uint64_t carry = c;
						for (uint32_t w = 0; ; w++) {
							const uint64_t word = my[w * MTF_STS];
							const uint64_t x = word ^ pat;
							const uint64_t m = (x - 0x0101010101010101ull) & ~x & 0x8080808080808080ull;   // 0x80 in (at least) the lowest byte equal to c
							if (m) {
								const uint32_t j = (uint32_t)(__ffsll((long long)m) - 1) >> 3;        // lowest matching byte: borrows only spoil higher ones
								const uint64_t low = j ? (word & (~0ull >> (64 - 8 * j))) : 0ull;   // bytes below it
								const uint64_t keep = (j == 7) ? 0ull : (word & (~0ull << (8 * (j + 1))));
								my[w * MTF_STS] = keep | (low << 8) | carry;
								r = 8 * w + j;
								break;
							}
							my[w * MTF_STS] = (word << 8) | carry;
							carry = word >> 56;
						}
						front = c;
					}
					outw |= r << (8 * k);
				}
			}
			rk32[i4 >> 2] = outw;
		}
	}
	#undef ST_BYTE
	// ---- 4. zero-run coding. A run is emitted by the chunk in which it ends.
	__syncthreads();
	uint32_t lead = 0, trail = 0;                            // leading / trailing zero ranks of my chunk
	{
		bool open = true;
		WordReader<1> rr1;
		if (c0 < c1) rr1.init(rk32, c0 >> 2, nwords);
		for (uint32_t i4 = c0; i4 < c1; i4 += 4) {
			const uint32_t w = rr1.get(i4 >> 2);
			#pragma unroll
			for (int k = 0; k < 4; k++) if (i4 + k < c1) {
				const bool z0 = ((w >> (8 * k)) & 255u) == 0;
				if (open) { if (z0) lead++; else open = false; }
				trail = z0 ? trail + 1 : 0;
			}
		}
	}
	// run carried INTO each chunk: scan of (all zero?, value) with  a . b = b.allzero ? (a.allzero, a.v + b.v) : (false, b.v)
	uint32_t zin_mine, zpend_end;
	{
		const bool my_az = (lead == c1 - c0);
		uint32_t az = my_az ? 1u : 0u, vv = my_az ? (c1 - c0) : trail;
		#pragma unroll
		for (int o = 1; o < 32; o <<= 1) {
			const uint32_t paz = __shfl_up_sync(0xffffffffu, az, o), pv = __shfl_up_sync(0xffffffffu, vv, o);
			if (lane >= (uint32_t)o) { if (az) { vv += pv; az = paz; } }
		}
		if (lane == 31) { cnt[wid] = az; cnt[8 + wid] = vv; }
		__syncthreads();
		uint32_t bv = 0;                                       // run pending after all the warps before mine
		for (uint32_t ww = 0; ww < wid; ww++) { const uint32_t a2 = cnt[ww], v2 = cnt[8 + ww]; bv = a2 ? bv + v2 : v2; }
		uint32_t eaz = __shfl_up_sync(0xffffffffu, az, 1), ev = __shfl_up_sync(0xffffffffu, vv, 1);
		if (lane == 0) { eaz = 1u; ev = 0; }
		zin_mine = eaz ? bv + ev : ev;                         // exclusive prefix = run pending at my chunk start
		const uint32_t incl_v = az ? bv + vv : vv;
		if (tid == MTF_NT - 1) red[40] = incl_v;               // run still pending at the end of the block
		__syncthreads();
		zpend_end = red[40];
	}
	auto ndigits = [](uint32_t r) { return r ? (uint32_t)(31 - __clz(r + 1)) : 0u; };
	uint32_t outc = 0;
	{
		uint32_t z = zin_mine;
		WordReader<1> rr2;
		if (c0 < c1) rr2.init(rk32, c0 >> 2, nwords);
		for (uint32_t i4 = c0; i4 < c1; i4 += 4) {
			const uint32_t w = rr2.get(i4 >> 2);
			#pragma unroll
			for (int k = 0; k < 4; k++) if (i4 + k < c1) {
				if (((w >> (8 * k)) & 255u) == 0) z++;
				else { outc += ndigits(z) + 1; z = 0; }
			}
		}
	}
	// the thread that owns the last byte also flushes the final run and writes EOB
	const bool owner_of_end = (n == 0) ? (tid == 0) : (c0 < n && c1 == n);
	if (owner_of_end) outc += ndigits(zpend_end) + 1;
	uint32_t total; uint32_t inc = block_scan_add<MTF_NT>(outc, red, &total);
	uint32_t o = inc - outc;
	{
		uint32_t z = zin_mine;
		auto put_run = [&](uint32_t zz) {
			if (!zz) return;
			uint32_t q = zz - 1;
			for (;;) { mtfv[o++] = (uint16_t)(q & 1u); if (q < 2) break; q = (q - 2) >> 1; }
		};
		WordReader<1> rr3;
		if (c0 < c1) rr3.init(rk32, c0 >> 2, nwords);
		for (uint32_t i4 = c0; i4 < c1; i4 += 4) {
			const uint32_t w = rr3.get(i4 >> 2);
			#pragma unroll
			for (int k = 0; k < 4; k++) if (i4 + k < c1) {
				const uint32_t r = (w >> (8 * k)) & 255u;
				if (r == 0) z++;
				else { put_run(z); z = 0; mtfv[o++] = (uint16_t)(r + 1); }
			}
		}
		if (owner_of_end) { put_run(zpend_end); mtfv[o++] = (uint16_t)EOB; }
	}
	if (tid == 0) { jobs[job].n_mtf = total; jobs[job].n_in_use = n_in_use; }
}

size_t mtf_smem_bytes() { return (size_t)64 * MTF_STS * 4 + 8 * MTF_NT * 4 + (MTF_NT * 2 + 64) * 4 + 512; }

// =====================================================================================================
// k_huff_pack : one CTA (8 warps) per block; warp t owns coding table t.
//   * symbol histogram, number of tables, initial partition                      (compress.c:268-316)
//   * 4 refinement passes: cost of every 50-symbol group under every table in parallel over the groups, then
//     exact bzip2 code lengths per table: lane 0 of the table's warp runs the heap with (weight, node) packed in one
//     64-bit shared-memory word -- one load per heap level -- and the 32 lanes walk the parent links (huffman.c:63-148)
//   * canonical codes by a warp counting pass                                     (huffman.c:152-166)
//   * the bit stream: every field's length is known before anything is written, so offsets come from scans and all
//     threads OR their bits into the zeroed output (selectors, delta-coded lengths, symbols)  (compress.c:482-600)
// =====================================================================================================
constexpr int HP_NT = 256;
constexpr int HP_SYMS = 8;     // symbols per thread per packing tile
constexpr uint16_t HP_NOPARENT = 0xFFFFu;

constexpr int HP_HEAP = 2 * kMaxAlpha + 8;          // heap slots per table: every child index of a live node exists
constexpr uint32_t HP_INF = 0xFFFFFFFFu;             // weight of an empty heap slot (real weights stay below 2^29)

// Exact restatement of the tree construction of BZ2_hbMakeCodeLengths (huffman.c:63-148) for ONE table, run by ONE
// lane: same heap discipline (strict '<' everywhere), same weight arithmetic.  The lanes of a warp build the tables
// of a block side by side (one lane per table), so the sequential part costs the issue slots of one warp.
//   heap entry = weight << 32 | node, ordered by weight only; slot 0 holds weight 0 (every up-heap stops there);
//   slots past the heap hold HP_INF, and both children of a slot sit in one 16-byte word: a down-heap level is one
//   shared-memory load, two compares and one store, with no bounds test.
// Leaves are nodes 1..alpha with weights lw[1..alpha]; parent[] receives the links (HP_NOPARENT at the root).
__device__ __forceinline__ void hp_build_tree(uint64_t* heap, uint16_t* parent, const uint32_t* lw, int alpha)
{
	// (heap walks without data-dependent branches, see hp_build_tree32 below)
	for (int i = 0; i < 2 * alpha + 6; i++) heap[i] = (uint64_t)HP_INF << 32;
	heap[0] = 0;
	auto up_heap = [&](int z, uint32_t wt, uint32_t node) {
		uint64_t anc[9];                                              // the heap never holds more than 2^9 - 1 entries
		#pragma unroll
		for (int k = 0; k < 9; k++) anc[k] = heap[z >> (k + 1)];
		int m = 0;
		#pragma unroll
		for (int k = 0; k < 9; k++) {                                 // keys do not increase towards the root: the first m ancestors move down
			const bool mv = wt < (uint32_t)(anc[k] >> 32);
			if (mv) heap[z >> k] = anc[k];
			m += mv ? 1 : 0;
		}
		heap[z >> m] = ((uint64_t)wt << 32) | node;
	};
	int n_heap = 0;
	for (int i = 1; i <= alpha; i++) {
		parent[i] = HP_NOPARENT;
		up_heap(++n_heap, lw[i], (uint32_t)i);
	}
	int n_nodes = alpha;
	while (n_heap > 1) {
		uint64_t pick[2];
		#pragma unroll
		for (int q = 0; q < 2; q++) {
			pick[q] = heap[1];
			const uint64_t tmp = heap[n_heap];
			heap[n_heap] = (uint64_t)HP_INF << 32;
			n_heap--;
			const uint32_t tw = (uint32_t)(tmp >> 32);
			int z = 1;
			// down-heap, TWO levels per shared-memory round trip: the four grandchildren and the eight great-grandchildren of the
			// current slot are fetched while its children (already in registers) are being compared; slots below the heap hold
			// HP_INF, so the walk stops there by itself (clamped addresses are never used: their parents are HP_INF)
			const int levels = 31 - __clz(n_heap | 1);
			ulonglong2 ch = *reinterpret_cast<const ulonglong2*>(heap + 2);               // children of the root
			bool going = n_heap >= 1;
			#pragma unroll 1
			for (int it = 0; it < levels; it += 2) {
				const int g = min(4 * z, HP_HEAP - 4), q8 = 8 * z;
				const ulonglong2 ga = *reinterpret_cast<const ulonglong2*>(heap + g);
				const ulonglong2 gb = *reinterpret_cast<const ulonglong2*>(heap + g + 2);
				const ulonglong2 q0 = *reinterpret_cast<const ulonglong2*>(heap + min(q8, HP_HEAP - 2));
				const ulonglong2 q1 = *reinterpret_cast<const ulonglong2*>(heap + min(q8 + 2, HP_HEAP - 2));
				const ulonglong2 q2 = *reinterpret_cast<const ulonglong2*>(heap + min(q8 + 4, HP_HEAP - 2));
				const ulonglong2 q3 = *reinterpret_cast<const ulonglong2*>(heap + min(q8 + 6, HP_HEAP - 2));
				const bool r1 = (uint32_t)(ch.y >> 32) < (uint32_t)(ch.x >> 32);
				const uint64_t c1 = r1 ? ch.y : ch.x;
				going = going & !(tw < (uint32_t)(c1 >> 32));
				if (going) heap[z] = c1;
				z = going ? 2 * z + (r1 ? 1 : 0) : z;
				const ulonglong2 ch2 = r1 ? gb : ga;
				const bool r2 = (uint32_t)(ch2.y >> 32) < (uint32_t)(ch2.x >> 32);
				const uint64_t c2 = r2 ? ch2.y : ch2.x;
				going = going & !(tw < (uint32_t)(c2 >> 32));
				if (going) heap[z] = c2;
				z = going ? 2 * z + (r2 ? 1 : 0) : z;
				ch = r1 ? (r2 ? q3 : q2) : (r2 ? q1 : q0);
			}
			if (n_heap >= 1) heap[z] = tmp;
		}
		n_nodes++;
		parent[(uint32_t)pick[0]] = (uint16_t)n_nodes; parent[(uint32_t)pick[1]] = (uint16_t)n_nodes;
		const uint32_t w1 = (uint32_t)(pick[0] >> 32), w2 = (uint32_t)(pick[1] >> 32);
		const uint32_t d1 = w1 & 0xffu, d2 = w2 & 0xffu;
		const uint32_t nwt = ((w1 & 0xffffff00u) + (w2 & 0xffffff00u)) | (1u + (d1 > d2 ? d1 : d2));
		parent[n_nodes] = HP_NOPARENT;
		up_heap(++n_heap, nwt, (uint32_t)n_nodes);
	}
}

// The same construction with 32-bit heap entries, for blocks of fewer than 2^17 symbols (every 96x96x1 block; the tree build is
// bound by the instructions its single lane issues, and 64-bit entries cost two registers per move / select):
//   entry = frequency sum << 15 | depth << 10 | node      (bzip2's weight is frequency << 8 | depth: the same order, huffman.c:70-71)
// compared on entry >> 10.  Depths above 31 do not fit: the function then returns false and the caller runs the 64-bit version.
__device__ __forceinline__ bool hp_build_tree32(uint32_t* heap, uint16_t* parent, const uint32_t* lw, int alpha)
{
	// A lone lane pays ~4 cycles per instruction and ~25 per branch it has to resolve, so both heap walks are written WITHOUT
	// data-dependent branches: a walk that has found its place keeps going as a no-op (predicated stores, selects) for the
	// fixed number of levels the heap has.
	constexpr uint32_t INF = 0xFFFFFFFFu;
	constexpr int SLOTS = 2 * HP_HEAP;                                  // uint32 slots in the table's heap row
	for (int i = 0; i < 2 * alpha + 6; i++) heap[i] = INF;
	heap[0] = 0;
	// up-heap: all ancestors are fetched at once; their keys do not increase towards the root, so "wt < key" holds for the first
	// m of them and m is a sum of independent compares; ancestor k moves down to the slot of ancestor k - 1, the entry lands above
	auto up_heap = [&](int z, uint32_t e) {
		uint32_t anc[9];
		#pragma unroll
		for (int k = 0; k < 9; k++) anc[k] = heap[z >> (k + 1)];
		const uint32_t wt = e >> 10;
		int m = 0;
		#pragma unroll
		for (int k = 0; k < 9; k++) {
			const bool mv = wt < (anc[k] >> 10);
			if (mv) heap[z >> k] = anc[k];
			m += mv ? 1 : 0;
		}
		heap[z >> m] = e;
	};
	int n_heap = 0;
	for (int i = 1; i <= alpha; i++) {
		parent[i] = HP_NOPARENT;
		up_heap(++n_heap, ((lw[i] >> 8) << 15) | (uint32_t)i);          // leaf weights are frequency << 8, depth 0
	}
	int n_nodes = alpha;
	bool ok = true;
	while (n_heap > 1) {
		uint32_t pick[2];
		#pragma unroll
		for (int q = 0; q < 2; q++) {
			pick[q] = heap[1];
			const uint32_t tmp = heap[n_heap];
			heap[n_heap] = INF;
			n_heap--;
			const uint32_t tw = tmp >> 10;
			int z = 1;
			// down-heap, two levels per shared-memory round trip (grandchildren: one 16-byte load, great-grandchildren: two); slots
			// below the heap hold INF, so the walk stops there by itself (clamped addresses are never used: their parents are INF)
			const int levels = 31 - __clz(n_heap | 1);                            // deepest level that holds an entry (root = 0)
			uint2 ch = *reinterpret_cast<const uint2*>(heap + 2);                 // children of the root
			bool going = n_heap >= 1;
			#pragma unroll 1
			for (int it = 0; it < levels; it += 2) {
				const uint4 g = *reinterpret_cast<const uint4*>(heap + min(4 * z, SLOTS - 4));
				const uint4 qa = *reinterpret_cast<const uint4*>(heap + min(8 * z, SLOTS - 4));
				const uint4 qb = *reinterpret_cast<const uint4*>(heap + min(8 * z + 4, SLOTS - 4));
				const bool r1 = (ch.y >> 10) < (ch.x >> 10);
				const uint32_t c1 = r1 ? ch.y : ch.x;
				going = going & !(tw < (c1 >> 10));
				if (going) heap[z] = c1;
				z = going ? 2 * z + (r1 ? 1 : 0) : z;
				const uint32_t a0 = r1 ? g.z : g.x, a1 = r1 ? g.w : g.y;
				const bool r2 = (a1 >> 10) < (a0 >> 10);
				const uint32_t c2 = r2 ? a1 : a0;
				going = going & !(tw < (c2 >> 10));
				if (going) heap[z] = c2;
				z = going ? 2 * z + (r2 ? 1 : 0) : z;
				const uint4 qq = r1 ? qb : qa;
				ch.x = r2 ? qq.z : qq.x; ch.y = r2 ? qq.w : qq.y;
			}
			if (n_heap >= 1) heap[z] = tmp;
		}
		n_nodes++;
		parent[pick[0] & 1023u] = (uint16_t)n_nodes; parent[pick[1] & 1023u] = (uint16_t)n_nodes;
		const uint32_t d1 = (pick[0] >> 10) & 31u, d2 = (pick[1] >> 10) & 31u;
		const uint32_t nd = 1u + (d1 > d2 ? d1 : d2);
		ok = ok & (nd <= 31u);
		parent[n_nodes] = HP_NOPARENT;
		up_heap(++n_heap, (((pick[0] >> 15) + (pick[1] >> 15)) << 15) | ((nd & 31u) << 10) | (uint32_t)n_nodes);
	}
	return ok;
}

// sequential MSB-first bit writer used by thread 0 for the fixed part of the block header (whole big-endian words)
struct HdrWriter {
	uint32_t* out; uint64_t acc; uint32_t live; uint32_t words;
	__device__ void put(uint32_t nbits, uint32_t v) {
		acc = (acc << nbits) | (uint64_t)v; live += nbits;
		if (live >= 32) {
			uint32_t wv = (uint32_t)(acc >> (live - 32));
			out[words++] = __byte_perm(wv, 0, 0x0123);
			live -= 32;
		}
	}
	__device__ uint32_t bits() const { return words * 32 + live; }
	// the < 32 leftover bits are OR-ed into the (zeroed) next word
	__device__ void finish() { if (live) { uint32_t wv = (uint32_t)(acc << (32 - live)); atomicOr(&out[words], __byte_perm(wv, 0, 0x0123)); } }
};

// OR `nbits` (<= 32) bits of v into the big-endian bit stream at bit position bitpos (words pre-zeroed)
__device__ __forceinline__ void or_bits(uint32_t* out, uint32_t bitpos, uint32_t nbits, uint32_t v)
{
	uint32_t wi = bitpos >> 5, off = bitpos & 31u;
	uint64_t x = (uint64_t)v << (64 - off - nbits);
	uint32_t hi = (uint32_t)(x >> 32), lo = (uint32_t)x;
	if (hi) atomicOr(&out[wi], __byte_perm(hi, 0, 0x0123));
	if (lo) atomicOr(&out[wi + 1], __byte_perm(lo, 0, 0x0123));
}

__global__ void __launch_bounds__(HP_NT)
k_huff_pack(const uint16_t* __restrict__ mtfv_all, uint32_t mcap, EncJob* __restrict__ jobs, uint32_t njobs,
            uint8_t* __restrict__ sel_all, uint32_t selcap, uint8_t* __restrict__ out_all, uint32_t ocap, int level)
{
	__shared__ uint32_t freq[kMaxAlpha + 6];
	__shared__ uint32_t rfreq[kGroups][kMaxAlpha + 2];
	__shared__ uint8_t  len[kGroups][kMaxAlpha + 2];
	__shared__ uint32_t code[kGroups][kMaxAlpha + 2];
	extern __shared__ __align__(16) uint8_t hp_smem[];
	uint64_t (*hheap)[HP_HEAP] = reinterpret_cast<uint64_t (*)[HP_HEAP]>(hp_smem);     // [kGroups][HP_HEAP], 16-byte aligned rows
	__shared__ uint16_t hparent[kGroups][kMaxAlpha * 2 + 4];
	__shared__ uint32_t hlw[kGroups][kMaxAlpha + 2];
	__shared__ __align__(16) uint4 lenpack[kMaxAlpha + 2];            // code lengths of tables (0,1) (2,3) (4,5), 16 bits each
	__shared__ uint32_t red[64];
	__shared__ uint32_t s_tbits[kGroups + 2];
	__shared__ uint32_t s_ngroups;
	__shared__ uint32_t s_redo;
	uint32_t* win = reinterpret_cast<uint32_t*>(hp_smem);          // packing window; reused once the tables are final
	static_assert(sizeof(uint64_t) * kGroups * HP_HEAP >= (HP_NT * HP_SYMS * 20 / 32 + 4) * 4, "window must fit");
	static_assert((HP_HEAP * 8) % 16 == 0, "heap rows must stay 16-byte aligned");

	const uint32_t tid = threadIdx.x, lane = lane_id(), wid = warp_id();
	const uint32_t job = blockIdx.x;
	if (job >= njobs) return;
	EncJob& J = jobs[job];
	const uint32_t n_mtf = J.n_mtf, n_in_use = J.n_in_use;
	const int alpha = (int)n_in_use + 2;
	const uint16_t* mtfv = mtfv_all + (size_t)job * mcap;
	uint8_t* selector = sel_all + (size_t)job * selcap * 2;          // [selcap] table ids, then [selcap] their MTF codes
	uint8_t* selmtf = selector + selcap;
	uint32_t* out = reinterpret_cast<uint32_t*>(out_all + (size_t)job * ocap);

	if (J.flags & kSubUnused) { if (tid == 0) { J.total_bits = 0; J.out_bytes = 0; J.n_groups = 0; J.n_sel = 0; } return; }
	const bool first_blk = (J.flags & kSubFirst) != 0, last_blk = (J.flags & kSubLast) != 0;
	if (J.n == 0) {     // empty input: stream header + trailer only (compress.c:603-676 with nblock == 0)
		if (tid == 0) {
			out[0] = 0; out[1] = 0; out[2] = 0; out[3] = 0;
			HdrWriter hw{ out, 0, 0, 0 };
			hw.put(8, 'B'); hw.put(8, 'Z'); hw.put(8, 'h'); hw.put(8, (uint32_t)('0' + level));
			hw.put(24, 0x177245); hw.put(24, 0x385090); hw.put(32, 0);
			hw.finish();
			J.total_bits = hw.bits(); J.out_bytes = (hw.bits() + 7) / 8; J.n_groups = 0; J.n_sel = 0;
		}
		return;
	}

	// ---- symbol frequencies
	for (uint32_t i = tid; i < kMaxAlpha + 6; i += HP_NT) freq[i] = 0;
	__syncthreads();
	for (uint32_t i = tid; i < n_mtf; i += HP_NT) atomicAdd(&freq[mtfv[i]], 1u);
	__syncthreads();

	// ---- number of tables + initial partition (compress.c:268-316)
	if (tid == 0) {
		int ng = n_mtf < 200 ? 2 : n_mtf < 600 ? 3 : n_mtf < 1200 ? 4 : n_mtf < 2400 ? 5 : 6;
		s_ngroups = ng;
		int n_part = ng, rem = (int)n_mtf, gs = 0;
		while (n_part > 0) {
			int target = rem / n_part, ge = gs - 1, acc = 0;
			while (acc < target && ge < alpha - 1) { ge++; acc += (int)freq[ge]; }
			if (ge > gs && n_part != ng && n_part != 1 && ((ng - n_part) % 2 == 1)) { acc -= (int)freq[ge]; ge--; }
			// table n_part-1 is cheap (0) inside [gs, ge], expensive (15) outside; written below by all threads
			hlw[0][2 * (n_part - 1)] = (uint32_t)gs; hlw[0][2 * (n_part - 1) + 1] = (uint32_t)(ge + 1);
			n_part--; gs = ge + 1; rem -= acc;
		}
	}
	__syncthreads();
	const int ng = (int)s_ngroups;
	for (uint32_t i = tid; i < (uint32_t)ng * (uint32_t)alpha; i += HP_NT) {
		uint32_t t = i / (uint32_t)alpha, v = i - t * (uint32_t)alpha;
		len[t][v] = (v >= hlw[0][2 * t] && v < hlw[0][2 * t + 1]) ? 0 : 15;
	}
	__syncthreads();
	const uint32_t n_sel = (n_mtf + kGSize - 1) / kGSize;

	// ---- 4 refinement passes (compress.c:321-453)
	const uint32_t* mtfv32 = reinterpret_cast<const uint32_t*>(mtfv);          // slots are 16-byte aligned, groups start on even indices
	for (int iter = 0; iter < 4; iter++) {
		for (uint32_t i = tid; i < kGroups * (kMaxAlpha + 2); i += HP_NT) (&rfreq[0][0])[i] = 0;
		for (uint32_t i = tid; i < (uint32_t)alpha; i += HP_NT) {             // the cost of a symbol under all tables in one 16-byte word
			uint4 q;
			q.x = (uint32_t)len[0][i] | ((uint32_t)len[1][i] << 16);
			q.y = ng > 2 ? ((uint32_t)len[2][i] | ((ng > 3 ? (uint32_t)len[3][i] : 255u) << 16)) : 0x00ff00ffu;
			q.z = ng > 4 ? ((uint32_t)len[4][i] | ((ng > 5 ? (uint32_t)len[5][i] : 255u) << 16)) : 0x00ff00ffu;
			q.w = 0;
			lenpack[i] = q;
		}
		__syncthreads();
		for (uint32_t gi = tid; gi < n_sel; gi += HP_NT) {
			const uint32_t gs = gi * kGSize, ge = min(gs + kGSize, n_mtf);
			uint32_t c01 = 0, c23 = 0, c45 = 0;
			const uint32_t full = (ge - gs) >> 1;
			#pragma unroll 5
			for (uint32_t j = 0; j < full; j++) {
				const uint32_t two = __ldg(mtfv32 + (gs >> 1) + j);
				const uint4 a = lenpack[two & 0xffffu], b = lenpack[two >> 16];
				c01 += a.x + b.x; c23 += a.y + b.y; c45 += a.z + b.z;
			}
			if ((ge - gs) & 1u) { const uint4 a = lenpack[mtfv[ge - 1]]; c01 += a.x; c23 += a.y; c45 += a.z; }
			// tables that do not exist cost 255 per symbol: never chosen (a real table costs at most 20 per symbol);
			// ties go to the lowest table, as in compress.c:383-386
			uint32_t bc = c01 & 0xffffu; int bt = 0;
			if ((c01 >> 16) < bc) { bc = c01 >> 16; bt = 1; }
			if ((c23 & 0xffffu) < bc) { bc = c23 & 0xffffu; bt = 2; }
			if ((c23 >> 16) < bc) { bc = c23 >> 16; bt = 3; }
			if ((c45 & 0xffffu) < bc) { bc = c45 & 0xffffu; bt = 4; }
			if ((c45 >> 16) < bc) { bc = c45 >> 16; bt = 5; }
			selector[gi] = (uint8_t)bt;
			uint32_t* rf = rfreq[bt];
			for (uint32_t j = 0; j < full; j++) {
				const uint32_t two = __ldg(mtfv32 + (gs >> 1) + j);
				atomicAdd(&rf[two & 0xffffu], 1u); atomicAdd(&rf[two >> 16], 1u);
			}
			if ((ge - gs) & 1u) atomicAdd(&rf[mtfv[ge - 1]], 1u);
		}
		__syncthreads();
		// exact bzip2 code lengths (huffman.c:63-148): leaf weights, then [tree by one lane per table -> depths by one warp
		// per table -> halve the weights of a table whose depth exceeds 17 and rebuild it], usually a single round
		for (uint32_t i = tid; i < (uint32_t)ng * (uint32_t)alpha; i += HP_NT) {
			const uint32_t t = i / (uint32_t)alpha, v2 = i - t * (uint32_t)alpha;
			const uint32_t fq = rfreq[t][v2];
			hlw[t][v2 + 1] = (fq == 0 ? 1u : fq) << 8;
		}
		uint32_t redo = (1u << ng) - 1u;
		for (;;) {
			__syncthreads();
			if (tid == 0) s_redo = 0;
			// the tables side by side in the lanes of one warp (one warp per table, one active lane each, was measured slower: the
			// SM becomes issue bound, c2 2.2 ms against 1.0 ms on B200)
			if (wid == 0 && (int)lane < ng && ((redo >> lane) & 1u)) {
				if (!(n_mtf < (1u << 17) - 1024u) || !hp_build_tree32(reinterpret_cast<uint32_t*>(hheap[lane]), hparent[lane], hlw[lane], alpha))
					hp_build_tree(hheap[lane], hparent[lane], hlw[lane], alpha);
			}
			__syncthreads();
			if ((int)wid < ng && ((redo >> wid) & 1u)) {
				const uint16_t* parent = hparent[wid];
				bool too_long = false;
				for (int i = (int)lane + 1; i <= alpha; i += 32) {
					int j = 0, k2 = i;
					while (parent[k2] != HP_NOPARENT) { k2 = parent[k2]; j++; }
					len[wid][i - 1] = (uint8_t)j;
					if (j > 17) too_long = true;
				}
				if (__any_sync(0xffffffffu, too_long)) {
					for (int i = (int)lane + 1; i <= alpha; i += 32) { uint32_t j = hlw[wid][i] >> 8; j = 1 + (j / 2); hlw[wid][i] = j << 8; }
					if (lane == 0) atomicOr(&s_redo, 1u << wid);
				}
			}
			__syncthreads();
			redo = s_redo;
			if (redo == 0) break;
		}
	}

	// ---- canonical codes (huffman.c:152-166): code = first code of the length + rank among equal lengths
	if ((int)wid < ng) {
		const int t = (int)wid;
		uint32_t* cnt = hlw[t];                              // [0..20] per-length counters, then first codes
		if (lane < 24) cnt[lane] = 0;
		__syncwarp();
		for (int base = 0; base < alpha; base += 32) {       // rank inside the length class, in symbol order
			const int i = base + (int)lane;
			const bool act = i < alpha;
			const uint32_t am = __ballot_sync(0xffffffffu, act);
			if (act) {
				const uint32_t l = len[t][i];
				const uint32_t peers = __match_any_sync(am, l);
				const uint32_t before = cnt[l];
				code[t][i] = before + __popc(peers & ((1u << lane) - 1u));      // rank for now
				__syncwarp(am);
				if (lane == (uint32_t)(__ffs(peers) - 1)) cnt[l] = before + __popc(peers);
			}
			__syncwarp();
		}
		if (lane == 0) {                                     // first code of each length
			uint32_t vec = 0;
			for (int l = 1; l <= 20; l++) { uint32_t c = cnt[l]; cnt[l] = vec; vec = (vec + c) << 1; }
		}
		__syncwarp();
		for (int i = (int)lane; i < alpha; i += 32) code[t][i] += cnt[len[t][i]];
	}
	__syncthreads();

	// ---- sizes: symbol bits from the last pass' usage counts, header from the field lengths
	uint32_t sym_bits_local = 0;
	for (uint32_t i = tid; i < (uint32_t)ng * (uint32_t)alpha; i += HP_NT) {
		uint32_t t = i / (uint32_t)alpha, v = i % (uint32_t)alpha;
		sym_bits_local += rfreq[t][v] * len[t][v];      // rfreq of the last pass == usage with the final selectors
	}
	uint32_t sym_bits; block_scan_add<HP_NT>(sym_bits_local, red, &sym_bits);
	// selectors: move-to-front codes (compress.c:462-479).  The list after a chunk of selectors is
	//   recency(chunk) ++ (list before \ recency(chunk)),   an associative operation on (<= 6 entry) recency lists:
	// every thread reduces its chunk to a recency list (nibble-packed, most recent first), a CTA-wide scan composes
	// them, and each thread replays its chunk from its now known start list.
	{
		const uint32_t per = (n_sel + HP_NT - 1) / HP_NT;
		const uint32_t s0 = min(n_sel, tid * per), s1 = min(n_sel, s0 + per);
		auto push_front = [](uint32_t& list, uint32_t& mask, uint32_t sv) {           // move sv to the front of a recency list
			if ((mask >> sv) & 1u) {
				uint32_t j = 0;
				while (((list >> (4 * j)) & 15u) != sv) j++;
				const uint32_t lowmask = (1u << (4 * j)) - 1u;
				list = (list & ~((lowmask << 4) | 15u)) | ((list & lowmask) << 4) | sv;
			} else { list = (list << 4) | sv; mask |= 1u << sv; }
		};
		auto then = [](uint32_t la, uint32_t ma, uint32_t lb, uint32_t mb, uint32_t& lo, uint32_t& mo) {   // a first, then b
			uint32_t nb = (uint32_t)__popc(mb), l = lb;
			const uint32_t na = (uint32_t)__popc(ma);
			for (uint32_t j = 0; j < na; j++) {
				const uint32_t vv = (la >> (4 * j)) & 15u;
				if (!((mb >> vv) & 1u)) { l |= vv << (4 * nb); nb++; }
			}
			lo = l; mo = ma | mb;
		};
		uint32_t rl = 0, rm = 0;
		for (uint32_t i = s0; i < s1; i++) push_front(rl, rm, selector[i]);
		__syncthreads();                                                          // red[] is still being read by the scan above
		// inclusive scan inside the warp, then across the 8 warps
		uint32_t il = rl, im = rm;
		#pragma unroll
		for (int o = 1; o < 32; o <<= 1) {
			const uint32_t pl = __shfl_up_sync(0xffffffffu, il, o), pm = __shfl_up_sync(0xffffffffu, im, o);
			if (lane >= (uint32_t)o) then(pl, pm, il, im, il, im);
		}
		if (lane == 31) { red[wid] = il; red[16 + wid] = im; }
		__syncthreads();
		uint32_t bl = 0, bm = 0;                                                  // everything before my warp
		for (uint32_t ww = 0; ww < wid; ww++) then(bl, bm, red[ww], red[16 + ww], bl, bm);
		uint32_t el = __shfl_up_sync(0xffffffffu, il, 1), em = __shfl_up_sync(0xffffffffu, im, 1);
		if (lane == 0) { el = 0; em = 0; }
		then(bl, bm, el, em, el, em);                                             // exclusive prefix of this thread
		uint32_t pos, pm2;
		then(0x543210u, 0x3fu, el, em, pos, pm2);                                 // start list: prefix recency ++ rest of 0..5
		for (uint32_t i = s0; i < s1; i++) {
			const uint32_t sv = selector[i];
			uint32_t j = 0;
			while (((pos >> (4 * j)) & 15u) != sv) j++;
			const uint32_t lowmask = (1u << (4 * j)) - 1u;
			pos = (pos & ~((lowmask << 4) | 15u)) | ((pos & lowmask) << 4) | sv;
			selmtf[i] = (uint8_t)j;
		}
		__syncthreads();
	}
	// delta-coded lengths: bits per table
	if ((int)wid < ng) {
		uint32_t b = 0;
		for (int i = (int)lane; i < alpha; i += 32) {
			int d = i ? (int)len[wid][i] - (int)len[wid][i - 1] : 0;
			b += 2u * (uint32_t)abs(d) + 1u;
		}
		#pragma unroll
		for (int o = 16; o; o >>= 1) b += __shfl_xor_sync(0xffffffffu, b, o);
		if (lane == 0) s_tbits[wid] = b + 5;
	}
	__syncthreads();
	uint32_t sel_bits_local = 0;
	const uint32_t sel_per = (n_sel + HP_NT - 1) / HP_NT;
	const uint32_t sb0 = min(n_sel, tid * sel_per), sb1 = min(n_sel, sb0 + sel_per);
	for (uint32_t i = sb0; i < sb1; i++) sel_bits_local += selmtf[i] + 1u;
	uint32_t sel_bits; const uint32_t sel_inc = block_scan_add<HP_NT>(sel_bits_local, red, &sel_bits);
	uint32_t used16n = 0;
	for (int i = 0; i < 16; i++) if ((J.in_use[i >> 1] >> ((i & 1) * 16)) & 0xffffu) used16n++;
	const uint32_t fixed_bits = (first_blk ? 32u : 0u) + 48 + 32 + 1 + 24 + 16 + 16 * used16n + 3 + 15;   // "BZh" + level only before the first block
	uint32_t len_bits = 0;
	for (int t = 0; t < ng; t++) len_bits += s_tbits[t];
	const uint32_t hdr_bits = fixed_bits + sel_bits + len_bits;
	{
		uint32_t words = (hdr_bits + sym_bits + 80 + 31) / 32 + 2;
		if ((size_t)words * 4 > ocap) { if (tid == 0) { J.status = 2; J.out_bytes = 0; } return; }
		for (uint32_t i = tid; i < words; i += HP_NT) out[i] = 0;
	}
	__syncthreads();

	// ---- header: fixed part by thread 0, selectors by everybody, one table of lengths per warp
	if (tid == 0) {
		HdrWriter hw{ out, 0, 0, 0 };
		if (first_blk) { hw.put(8, 'B'); hw.put(8, 'Z'); hw.put(8, 'h'); hw.put(8, (uint32_t)('0' + level)); }
		hw.put(24, 0x314159); hw.put(24, 0x265359);
		hw.put(32, J.crc);
		hw.put(1, 0);
		hw.put(24, J.orig_ptr);
		uint32_t iu[8]; uint32_t used16 = 0;
		for (int k = 0; k < 8; k++) { iu[k] = J.in_use[k]; }
		for (int i = 0; i < 16; i++) { uint32_t chunk = (iu[i >> 1] >> ((i & 1) * 16)) & 0xffffu; if (chunk) used16 |= 1u << (15 - i); }
		hw.put(16, used16);
		for (int i = 0; i < 16; i++) {
			uint32_t chunk = (iu[i >> 1] >> ((i & 1) * 16)) & 0xffffu;
			if (chunk) hw.put(16, __brev(chunk) >> 16);     // bit j of the chunk is sent j-th (MSB first)
		}
		hw.put(3, (uint32_t)ng);
		hw.put(15, n_sel);
		hw.finish();
	}
	{
		uint32_t bp = fixed_bits + sel_inc - sel_bits_local;
		for (uint32_t i = sb0; i < sb1; i++) {                // j ones then a zero
			const uint32_t j = selmtf[i];
			or_bits(out, bp, j + 1, ((1u << j) - 1u) << 1);
			bp += j + 1;
		}
	}
	if ((int)wid < ng) {
		const int t = (int)wid;
		uint32_t tb = fixed_bits + sel_bits;
		for (int q = 0; q < t; q++) tb += s_tbits[q];
		if (lane == 0) or_bits(out, tb, 5, len[t][0]);
		tb += 5;
		// lane owns a contiguous run of symbols; warp scan of the bit counts
		const int per = (alpha + 31) / 32;
		const int i0 = min(alpha, (int)lane * per), i1 = min(alpha, i0 + per);
		uint32_t mybits = 0;
		for (int i = i0; i < i1; i++) { int d = i ? (int)len[t][i] - (int)len[t][i - 1] : 0; mybits += 2u * (uint32_t)abs(d) + 1u; }
		uint32_t incl = mybits;
		#pragma unroll
		for (int o = 1; o < 32; o <<= 1) { uint32_t v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= (uint32_t)o) incl += v; }
		uint32_t bp = tb + incl - mybits;
		for (int i = i0; i < i1; i++) {
			int d = i ? (int)len[t][i] - (int)len[t][i - 1] : 0;
			uint32_t ad = (uint32_t)abs(d);
			const uint32_t pair = d > 0 ? 2u : 3u;            // "10" = +1, "11" = -1
			while (ad >= 16) { uint32_t v = 0; for (int r = 0; r < 16; r++) v = (v << 2) | pair; or_bits(out, bp, 32, v); bp += 32; ad -= 16; }
			uint32_t v = 0;
			for (uint32_t r = 0; r < ad; r++) v = (v << 2) | pair;
			or_bits(out, bp, 2 * ad + 1, v << 1);             // ... then the terminating 0
			bp += 2 * ad + 1;
		}
	}
	__syncthreads();

	// ---- symbols: tiles of HP_NT*HP_SYMS, bit offsets by block scan, assembled in a shared window
	uint32_t bitpos = hdr_bits;
	constexpr uint32_t TILE = HP_NT * HP_SYMS;
	constexpr uint32_t WIN_WORDS = HP_NT * HP_SYMS * 20 / 32 + 4;
	for (uint32_t t0 = 0; t0 < n_mtf; t0 += TILE) {
		for (uint32_t i = tid; i < WIN_WORDS; i += HP_NT) win[i] = 0;
		uint32_t i0 = t0 + tid * HP_SYMS;
		uint32_t l[HP_SYMS], c[HP_SYMS], sum = 0;
		#pragma unroll
		for (int k = 0; k < HP_SYMS; k++) {
			uint32_t i = i0 + k;
			l[k] = 0; c[k] = 0;
			if (i < n_mtf) { uint32_t t = selector[i / kGSize], sy = mtfv[i]; l[k] = len[t][sy]; c[k] = code[t][sy]; }
			sum += l[k];
		}
		uint32_t tot; uint32_t inc = block_scan_add<HP_NT>(sum, red, &tot);   // includes the barrier after zeroing win
		uint32_t rel = (bitpos & 31u) + inc - sum;
		#pragma unroll
		for (int k = 0; k < HP_SYMS; k++) {
			if (l[k]) {
				uint32_t wi = rel >> 5, off = rel & 31u;
				uint64_t v = (uint64_t)c[k] << (64 - off - l[k]);
				atomicOr(&win[wi], (uint32_t)(v >> 32));
				uint32_t lo = (uint32_t)v;
				if (lo) atomicOr(&win[wi + 1], lo);
				rel += l[k];
			}
		}
		__syncthreads();
		uint32_t nwords = ((bitpos & 31u) + tot + 31) / 32;
		uint32_t w0 = bitpos >> 5;
		for (uint32_t i = tid; i < nwords; i += HP_NT) {
			uint32_t wv = win[i];
			if (wv) atomicOr(&out[w0 + i], __byte_perm(wv, 0, 0x0123));
		}
		bitpos += tot;
		__syncthreads();
	}

	// ---- trailer after the last block of the stream: end-of-stream magic + combined CRC; the stream is padded to a byte
	// when the blocks are put together (k_compact)
	if (tid == 0) {
		uint32_t total = bitpos;
		if (last_blk) {
			or_bits(out, bitpos, 24, 0x177245u);
			or_bits(out, bitpos + 24, 24, 0x385090u);
			or_bits(out, bitpos + 48, 32, J.stream_crc);
			total = bitpos + 80;
		}
		J.total_bits = total; J.out_bytes = (total + 7) / 8; J.n_groups = (uint32_t)ng; J.n_sel = n_sel;
	}
}

// ------------------------------------------------------------------------------------------------ launchers
void launch_rle1(const uint16_t* sym, const Geom& g, uint64_t first_block, uint32_t njobs, uint8_t* txt, uint8_t* raw_scratch,
                 uint32_t cap, uint32_t nsub, uint32_t max_raw_bytes, uint32_t nblock_max, EncJob* jobs, cudaStream_t st)
{
	const int in_smem = max_raw_bytes + 16 <= 200 * 1024;
	const size_t smem = in_smem ? (size_t)max_raw_bytes + 16 : 0;
	if (max_raw_bytes > 48 * 1024) {
		cudaFuncSetAttribute(k_rle1<1024>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
		k_rle1<1024><<<njobs, 1024, smem, st>>>(sym, g, first_block, njobs, txt, raw_scratch, cap, nsub, jobs, in_smem, nblock_max);
	} else {
		cudaFuncSetAttribute(k_rle1<RLE_NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
		k_rle1<RLE_NT><<<njobs, RLE_NT, smem, st>>>(sym, g, first_block, njobs, txt, raw_scratch, cap, nsub, jobs, in_smem, nblock_max);
	}
}
void launch_mtf(const uint8_t* bwt, uint8_t* rank_scratch, uint32_t cap, EncJob* jobs, uint32_t njobs, uint16_t* mtfv, uint32_t mcap, cudaStream_t st)
{
	size_t smem = mtf_smem_bytes();
	cudaFuncSetAttribute(k_mtf, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
	k_mtf<<<njobs, MTF_NT, smem, st>>>(bwt, rank_scratch, cap, jobs, njobs, mtfv, mcap);
}
void launch_huff_pack(const uint16_t* mtfv, uint32_t mcap, EncJob* jobs, uint32_t njobs, uint8_t* sel, uint32_t selcap,
                      uint8_t* out, uint32_t ocap, int level, cudaStream_t st)
{
	const size_t smem = sizeof(uint64_t) * kGroups * HP_HEAP;
	cudaFuncSetAttribute(k_huff_pack, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
	k_huff_pack<<<njobs, HP_NT, smem, st>>>(mtfv, mcap, jobs, njobs, sel, selcap, out, ocap, level);
}

}  // namespace lfm
