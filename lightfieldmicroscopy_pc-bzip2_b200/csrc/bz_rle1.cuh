// bz_rle1.cuh -- bzip2's initial run-length coding of a byte range by one CTA (bzlib.c:216-354 ADD_CHAR_TO_BLOCK /
// add_pair_to_block / flush_RL), phases B-D of k_rle1 (bz_encode.cu).  Shared by k_rle1 (one KLB block = one stream) and the
// kernels of the standalone stream encoder (bz_stream.cu: one tile of the input, or one bzip2 block of it).
//
// Coordinates are absolute indices into `b`.  A CTA covers the range [lo, hi); every thread owns a contiguous chunk of it
// (chunks right aligned: only the first non-empty one is short).  The run context outside the range comes from the caller:
//   lo_is_head   b[lo] starts a run whatever b[lo - 1] is (a KLB block, a bzip2 block: records restart there);
//   out_open     start of the run that is open at lo when b[lo] is not a head;
//   out_next     first run head at or after hi (hi when the range ends the runs).
#pragma once
#include "lfm_device.cuh"

namespace lfm {

constexpr uint32_t kCrcPoly = 0x04C11DB7u;

__device__ __forceinline__ uint32_t crc_mulmod(uint32_t a, uint32_t b)      // a * b in GF(2)[x] / P, bit k <-> x^k
{
	uint32_t r = 0;
	#pragma unroll 8
	for (int i = 31; i >= 0; i--) {
		r = (r << 1) ^ ((r & 0x80000000u) ? kCrcPoly : 0u);
		if ((b >> i) & 1u) r ^= a;
	}
	return r;
}
__device__ __forceinline__ uint32_t crc_xpow8(uint32_t nbytes)              // x^(8 nbytes) mod P
{
	uint32_t e = nbytes * 8u, r = 1u;
	for (int i = 31 - __clz(e | 1u); i >= 0; i--) {
		r = crc_mulmod(r, r);
		if ((e >> i) & 1u) r = (r << 1) ^ ((r & 0x80000000u) ? kCrcPoly : 0u);
	}
	return r;
}
__device__ __forceinline__ uint32_t rle_g(uint32_t x)                        // outputs produced by run positions [0, x)
{
	uint32_t m = x % 255u;
	return (x / 255u) * 5u + min(m, 4u) + (m >= 4u ? 1u : 0u);
}

struct Rle1Chunk {
	uint32_t lo, e0, e1;       // range start; my chunk [e0, e1)
	uint32_t open_start;       // start of the run open at e0
	uint32_t next_head;        // first run head at or after e1
	bool lo_is_head;
	__device__ __forceinline__ bool head(const uint8_t* b, uint32_t i) const { return (i == lo && lo_is_head) || b[i] != b[i - 1]; }
};

// ---- B. my chunk and the run boundaries around it: max-scan of the last head of every chunk, suffix min-scan of the first.
// s_a, s_b: [NT] shared words; red: >= 64 shared words.  Contains barriers.
template <int NT>
__device__ __forceinline__ Rle1Chunk rle1_chunk(const uint8_t* b, uint32_t lo, uint32_t hi, bool lo_is_head, uint32_t out_open,
                                                uint32_t out_next, uint32_t* red, uint32_t* s_a, uint32_t* s_b)
{
	const uint32_t tid = threadIdx.x, lane = lane_id(), wid = warp_id();
	const uint32_t gcount = hi - lo;
	uint32_t CH = ((gcount + NT - 1) / NT + 3) & ~3u;              // whole words, and an odd number of them:
	if (((CH >> 2) & 1u) == 0) CH += 4;                                 // threads then hit distinct shared-memory banks
	const uint32_t after = (NT - 1 - tid) * CH;                     // bytes owned by later threads
	Rle1Chunk c;
	c.lo = lo; c.lo_is_head = lo_is_head;
	const uint32_t x1 = gcount > after ? gcount - after : 0;
	c.e1 = lo + x1; c.e0 = lo + (x1 > CH ? x1 - CH : 0);
	const uint32_t NONE = 0xFFFFFFFFu;
	uint32_t first_head = NONE, last_head = NONE;
	for (uint32_t i = c.e0; i < c.e1; i++) {
		if (c.head(b, i)) { if (first_head == NONE) first_head = i; last_head = i; }
	}
	// start of the run that is open at my chunk start = last head before e0 (max-scan; heads ascend with the thread)
	const uint32_t incl = block_scan_max<NT>(last_head == NONE ? 0u : last_head - lo + 1u, red);     // +1 so that 0 = none
	uint32_t prev_incl = __shfl_up_sync(0xffffffffu, incl, 1);
	if (lane == 0) prev_incl = wid ? red[wid - 1] : 0;
	c.open_start = prev_incl ? lo + prev_incl - 1u : out_open;
	// first head after my chunk: reverse min-scan done through shared memory
	s_a[tid] = first_head;
	__syncthreads();
	{
		// thread r looks at chunk NT-1-r: an inclusive max-scan of ~first_head over r is a suffix min-scan over the chunks
		const uint32_t rv = s_a[NT - 1 - tid];
		const uint32_t rincl = block_scan_max<NT>(~rv, red);                           // NONE -> 0
		uint32_t rprev = __shfl_up_sync(0xffffffffu, rincl, 1);
		if (lane == 0) rprev = wid ? red[wid - 1] : 0;
		s_b[NT - 1 - tid] = rprev ? ~rprev : out_next;                                    // heads strictly after the chunk
	}
	__syncthreads();
	c.next_head = s_b[tid];
	return c;
}

// ---- C (count). Output bytes of my chunk: walk it run segment by run segment.
__device__ __forceinline__ uint32_t rle1_count(const uint8_t* b, const Rle1Chunk& c)
{
	uint32_t outc = 0, i = c.e0, rs = c.open_start;
	while (i < c.e1) {
		if (c.head(b, i)) rs = i;
		uint32_t e = i + 1;
		while (e < c.e1 && b[e] == b[e - 1]) e++;
		outc += rle_g(e - rs) - rle_g(i - rs);
		i = e;
	}
	return outc;
}

// ---- C (walk). One walk of my chunk in output order, starting at output offset o.  A RECORD is (a part of) a run of at most
// 255 equal bytes: up to 4 literals and, from 4 on, a count byte.  emit(o, byte) is called for every output byte, rec_end(o,
// in_end) after the last byte of every record that ends in this chunk's output (o = output offset after it, in_end = input
// index after it).
template <class Emit, class RecEnd>
__device__ __forceinline__ void rle1_walk(const uint8_t* b, const Rle1Chunk& c, uint32_t o, Emit emit, RecEnd rec_end)
{
	uint32_t i = c.e0, rs = c.open_start;
	while (i < c.e1) {
		if (c.head(b, i)) rs = i;
		const uint32_t ch = b[i];
		uint32_t e = i + 1;
		while (e < c.e1 && b[e] == b[e - 1]) e++;
		const uint32_t run_end = (e < c.e1) ? e : c.next_head;     // where the whole run stops
		const uint32_t run_len = run_end - rs;
		uint32_t p = i;
		while (p < e) {
			const uint32_t r = p - rs, q = r % 255u;
			if (q < 4) {
				const uint32_t reclen = min(255u, run_len - (r - q));
				emit(o++, (uint8_t)ch);
				if (q == 3) { emit(o++, (uint8_t)(reclen - 4)); rec_end(o, rs + (r - 3) + reclen); }
				else if (q + 1 == reclen) rec_end(o, rs + r + 1);
				p++;
			} else p += 255u - q;                                   // the rest of this 255-record emits nothing
		}
		i = e;
	}
}

// 8 wrap-around bytes after a block's text (the sort reads text[i + 0..7]) and zero padding to a multiple of 4; t = 0..11
__device__ __forceinline__ void rle1_wrap(uint8_t* ok, uint32_t nk, uint32_t t)
{
	const uint32_t pos = nk + t;
	if (t < 8) ok[pos] = ok[t % nk];
	else if (pos < ((nk + 8 + 3) & ~3u)) ok[pos] = 0;
}

// ---- D. CRC-32 of b[lo, lo + len): per-chunk table CRC (chunks right aligned inside the range: only the first non-empty one is
// short and carries the 0xFFFFFFFF start value), combined in a binary tree with carry-less multiplications by x^(8 len) mod P.
// Returns the block CRC (bzip2's final complement applied) in every thread.  Contains barriers.
template <int NT>
__device__ __forceinline__ uint32_t rle1_crc(const uint8_t* b, uint32_t lo, uint32_t len, const uint32_t* crc_tab, uint32_t* s_a, uint32_t* s_b)
{
	const uint32_t tid = threadIdx.x;
	uint32_t CC = ((len + NT - 1) / NT + 3) & ~3u;
	if (((CC >> 2) & 1u) == 0) CC += 4;
	const uint32_t aft = (NT - 1 - tid) * CC;
	const uint32_t x1 = len > aft ? len - aft : 0;
	const uint32_t x0 = x1 > CC ? x1 - CC : 0;
	uint32_t crc = 0;
	if (x1 > x0) {
		crc = (x0 == 0) ? 0xFFFFFFFFu : 0u;
		for (uint32_t j = lo + x0; j < lo + x1; j++) crc = (crc << 8) ^ crc_tab[(crc >> 24) ^ b[j]];
	}
	__syncthreads();
	s_a[tid] = crc;
	__syncthreads();
	// x^(8 CC 2^k) mod P for the k-th tree level: thread k squares k times (instead of every thread squaring at every level)
	if (tid < 12) { uint32_t M = crc_xpow8(CC); for (uint32_t q = 0; q < tid; q++) M = crc_mulmod(M, M); s_b[tid] = M; }
	__syncthreads();
	{
		uint32_t lvl = 0;
		for (uint32_t stride = 1; stride < NT; stride <<= 1, lvl++) {
			if ((tid & (2 * stride - 1)) == 0) s_a[tid] = crc_mulmod(s_a[tid], s_b[lvl]) ^ s_a[tid + stride];
			__syncthreads();
		}
	}
	return ~s_a[0];
}

}  // namespace lfm
