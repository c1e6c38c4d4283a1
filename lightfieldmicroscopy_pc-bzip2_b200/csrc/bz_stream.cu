// bz_stream.cu -- standalone bzip2 streams of arbitrary byte buffers, for sm_100a.
//
// Output byte-identical to BZ2_bzBuffToBuffCompress(dst, &len, src, n, level, 0, 30) for any n < 2^32 and level 1..9.  The per-block
// stages are those of the KLB path (k_bwt, k_mtf, k_huff_pack, with the stream header and trailer flags); what is new is what
// "one KLB block = one stream of at most kMaxSub blocks" does not cover:
//   k_sz_heads / k_sz_scan_heads   run heads of the whole input: first / last head of every tile, then the run open at every tile
//                                  start (exclusive max-scan) and the first head after every tile (suffix min-scan)
//   k_sz_tiles (count)             RLE1 output bytes of every tile (phases B/C of k_rle1, bz_rle1.cuh, with the run context of the
//                                  tile's neighbours), k_sz_scan_sum: tile output offsets
//   k_sz_tiles (ends)              bitmap of the record ends in output coordinates
//   k_sz_chain                     bzip2 block boundaries: block k+1 starts at the first record end >= start_k + nblockMAX, unless
//                                  only one more output byte follows (bzlib.c:216-354, handle_compress in BZ_FINISH mode).  The
//                                  only sequential loop: one bitmap word per block (record ends are at most 5 output bytes apart)
//   k_sz_locate                    input offset of every block start (one CTA re-walks the tile that holds it)
//   k_sz_emit                      per block: RLE1 text into the block's slot, block CRC, EncJob record (phases B-D of k_rle1),
//                                  combined CRC as an XOR of rotated block CRCs
//   k_sz_offsets / k_sz_assemble   exclusive scan of the blocks' bit lengths; every thread assembles whole output words from the
//                                  blocks' bit strings (blocks are not byte aligned inside a stream, compress.c:603-676)
#include "bz_rle1.cuh"
#include "kernels.h"

namespace lfm {

constexpr int SZ_NT = 256;                 // tile kernels
constexpr int SE_NT = 1024;                // one CTA per bzip2 block
constexpr int SC_NT = 1024;                // single-CTA scans over the tile records

uint32_t sz_tiles(uint64_t n) { return (uint32_t)((n + kSzTile - 1) / kSzTile); }

// inclusive scan of 64-bit values over the CTA; *total = sum.  red64: >= 32 shared words.  Contains barriers.
template <int NT>
__device__ __forceinline__ uint64_t block_scan_add64(uint64_t v, uint64_t* red64, uint64_t* total)
{
	const uint32_t lane = lane_id(), w = warp_id();
	#pragma unroll
	for (int o = 1; o < 32; o <<= 1) { const uint64_t t = __shfl_up_sync(0xffffffffu, v, o); if (lane >= (uint32_t)o) v += t; }
	__syncthreads();
	if (lane == 31) red64[w] = v;
	__syncthreads();
	if (w == 0) {
		uint64_t s = lane < NT / 32 ? red64[lane] : 0;
		#pragma unroll
		for (int o = 1; o < 32; o <<= 1) { const uint64_t t = __shfl_up_sync(0xffffffffu, s, o); if (lane >= (uint32_t)o) s += t; }
		red64[lane] = s;
	}
	__syncthreads();
	const uint64_t off = w ? red64[w - 1] : 0;
	*total = red64[NT / 32 - 1];
	return v + off;
}

// ---- first / last run head of every tile (global index + 1, 0 = none)
__global__ void __launch_bounds__(SZ_NT)
k_sz_heads(const uint8_t* __restrict__ src, uint32_t n, uint32_t* __restrict__ tfirst, uint32_t* __restrict__ tlast)
{
	__shared__ uint32_t red[64];
	const uint32_t lo = blockIdx.x * kSzTile, hi = (uint32_t)min((uint64_t)n, (uint64_t)lo + kSzTile);
	constexpr uint32_t PER = kSzTile / SZ_NT;
	const uint32_t a = min(hi, lo + threadIdx.x * PER), b = min(hi, a + PER);
	uint32_t first = 0, last = 0;
	for (uint32_t i = a; i < b; i++)
		if (i == 0 || src[i] != src[i - 1]) { if (!first) first = i + 1; last = i + 1; }
	const uint32_t mx = block_scan_max<SZ_NT>(last, red);
	__syncthreads();
	const uint32_t mn = block_scan_max<SZ_NT>(first ? ~first : 0u, red);       // max of ~v = min of v over the non-empty
	if (threadIdx.x == SZ_NT - 1) { tlast[blockIdx.x] = mx; tfirst[blockIdx.x] = mn ? ~mn : 0u; }
}

// ---- run context of every tile: topen[t] = start of the run open at the tile start, tnext[t] = first head at or after its end.
// One CTA, each thread a contiguous segment of tiles (the tile records are 1/kSzTile of the input).
__global__ void __launch_bounds__(SC_NT)
k_sz_scan_heads(uint32_t ntiles, uint32_t n, const uint32_t* __restrict__ tfirst, const uint32_t* __restrict__ tlast,
                uint32_t* __restrict__ topen, uint32_t* __restrict__ tnext)
{
	__shared__ uint32_t red[64];
	const uint32_t tid = threadIdx.x, lane = lane_id(), wid = warp_id();
	const uint32_t P = (ntiles + SC_NT - 1) / SC_NT;
	const uint32_t a = min(ntiles, tid * P), b = min(ntiles, a + P);
	uint32_t mx = 0;
	for (uint32_t t = a; t < b; t++) mx = max(mx, tlast[t]);
	uint32_t incl = block_scan_max<SC_NT>(mx, red);
	uint32_t prev = __shfl_up_sync(0xffffffffu, incl, 1);
	if (lane == 0) prev = wid ? red[wid - 1] : 0;
	for (uint32_t t = a; t < b; t++) { topen[t] = prev ? prev - 1 : 0; prev = max(prev, tlast[t]); }
	__syncthreads();
	// suffix min of tfirst: thread r owns segment SC_NT-1-r, a max-scan of ~first over r
	const uint32_t r = SC_NT - 1 - tid;
	const uint32_t ra = min(ntiles, r * P), rb = min(ntiles, ra + P);
	uint32_t mn = 0;                                          // ~(min first) over the segment, 0 = none
	for (uint32_t t = ra; t < rb; t++) if (tfirst[t]) mn = max(mn, ~tfirst[t]);
	incl = block_scan_max<SC_NT>(mn, red);
	prev = __shfl_up_sync(0xffffffffu, incl, 1);
	if (lane == 0) prev = wid ? red[wid - 1] : 0;
	for (uint32_t t = rb; t-- > ra;) {
		tnext[t] = prev ? ~prev - 1 : n;
		if (tfirst[t]) prev = max(prev, ~tfirst[t]);
	}
}

// ---- tobase[t] = RLE1 output offset of tile t (exclusive scan), tobase[ntiles] = total
__global__ void __launch_bounds__(SC_NT)
k_sz_scan_sum(uint32_t ntiles, const uint32_t* __restrict__ tcount, uint64_t* __restrict__ tobase)
{
	__shared__ uint64_t red64[32];
	const uint32_t tid = threadIdx.x;
	const uint32_t P = (ntiles + SC_NT - 1) / SC_NT;
	const uint32_t a = min(ntiles, tid * P), b = min(ntiles, a + P);
	uint64_t s = 0;
	for (uint32_t t = a; t < b; t++) s += tcount[t];
	uint64_t total; uint64_t o = block_scan_add64<SC_NT>(s, red64, &total) - s;
	for (uint32_t t = a; t < b; t++) { tobase[t] = o; o += tcount[t]; }
	if (tid == 0) tobase[ntiles] = total;
}

// ---- one tile with the run context of its neighbours.  count: its RLE1 output bytes.  ends: its record ends into the bitmap
// (bit p set = a record ends after output byte p).
__global__ void __launch_bounds__(SZ_NT)
k_sz_tiles(const uint8_t* __restrict__ src, uint32_t n, const uint32_t* __restrict__ topen, const uint32_t* __restrict__ tnext,
           int ends, uint32_t* __restrict__ tcount, const uint64_t* __restrict__ tobase, uint32_t* __restrict__ bitmap)
{
	__shared__ uint32_t red[64];
	__shared__ uint32_t s_a[SZ_NT], s_b[SZ_NT];
	const uint32_t t = blockIdx.x, lo = t * kSzTile, hi = (uint32_t)min((uint64_t)n, (uint64_t)lo + kSzTile);
	const Rle1Chunk ck = rle1_chunk<SZ_NT>(src, lo, hi, lo == 0, topen[t], tnext[t], red, s_a, s_b);
	const uint32_t outc = rle1_count(src, ck);
	uint32_t total; const uint32_t incs = block_scan_add<SZ_NT>(outc, red, &total);
	if (!ends) { if (threadIdx.x == 0) tcount[t] = total; return; }
	const uint64_t base = tobase[t];
	uint64_t cw = ~0ull; uint32_t bits = 0;                   // my outputs are contiguous: one atomic per word touched
	rle1_walk(src, ck, incs - outc, [](uint32_t, uint8_t) {}, [&](uint32_t o, uint32_t) {
		const uint64_t p = base + o - 1, w = p >> 5;
		if (w != cw) { if (bits) atomicOr(&bitmap[cw], bits); cw = w; bits = 0; }
		bits |= 1u << (p & 31u);
	});
	if (bits) atomicOr(&bitmap[cw], bits);
}

// ---- block boundaries in output coordinates: bout[0..nb], *nb_out = nb.  One thread; one bitmap word per block (the first record
// end at or after T lies in [T, T + 4]).
__global__ void k_sz_chain(const uint32_t* __restrict__ bitmap, const uint64_t* __restrict__ n_out_p, uint32_t nblock_max, uint32_t max_blocks,
                           uint64_t* __restrict__ bout, uint32_t* __restrict__ nb_out)
{
	if (threadIdx.x != 0) return;
	const uint64_t n_out = *n_out_p;
	uint64_t s = 0;
	uint32_t k = 0;
	bout[0] = 0;
	for (;;) {
		const uint64_t T = s + nblock_max;
		if (T + 1 >= n_out || k + 1 >= max_blocks) break;
		uint64_t w = (T - 1) >> 5;
		uint32_t word = bitmap[w] & (0xFFFFFFFFu << ((T - 1) & 31u));
		while (word == 0) word = bitmap[++w];               // the last record ends at n_out: always found
		const uint64_t bnd = (w << 5) + (uint64_t)(__ffs(word) - 1) + 1;
		if (bnd + 1 >= n_out) break;                        // one byte left: the last input byte, flushed into this block
		bout[++k] = bnd;
		s = bnd;
	}
	bout[k + 1] = n_out;
	*nb_out = k + 1;
}

// ---- bin[k] = input offset where block k starts (k = 1 .. nb-1): CTA k-1 re-walks the tile that holds output byte bout[k] - 1
__global__ void __launch_bounds__(SZ_NT)
k_sz_locate(const uint8_t* __restrict__ src, uint32_t n, uint32_t ntiles, const uint32_t* __restrict__ topen, const uint32_t* __restrict__ tnext,
            const uint64_t* __restrict__ tobase, const uint64_t* __restrict__ bout, uint32_t* __restrict__ bin)
{
	__shared__ uint32_t red[64];
	__shared__ uint32_t s_a[SZ_NT], s_b[SZ_NT];
	const uint32_t k = blockIdx.x + 1;
	const uint64_t s = bout[k];
	uint32_t l = 0, r = ntiles - 1;                           // last tile whose output starts at or before s - 1
	while (l < r) { const uint32_t m = (l + r + 1) >> 1; if (tobase[m] <= s - 1) l = m; else r = m - 1; }
	const uint32_t t = l, lo = t * kSzTile, hi = (uint32_t)min((uint64_t)n, (uint64_t)lo + kSzTile);
	const Rle1Chunk ck = rle1_chunk<SZ_NT>(src, lo, hi, lo == 0, topen[t], tnext[t], red, s_a, s_b);
	const uint32_t outc = rle1_count(src, ck);
	uint32_t total; const uint32_t incs = block_scan_add<SZ_NT>(outc, red, &total);
	const uint64_t base = tobase[t];
	const uint64_t o_first = base + incs - outc;
	if (outc != 0 && o_first < s && base + incs >= s)
		rle1_walk(src, ck, incs - outc, [](uint32_t, uint8_t) {}, [&](uint32_t o, uint32_t in_end) { if (base + o == s) bin[k] = in_end; });
}

// ---- one bzip2 block per CTA: RLE1 text of input [bin[k], bin[k+1]) into slot k - k0, block CRC, EncJob record.  A block starts
// at a record boundary, so the records inside it are those of a fresh run-length coder started there.
__global__ void __launch_bounds__(SE_NT)
k_sz_emit(const uint8_t* __restrict__ src, const uint32_t* __restrict__ bin, const uint64_t* __restrict__ bout, uint32_t k0, uint32_t nb,
          uint8_t* __restrict__ txt_all, uint32_t cap, EncJob* __restrict__ jobs, uint32_t* __restrict__ combined)
{
	__shared__ uint32_t crc_tab[256];
	__shared__ uint32_t red[64];
	__shared__ uint32_t s_a[SE_NT], s_b[SE_NT];
	const uint32_t tid = threadIdx.x, k = k0 + blockIdx.x;
	if (tid < 256) crc_tab[tid] = crc_table_entry(tid);
	const uint32_t lo = bin[k], hi = bin[k + 1];
	uint8_t* dst = txt_all + (size_t)blockIdx.x * cap;
	const Rle1Chunk ck = rle1_chunk<SE_NT>(src, lo, hi, true, lo, hi, red, s_a, s_b);
	const uint32_t outc = rle1_count(src, ck);
	uint32_t total; const uint32_t incs = block_scan_add<SE_NT>(outc, red, &total);
	const bool bad = (uint64_t)total != bout[k + 1] - bout[k] || total + 8 > cap;
	if (!bad) rle1_walk(src, ck, incs - outc, [&](uint32_t o, uint8_t v) { dst[o] = v; }, [](uint32_t, uint32_t) {});
	__syncthreads();
	if (!bad && total && tid < 12) rle1_wrap(dst, total, tid);
	const uint32_t bc = rle1_crc<SE_NT>(src, lo, hi - lo, crc_tab, s_a, s_b);
	if (tid == 0) {
		EncJob& J = jobs[blockIdx.x];
		J.raw_bytes = hi - lo; J.n = bad ? 0 : total; J.crc = bc; J.status = bad ? 2u : 0u; J.periodic = 0; J.orig_ptr = 0;
		for (int q = 0; q < 8; q++) J.in_use[q] = 0;          // k_bwt derives the inUse map from its byte histogram
		J.n_in_use = 0; J.n_mtf = 0;
		J.flags = (k == 0 ? kSubFirst : 0u) | (k + 1 == nb ? kSubLast : 0u);
		J.stream_crc = 0; J.total_bits = 0; J.out_bytes = 0;
		// combinedCRC = (combinedCRC << 1 | >> 31) ^ blockCRC over the blocks (bzlib.c) = XOR of blockCRC_k rotated by nb - 1 - k
		const uint32_t sh = (nb - 1 - k) & 31u;
		atomicXor(combined, sh ? (bc << sh) | (bc >> (32 - sh)) : bc);
	}
}

__global__ void k_sz_seal(EncJob* __restrict__ last, const uint32_t* __restrict__ combined)
{
	if (threadIdx.x == 0) last->stream_crc = *combined;
}

// ---- bit offsets of a batch's blocks in the stream: bitoff[0..nj], run->bits carried across batches
__global__ void __launch_bounds__(SC_NT)
k_sz_offsets(const EncJob* __restrict__ jobs, uint32_t nj, uint64_t* __restrict__ bitoff, SzRun* __restrict__ run)
{
	__shared__ uint64_t red64[32];
	__shared__ uint64_t s_base;
	if (threadIdx.x == 0) s_base = run->bits;
	__syncthreads();
	uint32_t err = 0;
	for (uint32_t j0 = 0; j0 < nj; j0 += SC_NT) {
		const uint32_t j = j0 + threadIdx.x;
		uint64_t v = 0;
		if (j < nj) { v = jobs[j].total_bits; err |= jobs[j].status; }
		uint64_t total; const uint64_t inc = block_scan_add64<SC_NT>(v, red64, &total);
		const uint64_t base = s_base;
		if (j < nj) bitoff[j] = base + inc - v;
		__syncthreads();
		if (threadIdx.x == 0) s_base = base + total;
		__syncthreads();
	}
	if (err) atomicOr(&run->err, err);
	if (threadIdx.x == 0) { bitoff[nj] = s_base; run->bits = s_base; }
}

// ---- output words [bitoff[0] / 32, ceil(bitoff[nj] / 32)): each thread one big-endian word at a time, from at most two blocks.
// Words shared with the previous / next batch are OR-ed into the zeroed output.
__global__ void __launch_bounds__(256)
k_sz_assemble(const uint8_t* __restrict__ slots, uint32_t ocap, uint32_t nj, const uint64_t* __restrict__ bitoff,
              uint32_t* __restrict__ out, uint64_t out_words)
{
	const uint64_t B0 = bitoff[0], B1 = bitoff[nj];
	const uint64_t w0 = B0 >> 5, w1 = min((B1 + 31) >> 5, out_words);
	for (uint64_t w = w0 + blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; w < w1; w += (uint64_t)gridDim.x * blockDim.x) {
		const uint64_t wb = w << 5, pe = min(wb + 32, B1);
		uint64_t pos = max(wb, B0);
		uint32_t l = 0, r = nj - 1;                          // last block starting at or before pos
		while (l < r) { const uint32_t m = (l + r + 1) >> 1; if (bitoff[m] <= pos) l = m; else r = m - 1; }
		uint32_t j = l, v = 0;
		while (pos < pe) {
			const uint64_t bend = bitoff[j + 1];
			if (pos >= bend) { j++; continue; }
			const uint32_t take = (uint32_t)(min(pe, bend) - pos);
			const uint64_t lb = pos - bitoff[j];             // bit inside block j's slot (the slot is zero-padded by >= 8 bytes)
			const uint8_t* p = slots + (size_t)j * ocap + (lb >> 3);
			uint64_t x = 0;
			#pragma unroll
			for (int q = 0; q < 8; q++) x = (x << 8) | p[q];
			const uint32_t bits = (uint32_t)((x << (lb & 7u)) >> (64 - take));
			v |= bits << (32 - (uint32_t)(pos - wb) - take);
			pos += take;
		}
		const uint32_t be = __byte_perm(v, 0, 0x0123);
		if (wb >= B0 && wb + 32 <= B1) out[w] = be;
		else atomicOr(&out[w], be);
	}
}

// =====================================================================================================
// Reading any .bz2 data: one or more concatenated streams, any level, randomised blocks.
//   k_bz_magic (count, write)   every bit offset of the input is tested for the block magic 0x314159265359 and the end-of-stream
//                               magic 0x177245385090 (a thread owns 32 byte positions, the 48-bit windows cross every border);
//                               the candidates are compacted in bit order: tile counts, k_sz_scan_sum, tile-local scan
//   k_huff_decode<SINGLE>       (bz_decode.cu) every candidate decoded as its own block from its bit: where it ends, its CRC
//   k_bz_link                   successor of every candidate = the candidate at its end bit
//   k_bz_chain                  streams from byte 0: "BZh" + level, first block at bit 32, then successor links until an
//                               end-of-stream magic, combined CRC, padding to a byte, next stream or the end.  A candidate off
//                               the chain is a false positive inside Huffman-coded data; a gap is corrupt data.
// =====================================================================================================
constexpr uint64_t kBlockMagic = 0x314159265359ull, kEosMagic = 0x177245385090ull;

__global__ void __launch_bounds__(SZ_NT)
k_bz_magic(const uint8_t* __restrict__ src, uint64_t n, int write, uint32_t* __restrict__ tcount, const uint64_t* __restrict__ tbase,
           uint64_t* __restrict__ cbit, uint8_t* __restrict__ ceos)
{
	__shared__ uint32_t red[64];
	constexpr uint32_t PER = kSzTile / SZ_NT;
	const uint64_t a = (uint64_t)blockIdx.x * kSzTile + threadIdx.x * PER, b = min(n, a + PER);
	const uint64_t nbits = n * 8;
	auto scan = [&](auto hit) {
		uint64_t w = 0;
		for (uint32_t q = 0; q < 8; q++) w = (w << 8) | (a + q < n ? src[a + q] : 0u);
		for (uint64_t i = a; i < b; i++) {
			#pragma unroll
			for (uint32_t j = 0; j < 8; j++) {
				const uint64_t v = (w >> (16 - j)) & 0xFFFFFFFFFFFFull;
				if ((v == kBlockMagic || v == kEosMagic) && i * 8 + j + 48 <= nbits) hit(i * 8 + j, v == kEosMagic);
			}
			w = (w << 8) | (i + 8 < n ? src[i + 8] : 0u);
		}
	};
	uint32_t c = 0;
	scan([&](uint64_t, bool) { c++; });
	uint32_t total; const uint32_t incs = block_scan_add<SZ_NT>(c, red, &total);
	if (!write) { if (threadIdx.x == 0) tcount[blockIdx.x] = total; return; }
	uint64_t o = tbase[blockIdx.x] + incs - c;
	scan([&](uint64_t bit, bool eos) { cbit[o] = bit; ceos[o] = eos ? 1 : 0; o++; });
}

__global__ void k_bz_link(const uint64_t* __restrict__ cbit, uint32_t nc, const uint64_t* __restrict__ cend, uint32_t* __restrict__ succ)
{
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= nc) return;
	const uint64_t e = cend[i];
	uint32_t l = 0, r = nc;
	while (l < r) { const uint32_t m = (l + r) >> 1; if (cbit[m] < e) l = m + 1; else r = m; }
	succ[i] = (e != ~0ull && l < nc && cbit[l] == e) ? l : 0xFFFFFFFFu;
}

// res[0] = blocks on the chain (bbit / blev: bit and stream level of each, in order), res[1] = 0 or 2 (corrupt)
__global__ void k_bz_chain(const uint8_t* __restrict__ src, uint64_t n, const uint64_t* __restrict__ cbit, const uint8_t* __restrict__ ceos,
                           uint32_t nc, const uint64_t* __restrict__ cend, const uint32_t* __restrict__ ccrc, const uint32_t* __restrict__ succ,
                           uint64_t* __restrict__ bbit, uint32_t* __restrict__ blev, uint32_t* __restrict__ res)
{
	if (threadIdx.x != 0) return;
	constexpr uint32_t NIL = 0xFFFFFFFFu;
	auto bits32 = [&](uint64_t b) {
		uint64_t x = 0;
		for (uint32_t q = 0; q < 5; q++) x = (x << 8) | ((b >> 3) + q < n ? src[(b >> 3) + q] : 0u);
		return (uint32_t)(x >> (8 - (b & 7)));
	};
	uint64_t pos = 0;
	uint32_t nb = 0, status = 0;
	do {
		if (pos + 4 > n || src[pos] != 'B' || src[pos + 1] != 'Z' || src[pos + 2] != 'h' || src[pos + 3] < '1' || src[pos + 3] > '9') { status = 2; break; }
		const uint32_t level = src[pos + 3] - '0';
		uint64_t bit = pos * 8 + 32;
		uint32_t l = 0, r = nc;                                   // once per stream: the candidate at bit 32
		while (l < r) { const uint32_t m = (l + r) >> 1; if (cbit[m] < bit) l = m + 1; else r = m; }
		uint32_t c = (l < nc && cbit[l] == bit) ? l : NIL, combined = 0;
		for (;;) {                                                // one dependent step per block
			if (c == NIL) { status = 2; break; }
			if (ceos[c]) {
				if (bit + 80 > n * 8 || bits32(bit + 48) != combined) status = 2;
				pos = (bit + 80 + 7) >> 3;
				break;
			}
			if (cend[c] == ~0ull) { status = 2; break; }
			bbit[nb] = bit; blev[nb] = level; nb++;
			combined = ((combined << 1) | (combined >> 31)) ^ ccrc[c];
			bit = cend[c]; c = succ[c];
		}
	} while (status == 0 && pos < n);
	res[0] = nb; res[1] = status;
}

// ------------------------------------------------------------------------------------------------ launchers
void launch_sz_runs(const uint8_t* src, uint32_t n, uint32_t* tfirst, uint32_t* tlast, uint32_t* topen, uint32_t* tnext, cudaStream_t st)
{
	const uint32_t nt = sz_tiles(n);
	k_sz_heads<<<nt, SZ_NT, 0, st>>>(src, n, tfirst, tlast);
	k_sz_scan_heads<<<1, SC_NT, 0, st>>>(nt, n, tfirst, tlast, topen, tnext);
}
void launch_sz_count(const uint8_t* src, uint32_t n, const uint32_t* topen, const uint32_t* tnext, uint32_t* tcount, uint64_t* tobase,
                     cudaStream_t st)
{
	const uint32_t nt = sz_tiles(n);
	k_sz_tiles<<<nt, SZ_NT, 0, st>>>(src, n, topen, tnext, 0, tcount, nullptr, nullptr);
	k_sz_scan_sum<<<1, SC_NT, 0, st>>>(nt, tcount, tobase);
}
void launch_sz_chain(const uint8_t* src, uint32_t n, const uint32_t* topen, const uint32_t* tnext, const uint64_t* tobase,
                     uint32_t* bitmap, uint64_t bitmap_words, uint32_t nblock_max, uint32_t max_blocks, uint64_t* bout,
                     uint32_t* nb_out, cudaStream_t st)
{
	const uint32_t nt = sz_tiles(n);
	cudaMemsetAsync(bitmap, 0, bitmap_words * 4, st);
	k_sz_tiles<<<nt, SZ_NT, 0, st>>>(src, n, topen, tnext, 1, nullptr, tobase, bitmap);
	k_sz_chain<<<1, 32, 0, st>>>(bitmap, tobase + nt, nblock_max, max_blocks, bout, nb_out);
}
void launch_sz_locate(const uint8_t* src, uint32_t n, const uint32_t* topen, const uint32_t* tnext, const uint64_t* tobase,
                      const uint64_t* bout, uint32_t* bin, uint32_t nb, cudaStream_t st)
{
	if (nb > 1) k_sz_locate<<<nb - 1, SZ_NT, 0, st>>>(src, n, sz_tiles(n), topen, tnext, tobase, bout, bin);
}
void launch_sz_emit(const uint8_t* src, const uint32_t* bin, const uint64_t* bout, uint32_t k0, uint32_t nj, uint32_t nb,
                    uint8_t* txt, uint32_t cap, EncJob* jobs, uint32_t* combined, cudaStream_t st)
{
	k_sz_emit<<<nj, SE_NT, 0, st>>>(src, bin, bout, k0, nb, txt, cap, jobs, combined);
	if (k0 + nj == nb) k_sz_seal<<<1, 32, 0, st>>>(jobs + (nj - 1), combined);
}
void launch_sz_assemble(const EncJob* jobs, uint32_t nj, const uint8_t* slots, uint32_t ocap, uint64_t* bitoff, SzRun* run,
                        uint8_t* out, uint64_t out_cap, int sm_count, cudaStream_t st)
{
	k_sz_offsets<<<1, SC_NT, 0, st>>>(jobs, nj, bitoff, run);
	k_sz_assemble<<<sm_count * 8, 256, 0, st>>>(slots, ocap, nj, bitoff, reinterpret_cast<uint32_t*>(out), out_cap / 4);
}

}  // namespace lfm

namespace lfm {
void launch_bz_magic(const uint8_t* src, uint64_t n, int write, uint32_t* tcount, uint64_t* tbase, uint64_t* cbit, uint8_t* ceos, cudaStream_t st)
{
	const uint32_t nt = sz_tiles(n);
	k_bz_magic<<<nt, SZ_NT, 0, st>>>(src, n, write, tcount, tbase, cbit, ceos);
	if (!write) k_sz_scan_sum<<<1, SC_NT, 0, st>>>(nt, tcount, tbase);
}
void launch_scan_u32(uint32_t count, const uint32_t* in, uint64_t* out, cudaStream_t st)
{
	k_sz_scan_sum<<<1, SC_NT, 0, st>>>(count, in, out);
}
void launch_bz_chain(const uint8_t* src, uint64_t n, const uint64_t* cbit, const uint8_t* ceos, uint32_t nc, const uint64_t* cend,
                     const uint32_t* ccrc, uint32_t* succ, uint64_t* bbit, uint32_t* blev, uint32_t* res, cudaStream_t st)
{
	k_bz_link<<<(nc + 255) / 256, 256, 0, st>>>(cbit, nc, cend, succ);
	k_bz_chain<<<1, 32, 0, st>>>(src, n, cbit, ceos, nc, cend, ccrc, succ, bbit, blev, res);
}
}  // namespace lfm
