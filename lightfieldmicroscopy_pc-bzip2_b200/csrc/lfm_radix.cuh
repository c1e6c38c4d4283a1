// lfm_radix.cuh -- CTA-wide stable 8-bit counting-sort pass and group-splitting helpers shared by the
// BWT (bz_bwt.cu) and the inverse BWT (bz_decode.cu).
#pragma once
#include "lfm_device.cuh"

namespace lfm {

constexpr int BWT_NT = 1024;
constexpr int BWT_R  = 12;                // elements per thread per radix tile (4-byte payloads)
constexpr int BWT_WS = 257;               // row stride (words) of the per-warp digit counters: conflict-free rows AND columns;
                                          // column 256 is the dummy digit of the lanes past the end of the data
constexpr int SPLIT_R = 4;                // elements per thread per tile in split_groups
#define LFM_WC(w, d) wcnt[(w) * BWT_WS + (d)]

struct Trip { uint32_t g, r, v; };

// One stable 8-bit counting-sort pass over m elements, tile by tile (tile = BWT_NT * R elements).
// run[256] (shared) must hold the exclusive bucket starts on entry; it is advanced as tiles are placed.
// wcnt: NT / 32 x BWT_WS shared words; every warp owns (and zeroes) its own row.
//   1. all loads of the tile are issued first (independent global loads in flight together);
//   2. ranking inside the warp: R match.any instructions back to back, then R shared-memory atomics by the group
//      leaders (issued back to back: the counter update is ordered by the memory pipe, not by a register dependency),
//      then R shuffles that hand the old counter value to the group -- three software-pipelined sweeps instead of
//      R serialised load/modify/store rounds;
//   3. the per-warp digit counts are scanned ACROSS warps by warp shuffles (warp w owns digits 8w..8w+7);
//   4. scatter; the warp clears its own counter row for the next tile (two CTA barriers per tile in all).
// NT = threads of the CTA: 1024 (one CTA per SM, blocks of 100 KB and more) or 256 (four CTAs per SM: small blocks, where whole
// 12288-element tiles and 148-CTA waves would leave a third of the machine idle).
template <int R, class P, int NT = BWT_NT, class LoadFn, class DigitFn, class StoreFn>
__device__ __forceinline__ void radix_scatter(uint32_t m, uint32_t* run, uint32_t* wcnt,
                                              LoadFn load, DigitFn digit, StoreFn store)
{
	const uint32_t lane = lane_id(), w = warp_id();
	const uint32_t lt = (1u << lane) - 1u;
	constexpr uint32_t TILE = NT * R;
	uint32_t* myc = wcnt + w * BWT_WS;
	__syncthreads();                                      // earlier users of wcnt / run are done
	for (uint32_t i = lane; i < BWT_WS; i += 32) myc[i] = 0;
	__syncwarp();
	for (uint32_t t0 = 0; t0 < m; t0 += TILE) {
		P pay[R]; uint32_t dl[R];                         // digit << 16 | rank inside the warp
		const uint32_t eb = t0 + w * (32 * R) + lane;
		#pragma unroll
		for (int r = 0; r < R; r++) if (eb + r * 32 < m) pay[r] = load(eb + r * 32);
		#pragma unroll
		for (int r = 0; r < R; r++) dl[r] = (eb + r * 32 < m) ? digit(pay[r]) : 256u;
		constexpr int RH = R > 8 ? R / 2 : R;                // ranking sweeps over at most 8 elements at a time (register budget)
		#pragma unroll
		for (int r0 = 0; r0 < R; r0 += RH) {
			uint32_t peers[RH], old[RH];
			#pragma unroll
			for (int r = 0; r < RH; r++) peers[r] = __match_any_sync(0xffffffffu, dl[r0 + r]);
			#pragma unroll
			for (int r = 0; r < RH; r++) {
				old[r] = 0;
				if ((peers[r] & lt) == 0) old[r] = atomicAdd(&myc[dl[r0 + r]], (uint32_t)__popc(peers[r]));
				__syncwarp();
			}
			#pragma unroll
			for (int r = 0; r < RH; r++) {
				const uint32_t o = __shfl_sync(0xffffffffu, old[r], __ffs(peers[r]) - 1);
				dl[r0 + r] = (dl[r0 + r] << 16) | (o + __popc(peers[r] & lt));
			}
		}
		__syncthreads();
		if constexpr (NT == 256) {
			// 8 warps: thread d owns the counters of digit d in all of them (bank = (i + d) mod 32: conflict free)
			const uint32_t d = threadIdx.x;
			uint32_t* col = wcnt + d;
			uint32_t c[8];
			#pragma unroll
			for (int i = 0; i < 8; i++) c[i] = col[i * BWT_WS];
			uint32_t acc = run[d];
			#pragma unroll
			for (int i = 0; i < 8; i++) { col[i * BWT_WS] = acc; acc += c[i]; }
			run[d] = acc;
		} else {
			// exclusive scan over the warps, digit by digit: thread (d, part) owns the counters of digit d in warps
			// 8*part .. 8*part+7 (bank = (8*part + i + d) mod 32: conflict free), the 4 parts are adjacent lanes
			static_assert(NT == 1024, "scan layouts exist for 1024 and 256 threads");
			const uint32_t d = threadIdx.x >> 2, part = threadIdx.x & 3u;
			uint32_t* col = wcnt + (part * 8) * BWT_WS + d;
			uint32_t c[8], tot = 0;
			#pragma unroll
			for (int i = 0; i < 8; i++) { c[i] = col[i * BWT_WS]; tot += c[i]; }
			uint32_t incl = tot;
			uint32_t t1 = __shfl_up_sync(0xffffffffu, incl, 1); if (part >= 1) incl += t1;
			uint32_t t2 = __shfl_up_sync(0xffffffffu, incl, 2); if (part >= 2) incl += t2;
			uint32_t acc = run[d] + incl - tot;
			#pragma unroll
			for (int i = 0; i < 8; i++) { col[i * BWT_WS] = acc; acc += c[i]; }
			__syncwarp();
			if (part == 3) run[d] = acc;
		}
		__syncthreads();
		#pragma unroll
		for (int r = 0; r < R; r++) if (eb + r * 32 < m) store(myc[dl[r] >> 16] + (dl[r] & 0xffffu), pay[r]);
		__syncwarp();
		for (uint32_t i = lane; i < BWT_WS; i += 32) myc[i] = 0;
		__syncwarp();
	}
	__syncthreads();
}

// per-warp private histograms (match.any aggregated) of an 8-bit digit over m elements,
// reduced and exclusive-scanned into run[256]
template <int NT = BWT_NT, class DigitOfIndex>
__device__ __forceinline__ void digit_starts(uint32_t m, uint32_t* run, uint32_t* wcnt, uint32_t* red, DigitOfIndex dig)
{
	const uint32_t lane = lane_id(), w = warp_id();
	const uint32_t lt = (1u << lane) - 1u;
	uint32_t* myc = wcnt + w * BWT_WS;
	constexpr int U = 4;
	__syncthreads();
	for (uint32_t i = lane; i < BWT_WS; i += 32) myc[i] = 0;
	__syncwarp();
	for (uint32_t e0 = w * (32 * U); e0 < m; e0 += NT * U) {        // warp-uniform trip count
		uint32_t d[U], peers[U];
		#pragma unroll
		for (int u = 0; u < U; u++) { const uint32_t e = e0 + u * 32 + lane; d[u] = e < m ? dig(e) : 256u; }
		#pragma unroll
		for (int u = 0; u < U; u++) peers[u] = __match_any_sync(0xffffffffu, d[u]);
		#pragma unroll
		for (int u = 0; u < U; u++) if ((peers[u] & lt) == 0) atomicAdd(&myc[d[u]], (uint32_t)__popc(peers[u]));
	}
	__syncthreads();
	if (threadIdx.x < 256) {
		uint32_t s = 0;
		#pragma unroll 8
		for (int ww = 0; ww < NT / 32; ww++) s += LFM_WC(ww, threadIdx.x);
		run[threadIdx.x] = s;
	}
	__syncthreads();
	scan256_excl<NT>(run, red);
}

// Walk cnt sorted entries; entry j is a group head when its 64-bit key differs from the key of entry j-1.
// group head value pos_of(j) is propagated to the members (max-scan, heads ascend), singleton groups are resolved,
// the others are appended (compacted, order kept) to the next unresolved set.
// emit(j, head, unresolved, slot) is called once per entry. Returns the number of unresolved entries.
template <int NT = BWT_NT, class KeyFn, class PosFn, class EmitFn>
__device__ __forceinline__ uint32_t split_groups(uint32_t cnt, uint32_t* red, KeyFn key_of, PosFn pos_of, EmitFn emit)
{
	uint32_t carry_head = 0, carry_cnt = 0;
	for (uint32_t t0 = 0; t0 < cnt; t0 += NT * SPLIT_R) {
		uint32_t i0 = t0 + threadIdx.x * SPLIT_R;
		bool hd[SPLIT_R + 1]; uint32_t gh[SPLIT_R];
		{
			uint64_t ky[SPLIT_R + 2];
			#pragma unroll
			for (int r = 0; r < SPLIT_R + 2; r++) { const uint32_t j = i0 + r; ky[r] = (j >= 1 && j <= cnt) ? key_of(j - 1) : 0; }
			#pragma unroll
			for (int r = 0; r <= SPLIT_R; r++) { const uint32_t j = i0 + r; hd[r] = (j == 0 || j >= cnt) ? true : (ky[r] != ky[r + 1]); }
		}
		uint32_t local = 0;
		#pragma unroll
		for (int r = 0; r < SPLIT_R; r++) { if (i0 + r < cnt && hd[r]) local = pos_of(i0 + r); gh[r] = local; }
		uint32_t incl = block_scan_max<NT>(local, red);
		uint32_t tile_max = red[NT / 32 - 1];
		uint32_t before = __shfl_up_sync(0xffffffffu, incl, 1);
		if (lane_id() == 0) before = warp_id() ? red[warp_id() - 1] : 0;
		before = max(before, carry_head);
		uint32_t c = 0; bool un[SPLIT_R];
		#pragma unroll
		for (int r = 0; r < SPLIT_R; r++) {
			gh[r] = max(gh[r], before);
			un[r] = (i0 + r < cnt) && !(hd[r] && hd[r + 1]);
			c += un[r];
		}
		uint32_t tot; uint32_t inc = block_scan_add<NT>(c, red, &tot);
		uint32_t o = carry_cnt + inc - c;
		#pragma unroll
		for (int r = 0; r < SPLIT_R; r++) if (i0 + r < cnt) { emit(i0 + r, gh[r], un[r], o); o += un[r]; }
		carry_cnt += tot;
		carry_head = max(carry_head, tile_max);
	}
	__syncthreads();
	return carry_cnt;
}

}  // namespace lfm
