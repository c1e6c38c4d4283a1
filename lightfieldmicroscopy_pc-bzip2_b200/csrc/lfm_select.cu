// lfm_select.cu -- "2-D entropy" predictor-mode selection on frame 0.
//
// Replaces klb_imageIO::predict_and_2DEntropy / bwt_entropy_2D (src/klb_imageIO.cpp:2030-2093, :2197-2225) and the
// kernels + thrust calls behind them (src/lfm_Predictors.cu:2833-2949: bwtKernel + sort_by_key, static_bwt_Kernel,
// sum_bwt_Kernel + reduce).  Per candidate and per 450000-pixel chunk:
//   1. pairs (key = b[j], val = b[j-1]) j = 0..n-1 with b[-1] = 0, plus (key 0, val b[n-1]); STABLE sort by key
//   2. histogram of adjacent value pairs (S[x] << 8 | S[x+1]), x = 0..n-1
//   3. E = sum over bins 0..65534 of -P ln P, P = (float)cnt / (float)n   (bin 65535 is never summed)
// The integer part is exact; the per-bin terms are fp32 like the reference, summed in a fixed order in fp64
// (the reference's fp32 thrust::reduce order is unspecified, SURVEY.md Appendix C).
#include "lfm_device.cuh"

namespace lfm {

struct CandPtrs { const uint16_t* p[8]; };

constexpr int SE_NT = 1024;
__global__ void __launch_bounds__(SE_NT)
k_select_entropy(const uint32_t* __restrict__ hist_all, uint64_t fpx, uint32_t chunk_px, uint32_t nchunks,
                 float* __restrict__ e_out)
{
	__shared__ double part[SE_NT];
	const uint32_t cc = blockIdx.x, chunk = cc % nchunks;
	const uint64_t px0 = (uint64_t)chunk * chunk_px;
	const uint32_t n = (uint32_t)(min((uint64_t)chunk_px, fpx - px0) * 2);
	const uint32_t* hist = hist_all + (size_t)cc * 65536;
	double acc = 0.0;
	const float fn = (float)n;
	for (uint32_t kbin = threadIdx.x * 64; kbin < threadIdx.x * 64 + 64; kbin++) {
		if (kbin >= 65535) break;
		uint32_t c = hist[kbin];
		if (c) { float P = (float)c / fn; float t = -1.0f * P * logf(P); acc += (double)t; }
	}
	part[threadIdx.x] = acc;
	__syncthreads();
	for (int s = SE_NT / 2; s > 0; s >>= 1) {
		if ((int)threadIdx.x < s) part[threadIdx.x] += part[threadIdx.x + s];
		__syncthreads();
	}
	if (threadIdx.x == 0) e_out[cc] = (float)part[0];
}

// ---- the same pair histogram WITHOUT the sort.  The stably sorted value list is, bucket after bucket, the values val(j) = b[j-1]
// of the positions j that hold key b[j] = c, in position order.  So its adjacent pairs are
//   (val(j), val(next(j)))   for every position j that has a later position next(j) with the same key, and
//   (val(last position of c), val(first position of c'))   for consecutive non-empty buckets c < c',
// and "the next position with the same key" needs no sort:
//   k_select_next   one warp per segment of SN_SEG positions walks it BACKWARD 32 positions at a time with a 256-entry table of the
//                   nearest later value per key (match.any finds the pairs inside a group of 32), counts the pairs it can close, and
//                   leaves, per key, the value at its first and at its last position of the segment;
//   k_select_link   one thread per key chains the segments (last of one -> first of the next one that holds the key) and one
//                   thread closes the bucket boundaries.
// Integer result identical to the sorted formulation (tests: entropies and winners against the reference's, file bytes).
constexpr uint32_t SN_SEG = 2048;                 // positions per warp and round
constexpr int SN_WARPS = 8;
constexpr int SN_PARTS = 8;                       // CTAs per (candidate, chunk): each walks every SN_PARTS-th group of SN_WARPS segments
constexpr uint32_t SN_HOT = 32;                   // pairs whose first byte is below this are counted in shared memory
constexpr uint16_t SN_NONE = 0xFFFFu;
// ncu of the first version (one match.any for the key, one to aggregate equal pairs before the global atomic): MIO bound, 24 % of
// the issue slots.  Now ONE match.any (the key peers; eight ballots were measured slower: 0.78 against 0.70 ms), and the pairs whose first byte is small -- high bytes and small
// residuals: most of them, and the ones that would contend for the same global counter -- go to a 32 x 256 shared-memory
// histogram that the CTA adds to the global one once, after ~55 segments; the others are spread over 57 K counters.
__global__ void __launch_bounds__(32 * SN_WARPS)
k_select_next(CandPtrs cands, uint64_t fpx, uint32_t chunk_px, uint32_t nchunks, uint16_t* __restrict__ tabs_all, uint32_t tstride,
              uint32_t* __restrict__ hist_all)
{
	extern __shared__ __align__(16) uint8_t sn_smem[];
	uint32_t* hot = reinterpret_cast<uint32_t*>(sn_smem);                            // [SN_HOT][256]
	uint16_t (*tab_s)[256] = reinterpret_cast<uint16_t (*)[256]>(sn_smem + SN_HOT * 256 * 4);
	uint8_t (*seg_s)[16 + SN_SEG] = reinterpret_cast<uint8_t (*)[16 + SN_SEG]>(sn_smem + SN_HOT * 256 * 4 + SN_WARPS * 256 * 2);
	const uint32_t lane = lane_id(), w = warp_id();
	const uint32_t chunk = blockIdx.y, cand = blockIdx.z, cc = cand * nchunks + chunk;
	const uint64_t px0 = (uint64_t)chunk * chunk_px;
	const uint32_t n = (uint32_t)(min((uint64_t)chunk_px, fpx - px0) * 2);          // positions 0 .. n (n + 1 of them)
	const uint32_t nseg = (n + 1 + SN_SEG - 1) / SN_SEG;
	const uint8_t* b = reinterpret_cast<const uint8_t*>(cands.p[cand] + px0);
	uint32_t* hist = hist_all + (size_t)cc * 65536;
	uint16_t* tab = tab_s[w];
	uint8_t* sb = seg_s[w] + 16;                                                     // sb[i] = b[j0 + i], sb[-1] = b[j0 - 1]
	const uint32_t lt_incl = (2u << lane) - 1u;                                      // lanes <= this one (lane 31: all)
	for (uint32_t i = threadIdx.x; i < SN_HOT * 256; i += 32 * SN_WARPS) hot[i] = 0;
	__syncthreads();
	for (uint32_t seg = blockIdx.x * SN_WARPS + w; seg < nseg; seg += SN_PARTS * SN_WARPS) {
		uint16_t* first = tabs_all + (size_t)cc * tstride + (size_t)seg * 512, * last = first + 256;
		for (uint32_t i = lane; i < 256; i += 32) { tab[i] = SN_NONE; last[i] = SN_NONE; }
		const uint32_t j0 = seg * SN_SEG, j1 = min(n + 1, j0 + SN_SEG);
		// the segment's bytes once, coalesced (a group of 32 positions per iteration would pay a DRAM latency per iteration)
		for (uint32_t q = lane * 16; q < SN_SEG; q += 32 * 16) {
			uint4 v = make_uint4(0u, 0u, 0u, 0u);
			if (j0 + q + 16 <= n && (reinterpret_cast<uintptr_t>(b + j0 + q) & 15u) == 0u) v = *reinterpret_cast<const uint4*>(b + j0 + q);   // (frames of odd sizes are not 16-byte aligned)
			else { uint32_t wv[4] = { 0u, 0u, 0u, 0u }; for (int k = 0; k < 16; k++) if (j0 + q + k < n) wv[k >> 2] |= (uint32_t)b[j0 + q + k] << (8 * (k & 3)); v = make_uint4(wv[0], wv[1], wv[2], wv[3]); }
			*reinterpret_cast<uint4*>(sb + q) = v;
		}
		if (lane == 0) sb[-1] = j0 ? b[j0 - 1] : (uint8_t)0;
		__syncwarp();
		for (uint32_t g1 = j1; g1 > j0; ) {                                          // groups of 32 positions, last group first
			const uint32_t g0 = g1 - j0 > 32u ? g1 - 32u : j0;
			// group [g0, g1): lane l holds position g0 + l; the first (partial) group of a segment is aligned at its START
			const uint32_t j = g0 + lane;
			const bool act = j < g1;
			const uint32_t am = __ballot_sync(0xffffffffu, act);
			uint32_t key = 0, val = 0;
			if (act) { key = sb[(int)(j - j0)]; val = sb[(int)(j - j0) - 1]; }         // position n holds key 0 (staged as 0), b[-1] = 0
			const uint32_t peers = __match_any_sync(0xffffffffu, act ? key : 256u) & am;   // lanes with the same key
			const uint32_t higher = peers & ~lt_incl;
			const uint32_t partner = (act && higher) ? (uint32_t)__ffs((int)higher) - 1u : lane;
			uint32_t pv = __shfl_sync(0xffffffffu, val, partner);
			if (act) {
				bool has = higher != 0u;
				if (!has) { const uint32_t t = tab[key]; has = t != SN_NONE; pv = t; if (!has) last[key] = (uint16_t)val; }   // no later position in the segment: its last one
				if (has) {
					if (val < SN_HOT) atomicAdd(&hot[val * 256 + pv], 1u);
					else atomicAdd(&hist[(val << 8) | pv], 1u);
				}
			}
			__syncwarp();
			if (act && (peers & (lt_incl >> 1)) == 0u) tab[key] = (uint16_t)val;       // first position of the key in the group: the nearest later one for what comes before
			__syncwarp();
			g1 = g0;
		}
		for (uint32_t i = lane; i < 256; i += 32) first[i] = tab[i];
		__syncwarp();
	}
	__syncthreads();
	for (uint32_t i = threadIdx.x; i < SN_HOT * 256; i += 32 * SN_WARPS) { const uint32_t c = hot[i]; if (c) atomicAdd(&hist[i], c); }
}

constexpr int SL_Q = 4;                            // segment ranges per key, chained by different threads
__global__ void __launch_bounds__(256 * SL_Q)
k_select_link(const uint16_t* __restrict__ tabs_all, uint32_t tstride, uint64_t fpx, uint32_t chunk_px, uint32_t nchunks,
              uint32_t* __restrict__ hist_all)
{
	__shared__ uint16_t first_q[SL_Q][256], last_q[SL_Q][256];
	__shared__ uint16_t first_all[256], last_all[256];
	const uint32_t cc = blockIdx.x, chunk = cc % nchunks, c = threadIdx.x & 255u, qd = threadIdx.x >> 8;
	const uint64_t px0 = (uint64_t)chunk * chunk_px;
	const uint32_t n = (uint32_t)(min((uint64_t)chunk_px, fpx - px0) * 2);
	const uint32_t nseg = (n + 1 + SN_SEG - 1) / SN_SEG;
	const uint32_t per = (nseg + SL_Q - 1) / SL_Q, sA = min(nseg, qd * per), sB = min(nseg, sA + per);
	const uint16_t* tabs = tabs_all + (size_t)cc * tstride;
	uint32_t* hist = hist_all + (size_t)cc * 65536;
	uint32_t carry = SN_NONE, f0 = SN_NONE;
	for (uint32_t s0 = sA; s0 < sB; s0 += 16) {                                      // sixteen segments' entries in flight
		uint32_t f[16], l[16];
		#pragma unroll
		for (int k = 0; k < 16; k++) {
			const uint32_t sg = s0 + k;
			f[k] = sg < sB ? tabs[(size_t)sg * 512 + c] : (uint32_t)SN_NONE;
			l[k] = sg < sB ? tabs[(size_t)sg * 512 + 256 + c] : (uint32_t)SN_NONE;
		}
		#pragma unroll
		for (int k = 0; k < 16; k++) if (f[k] != SN_NONE) {
			if (carry != SN_NONE) atomicAdd(&hist[(carry << 8) | f[k]], 1u);
			else f0 = f[k];
			carry = l[k];
		}
	}
	first_q[qd][c] = (uint16_t)f0; last_q[qd][c] = (uint16_t)carry;
	__syncthreads();
	if (qd == 0) {                                                                   // the ranges of a key, in order
		uint32_t cy = SN_NONE, fa = SN_NONE;
		#pragma unroll
		for (int q = 0; q < SL_Q; q++) {
			const uint32_t f = first_q[q][c], l = last_q[q][c];
			if (f != SN_NONE) {
				if (cy != SN_NONE) atomicAdd(&hist[(cy << 8) | f], 1u);
				else fa = f;
				cy = l;
			}
		}
		first_all[c] = (uint16_t)fa; last_all[c] = (uint16_t)cy;
	}
	__syncthreads();
	if (threadIdx.x == 0) {                                                          // bucket boundaries
		uint32_t prev = SN_NONE;
		for (int k = 0; k < 256; k++) if (first_all[k] != SN_NONE) {
			if (prev != SN_NONE) atomicAdd(&hist[(prev << 8) | first_all[k]], 1u);
			prev = last_all[k];
		}
	}
}

// tabs: select_table_bytes(); hist: ncand*nchunks*65536 uint32 (zeroed here); e_out: ncand*nchunks floats
static uint32_t select_segments(uint32_t chunk_px) { return (chunk_px * 2 + 1 + SN_SEG - 1) / SN_SEG; }
size_t select_table_bytes(int ncand, uint32_t chunk_px, uint32_t nchunks) { return (size_t)ncand * nchunks * select_segments(chunk_px) * 1024; }
void launch_select(const uint16_t* const cand_ptrs[8], int ncand, uint64_t fpx, uint32_t chunk_px, uint32_t nchunks,
                   uint16_t* tabs, uint32_t* hist, float* e_out, cudaStream_t st)
{
	CandPtrs cp;
	for (int i = 0; i < 8; i++) cp.p[i] = cand_ptrs[i < ncand ? i : 0];
	cudaMemsetAsync(hist, 0, (size_t)ncand * nchunks * 65536 * sizeof(uint32_t), st);
	const uint32_t tstride = select_segments(chunk_px) * 512;                          // uint16 elements per (candidate, chunk)
	const size_t sn_smem = (size_t)SN_HOT * 256 * 4 + (size_t)SN_WARPS * 256 * 2 + (size_t)SN_WARPS * (16 + SN_SEG);
	cudaFuncSetAttribute(k_select_next, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sn_smem);
	k_select_next<<<dim3(SN_PARTS, nchunks, ncand), 32 * SN_WARPS, sn_smem, st>>>(cp, fpx, chunk_px, nchunks, tabs, tstride, hist);
	k_select_link<<<ncand * nchunks, 256 * SL_Q, 0, st>>>(tabs, tstride, fpx, chunk_px, nchunks, hist);
	k_select_entropy<<<ncand * nchunks, SE_NT, 0, st>>>(hist, fpx, chunk_px, nchunks, e_out);
}

}  // namespace lfm
