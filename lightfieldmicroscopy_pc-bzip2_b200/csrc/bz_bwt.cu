// bz_bwt.cu -- Burrows-Wheeler transform of bzip2 blocks on sm_100a.
//
// Replaces BZ2_blockSort (src/external/bzip2-1.0.6/blocksort.c:1031-1090) as called from BZ2_compressBlock
// (compress.c:603-619) under klb_imageIO::blockCompressor (src/klb_imageIO.cpp:217).  Contract: order the n cyclic
// rotations of the post-RLE1 block, emit the last column and origPtr = rank of rotation 0.
//
// B200 design: ONE CTA per bzip2 block, persistent over the job list.  The whole block text (<= 184 KB for the
// default 96x96x8 uint16 KLB block) lives in shared memory, so each of the 8 LSD radix passes over the 8-byte
// rotation prefix only moves 4-byte rotation indices through L2 and fetches its digit from shared memory.
// Rotations that still tie after 8 bytes are finished by prefix doubling (Larsson-Sadakane) restricted to the
// unresolved set, with the same tile pass.  Exactly periodic blocks keep their ties; rotation 0 is placed last in
// its group (what bzip2 does for the periods met in practice, SURVEY.md Appendix D.3).
#include "lfm_radix.cuh"

namespace lfm {

// scratch layout per CTA (uint32 arrays of `cap` elements each)
enum { S_SA0 = 0, S_SA1, S_ISA, S_G0, S_G1, S_R0, S_R1, S_V0, S_V1, S_U0, S_U1, S_COUNT };

extern __shared__ __align__(16) uint8_t bwt_smem[];

// NT = 1024: one CTA per SM (text of up to 184 KB in shared memory); NT = 256: four CTAs per SM for small blocks (a 96x96x1
// uint16 KLB block is 18 KB: six whole 3072-element tiles per pass, and all 484 blocks of a 2048^2 frame resident at once
// instead of four waves of 148 CTAs with half-empty 12288-element tiles)
template <int NT>
__global__ void __launch_bounds__(NT, NT == 1024 ? 1 : 4)
k_bwt(const uint8_t* __restrict__ txt_all, uint32_t cap, EncJob* __restrict__ jobs, uint32_t njobs,
      uint8_t* __restrict__ bwt_all, uint32_t* __restrict__ scratch_all, int text_in_smem)
{
	constexpr int BWT_NT = NT;                       // shadows the namespace constant inside this kernel
	uint32_t* wcnt = reinterpret_cast<uint32_t*>(bwt_smem);
	uint32_t* base = reinterpret_cast<uint32_t*>(bwt_smem + (NT / 32) * BWT_WS * 4);
	uint32_t* run  = base + 256;
	uint32_t* red  = run + 256;          // 64
	uint32_t* misc = red + 64;           // 16
	uint8_t*  stext = reinterpret_cast<uint8_t*>(misc + 16);

	uint32_t* scr = scratch_all + (size_t)blockIdx.x * S_COUNT * cap;
	const uint32_t tid = threadIdx.x;

	for (uint32_t job = blockIdx.x; job < njobs; job += gridDim.x) {
		const uint32_t n = jobs[job].n;
		const uint8_t* gtext = txt_all + (size_t)job * cap;
		uint8_t* bwt = bwt_all + (size_t)job * cap;
		if (n == 0) { if (tid == 0) { jobs[job].orig_ptr = 0; jobs[job].periodic = 0; } continue; }

		// ---- phase 0: text -> shared (with 8 wrap-around bytes), byte histogram -> base[]
		const uint8_t* text;
		if (text_in_smem) {
			for (uint32_t i = tid * 4; i < n; i += BWT_NT * 4) {
				uint32_t wv = *reinterpret_cast<const uint32_t*>(gtext + i);   // cap is a multiple of 16: reading past n stays inside the job's slot
				*reinterpret_cast<uint32_t*>(stext + i) = wv;
			}
			__syncthreads();
			if (tid < 8) stext[n + tid] = stext[tid % n];
			text = stext;
		} else {
			text = gtext;    // the slot keeps 8 wrap bytes after n (written by k_rle1)
		}
		__syncthreads();
		digit_starts<NT>(n, base, wcnt, red, [&](uint32_t e) { return (uint32_t)text[e]; });
		if (tid < 256) {                                  // inUse map = byte values that occur (bzlib.c:226, :243-258)
			const uint32_t c = (tid == 255 ? n : base[tid + 1]) - base[tid];
			const uint32_t bal = __ballot_sync(0xffffffffu, c != 0);
			if ((tid & 31) == 0) jobs[job].in_use[tid >> 5] = bal;
		}

		// ---- phase 1: LSD passes over the rotation prefix (last byte first).  Prefix length: every byte costs a full pass, every
		// byte less leaves more ties to the doubling phase; measured on light-field residuals (uint16, high bytes mostly 0): 6 bytes
		// win on 18 KB blocks (c2 stage 0.61 -> 0.51 ms; 5: 0.66, 4: 0.82), 8 bytes on 147 KB blocks (12.1 ms; 6: 12.6, 4: 30.8)
		int prefix = n <= 49152u ? 6 : 8;
		asm volatile("" : "+r"(prefix));                  // opaque to the optimiser: loops specialised on 6 / 8 spill more in k_bwt<1024>
		uint32_t* src = nullptr; uint32_t* dst = scr + (size_t)S_SA0 * cap;
		for (int p = prefix - 1; p >= 0; p--) {
			if (tid < 256) run[tid] = base[tid];
			__syncthreads();
			const uint32_t* s = src; uint32_t* d = dst;
			radix_scatter<BWT_R, uint32_t, NT>(n, run, wcnt,
				[&](uint32_t e) { return s ? s[e] : e; },
				[&](uint32_t idx) { return (uint32_t)text[idx + p]; },
				[&](uint32_t pos, uint32_t idx) { d[pos] = idx; });
			src = dst;
			dst = (dst == scr + (size_t)S_SA0 * cap) ? scr + (size_t)S_SA1 * cap : scr + (size_t)S_SA0 * cap;
		}
		uint32_t* sa = src;                               // sorted by the prefix
		uint32_t* isa = scr + (size_t)S_ISA * cap;

		// ---- phase 2: group heads, ranks, unresolved set
		uint32_t* G[2] = { scr + (size_t)S_G0 * cap, scr + (size_t)S_G1 * cap };
		uint32_t* Rk[2] = { scr + (size_t)S_R0 * cap, scr + (size_t)S_R1 * cap };
		uint32_t* V[2] = { scr + (size_t)S_V0 * cap, scr + (size_t)S_V1 * cap };
		uint32_t* U[2] = { scr + (size_t)S_U0 * cap, scr + (size_t)S_U1 * cap };
		const uint64_t pmask = prefix >= 8 ? ~0ull : ((1ull << (8 * prefix)) - 1ull);
		uint32_t m = split_groups<NT>(n, red,
			[&](uint32_t j) -> uint64_t {                 // the sorted prefix of rotation sa[j]: three aligned words, shifted
				const uint32_t idx = sa[j], sh = (idx & 3u) * 8u;
				const uint32_t* tw = reinterpret_cast<const uint32_t*>(text + (idx & ~3u));
				const uint32_t w0 = tw[0], w1 = tw[1], w2 = tw[2];
				return (((uint64_t)__funnelshift_r(w1, w2, sh) << 32) | __funnelshift_r(w0, w1, sh)) & pmask;
			},
			[&](uint32_t j) { return j; },
			[&](uint32_t j, uint32_t head, bool un, uint32_t slot) {
				uint32_t sfx = sa[j];
				isa[sfx] = head;
				if (un) { G[0][slot] = head; V[0][slot] = sfx; U[0][slot] = j; }
			});

		// ---- phase 3: prefix doubling on the unresolved set
		const int npass = n <= (1u << 8) ? 1 : n <= (1u << 16) ? 2 : 3;
		int cur = 0, ucur = 0;
		uint64_t h = (uint64_t)prefix;
		while (m > 0 && h < n) {
			uint32_t hh = (uint32_t)h;
			for (uint32_t e = tid; e < m; e += BWT_NT) {
				uint32_t i = V[cur][e] + hh; if (i >= n) i -= n;     // hh < n
				Rk[cur][e] = isa[i];
			}
			__syncthreads();
			// LSD: secondary key (rank at distance h) first, then the group head
			for (int key = 0; key < 2; key++) {
				for (int ps = 0; ps < npass; ps++) {
					const uint32_t* kg = G[cur]; const uint32_t* kr = Rk[cur]; const uint32_t* kv = V[cur];
					uint32_t* og = G[cur ^ 1]; uint32_t* orr = Rk[cur ^ 1]; uint32_t* ov = V[cur ^ 1];
					const int sh = ps * 8;
					digit_starts<NT>(m, run, wcnt, red, [&](uint32_t e) { return ((key ? kg[e] : kr[e]) >> sh) & 255u; });
					radix_scatter<4, Trip, NT>(m, run, wcnt,
						[&](uint32_t e) { Trip t; t.g = kg[e]; t.r = kr[e]; t.v = kv[e]; return t; },
						[&](const Trip& t) { return ((key ? t.g : t.r) >> sh) & 255u; },
						[&](uint32_t pos, const Trip& t) { og[pos] = t.g; orr[pos] = t.r; ov[pos] = t.v; });
					cur ^= 1;
				}
			}
			// U was not moved by the sort: sorted entry s belongs at suffix-array position U[ucur][s].
			// Re-split the groups, update sa / isa, keep what is still unresolved.
			{
				const uint32_t* kg = G[cur]; const uint32_t* kr = Rk[cur]; const uint32_t* kv = V[cur];
				const uint32_t* up = U[ucur];
				uint32_t* ng = G[cur ^ 1]; uint32_t* nv = V[cur ^ 1]; uint32_t* nu = U[ucur ^ 1];
				const uint32_t mm = m;
				m = split_groups<NT>(mm, red,
					[&](uint32_t s) -> uint64_t { return ((uint64_t)kg[s] << 32) | kr[s]; },
					[&](uint32_t s) { return up[s]; },
					[&](uint32_t s, uint32_t head, bool un, uint32_t slot) {
						uint32_t sfx = kv[s], pos = up[s];
						sa[pos] = sfx;
						isa[sfx] = head;
						if (un) { ng[slot] = head; nv[slot] = sfx; nu[slot] = pos; }
					});
				cur ^= 1; ucur ^= 1;
			}
			__syncthreads();
			h <<= 1;
		}

		// ---- phase 4: last column, origPtr (ties left <=> exactly periodic block: rotation 0 goes last in its group)
		for (uint32_t j = tid * 4; j < n; j += BWT_NT * 4) {       // four rotations per thread: one 16-byte load, one word store
			const uint4 q = *reinterpret_cast<const uint4*>(sa + j);   // slots are 16-byte aligned; entries past n are never used
			const uint32_t sv[4] = { q.x, q.y, q.z, q.w };
			uint32_t wv = 0;
			#pragma unroll
			for (int k = 0; k < 4; k++) if (j + k < n) {
				const uint32_t s = sv[k];
				wv |= (uint32_t)text[s ? s - 1 : n - 1] << (8 * k);
				if (s == 0 && m == 0) jobs[job].orig_ptr = j + k;
			}
			*reinterpret_cast<uint32_t*>(bwt + j) = wv;
		}
		if (m > 0) {
			if (tid == 0) misc[1] = 0;
			__syncthreads();
			uint32_t g0 = isa[0], c = 0;
			for (uint32_t e = tid; e < m; e += BWT_NT) c += (G[cur][e] == g0);
			if (c) atomicAdd(&misc[1], c);
			__syncthreads();
			if (tid == 0) jobs[job].orig_ptr = g0 + misc[1] - 1;
		}
		if (tid == 0) jobs[job].periodic = m > 0;
		__syncthreads();
	}
}

static size_t bwt_smem_bytes_nt(uint32_t cap, int text_in_smem, int nt)
{
	size_t fixed = (size_t)(nt / 32) * BWT_WS * 4 + (256 + 256 + 64 + 16) * 4;
	return fixed + (text_in_smem ? (size_t)cap + 16 : 0);
}
size_t bwt_smem_bytes(uint32_t cap, int text_in_smem) { return bwt_smem_bytes_nt(cap, text_in_smem, BWT_NT); }
size_t bwt_scratch_elems_per_cta(uint32_t cap) { return (size_t)S_COUNT * cap; }
// resident CTAs per SM of the variant launch_bwt picks for this slot size: 4 (256 threads) when four texts fit shared memory
int bwt_ctas_per_sm(uint32_t cap, int text_in_smem)
{
	return (text_in_smem && bwt_smem_bytes_nt(cap, 1, 256) + 1024 <= (size_t)227 * 1024 / 4) ? 4 : 1;
}

void launch_bwt(const uint8_t* txt, uint32_t cap, EncJob* jobs, uint32_t njobs, uint8_t* bwt, uint32_t* scratch,
                int grid, int text_in_smem, cudaStream_t st)
{
	if (bwt_ctas_per_sm(cap, text_in_smem) == 4) {
		const size_t smem = bwt_smem_bytes_nt(cap, text_in_smem, 256);
		cudaFuncSetAttribute(k_bwt<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
		k_bwt<256><<<grid, 256, smem, st>>>(txt, cap, jobs, njobs, bwt, scratch, text_in_smem);
		return;
	}
	const size_t smem = bwt_smem_bytes_nt(cap, text_in_smem, 1024);
	cudaFuncSetAttribute(k_bwt<1024>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
	k_bwt<1024><<<grid, 1024, smem, st>>>(txt, cap, jobs, njobs, bwt, scratch, text_in_smem);
}

}  // namespace lfm
