// lfm_predict.cu -- forward predictor + symbolize, and the inverse (unsymbolize + wavefront un-predict).
//
// Forward replaces _predictorN_{tiles,angle,space} + symbolizeKernel + the per-frame cudaMemcpy loop of
// klb_imageIO::Predictor_{both,angle,space}[_GPU] (src/klb_imageIO.cpp:1227-1746): one fused launch over all frames.
// Inverse replaces unsymbolizeKernel + the single-threaded HOST loops unPredictorN_* (src/lfm_Predictors.cu:1470-2739,
// src/klb_imageIO.cpp:1748-1821) with a GPU wavefront, one CTA per frame, frames in parallel:
//   * schedule A, w = tx+ty+u+v (~ tilesX+tilesY+2T steps): valid whenever the near neighbours L/U/UL are only used
//     inside a tile -- every way/predictor except predictor 2 of the ways "tiles" and "angle";
//   * schedule B, row by row (H steps): predictor 2 of those two ways reads U across the tile border (first tile row
//     of interior tiles), which makes every image column one long chain. Rows then only depend on earlier rows, plus
//     short left-to-right chains inside the first tile column / the first image row, which one thread walks.
#include <algorithm>
#include <cstdlib>
#include <cooperative_groups.h>
#include "lfm_device.cuh"
#include "lfm_predict.cuh"

namespace cg = cooperative_groups;

#include <cuda.h>                                   // CUtensorMap (type and enums only: the encoder is fetched through the runtime)

namespace lfm {

// ---- TMA staging of the forward predictor's tile (cp.async.bulk.tensor: ONE thread issues the copy of the whole tile + halo box,
// out-of-image parts are zero-filled by the copy engine, completion on an mbarrier) -----------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
	asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
	asm volatile("fence.proxy.async.shared::cta;" ::: "memory");              // the init is visible to the async proxy
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
	asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2)
{
	asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
	             :: "r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
	uint32_t done;
	do {
		asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
		             : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
	} while (!done);
}


constexpr int PF_NT = 256;

// Forward predictor, row-marching form.  A CTA owns 256 image columns and walks down a band of rows:
//   * everything that depends on the column (tile index tx, in-tile u, first-tile-column tests) is a per-thread
//     constant, everything that depends on the row (ty, v) is uniform over the CTA -> the rule function's border
//     tests are either hoisted or warp-uniform branches;
//   * the row above is carried in registers (up = previous cur, upleft = previous left), the far neighbours
//     (distance T) are plain coalesced 2-byte loads that hit L1/L2: DRAM sees 2 B/px in and 2 B/px out;
//   * WAY and K are template parameters: the rule function collapses to the few adds of the selected predictor.
template <int WAY, int K>
__global__ void __launch_bounds__(PF_NT)
k_predict_fwd_rows(const uint16_t* __restrict__ img, uint16_t* __restrict__ sym, int W, int H, int T, int video,
                   uint32_t z0, int band)
{
	const int x = blockIdx.x * PF_NT + threadIdx.x;
	if (x >= W) return;
	const int y0 = blockIdx.y * band, y1 = min(H, y0 + band);
	const uint32_t z = z0 + blockIdx.z;
	const uint64_t fpx = (uint64_t)W * H;
	const uint16_t* cur = img + (uint64_t)z * fpx;
	uint16_t* out = sym + (uint64_t)z * fpx;
	const int tx = x / T, u = x - tx * T;
	int ty = y0 / T, v = y0 - ty * T;
	const bool zf = (video & (int)z & 1) != 0;                  // `i_or_v & z`: only odd frames look back (klb_imageIO.cpp:1243)
	int up = 0, upleft = 0;
	if (y0 > 0) {
		up = (int)__ldg(cur + (size_t)(y0 - 1) * W + x);
		if (x > 0) upleft = (int)__ldg(cur + (size_t)(y0 - 1) * W + x - 1);
	}
	const uint16_t* rp = cur + (size_t)y0 * W + x;
	uint16_t* op = out + (size_t)y0 * W + x;
	constexpr int RB = 8;                                        // rows whose DRAM loads are in flight together
	for (int yb = y0; yb < y1; yb += RB) {
		int cc[RB], ll[RB];
		#pragma unroll
		for (int r = 0; r < RB; r++) {
			cc[r] = 0; ll[r] = 0;
			if (yb + r < y1) {
				cc[r] = (int)__ldg(rp + (size_t)r * W);
				if (x > 0) ll[r] = (int)__ldg(rp + (size_t)r * W - 1);
			}
		}
		#pragma unroll
		for (int r = 0; r < RB; r++) {
			if (yb + r < y1) {
				const int y = yb + r, c = cc[r], left = ll[r];
				const uint16_t* rq = rp + (size_t)r * W;
				auto px = [&](int dx, int dy) -> int {
					if (dy == 0 && dx == -1) return left;
					if (dy == -1 && dx == 0) return up;
					if (dy == -1 && dx == -1) return upleft;
					return (int)__ldg(rq + (ptrdiff_t)dy * W + dx);
				};
				int p = predict0(px, T, WAY, K, tx, ty, u, v);
				if (WAY == 0 && zf) {
					const int P = (int)__ldg(rq - fpx);
					p = (x == 0 && y == 0) ? P : ((p + P) >> 1);
				}
				op[(size_t)r * W] = symbolize16(c - p);
				up = c; upleft = left;
				if (++v == T) { v = 0; ty++; }
			}
		}
		rp += (size_t)RB * W; op += (size_t)RB * W;
	}
}

// Forward predictor, shared-memory tile form (the HBM-rate path).  A CTA stages a tile of 256 columns x (band + T + 1)
// rows -- its output columns plus `hw` halo columns on the left (T+1 rounded to whole 16-byte vectors) and T+1 halo rows
// above -- with coalesced 16-byte loads, four rows per thread in flight (many bytes in flight per thread is what
// saturating HBM needs).  Then thread = tile column walks down the tile: every neighbour is a conflict-free 2-byte
// shared-memory load (consecutive lanes, consecutive pixels, compile-time row pitch); results leave as 64-byte warp
// stores.  DRAM sees 2 B/px in (+ the halo, mostly L2 hits) and 2 B/px out.
constexpr int PF_PITCH = PF_NT;                  // shared-memory row pitch in pixels = tile width incl. halo

template <int WAY, int K>
__global__ void __launch_bounds__(PF_NT)
k_predict_fwd(const uint16_t* __restrict__ img, uint16_t* __restrict__ sym, int W, int H, int T, int video,
              uint32_t z0, int band, int hw)
{
	extern __shared__ __align__(128) uint8_t pf_smem[];
	uint16_t* sm = reinterpret_cast<uint16_t*>(pf_smem);
	const int tid = (int)threadIdx.x;
	const int cols = PF_NT - hw;                                 // output columns per CTA
	const int x0 = blockIdx.x * cols, y0 = blockIdx.y * band, y1 = min(H, y0 + band);
	const uint32_t z = z0 + blockIdx.z;
	const uint64_t fpx = (uint64_t)W * H;
	const uint16_t* cur = img + (uint64_t)z * fpx;
	uint16_t* out = sym + (uint64_t)z * fpx;
	const int ys = y0 - (T + 1), xs = x0 - hw;                   // image coordinates of smem element (0, 0); may be negative
	const int yc = max(0, ys);                                   // staged rows [yc, y1): rows above the image stay unwritten
	const int nrows = y1 - yc;
	if (((W & 7) == 0) && ((((uintptr_t)img) & 15) == 0)) {
		// thread (cv, rr): 16-byte column cv (of 32) of rows rr, rr+8, ...
		const int cv = tid & 31, rr = tid >> 5;
		const int xv = xs + cv * 8;
		if (xv >= 0 && xv < W) {
			const uint4* g = reinterpret_cast<const uint4*>(cur + (size_t)yc * W + xv);
			uint16_t* d = sm + (yc - ys) * PF_PITCH + cv * 8;
			const uint32_t gstep = (uint32_t)(W >> 3);
			// asynchronous global -> shared copies (LDGSTS): every row of this thread is in flight at once, no staging registers
			uint32_t dsm = (uint32_t)__cvta_generic_to_shared(d) + (uint32_t)rr * (PF_PITCH * 2);
			const uint4* gp = g + (uint32_t)rr * gstep;
			for (int r = rr; r < nrows; r += 8, dsm += 8 * PF_PITCH * 2, gp += 8 * gstep)
				asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(dsm), "l"(gp) : "memory");
		}
		asm volatile("cp.async.commit_group;" ::: "memory");
		asm volatile("cp.async.wait_group 0;" ::: "memory");
	} else {
		const int xc = max(0, xs), nc = min(W, x0 + cols) - xc;
		for (int i = tid; i < nc * nrows; i += PF_NT) {
			const int r = i / nc, cx = i - r * nc;
			sm[(yc - ys + r) * PF_PITCH + (xc - xs) + cx] = __ldg(cur + (size_t)(yc + r) * W + xc + cx);
		}
	}
	__syncthreads();
	const int x = xs + tid;
	if (tid < hw || x >= W) return;
	const int tx = x / T, u = x - tx * T;
	int ty = y0 / T, v = y0 - ty * T;
	const bool zf = (video & (int)z & 1) != 0;                  // `i_or_v & z`: only odd frames look back (klb_imageIO.cpp:1243)
	const uint16_t* b = sm + (y0 - ys) * PF_PITCH + tid;
	uint16_t* op = out + (size_t)y0 * W + x;
	auto generic_row = [&](int y) {
		auto px = [&](int dx, int dy) -> int { return (int)b[dy * PF_PITCH + dx]; };
		int p = predict0(px, T, WAY, K, tx, ty, u, v);
		if (WAY == 0 && zf) {
			const int P = (int)__ldg(cur + (size_t)y * W + x - fpx);
			p = (x == 0 && y == 0) ? P : ((p + P) >> 1);
		}
		*op = symbolize16((int)b[0] - p);
	};
	// walk the band tile row by tile row: inside a tile row ty is fixed and, after its first image row, v > 0 -- the
	// straight-line interior rule then needs no per-row test at all (tx > 0 only splits the warp over the first tile column)
	int y = y0;
	while (y < y1) {
		const int yend = min(y1, y + (T - v));                    // end of this tile row inside the band
		if (WAY != 2 && v == 0) { generic_row(y); y++; v++; b += PF_PITCH; op += W; }
		if (tx > 0 && ty > 0 && !(WAY == 0 && zf)) {
			#pragma unroll 4
			for (; y < yend; y++, v++, b += PF_PITCH, op += W) {
				auto px = [&](int dx, int dy) -> int { return (int)b[dy * PF_PITCH + dx]; };
				*op = symbolize16((int)b[0] - predict_interior<WAY, K>(px, px, T, u, v));
			}
		} else {
			for (; y < yend; y++, v++, b += PF_PITCH, op += W) generic_row(y);
		}
		v = 0; ty++;
	}
}

// Two pixels per thread (the form used whenever rows are whole 16-byte vectors): same tile, 128 threads, each owning
// the adjacent tile columns 2t and 2t+1.  The pair is read with one 32-bit shared load and written with one 32-bit
// store; in the interior rule the row above (up, up-left) is carried in registers and the left neighbour of the second
// pixel is the first pixel itself, so the near-neighbour ways cost two shared loads per PAIR and the loop overhead is
// halved -- this is what takes the kernel from issue-bound to HBM-bound.
constexpr int PF2_NT = PF_NT / 2;

template <int WAY, int K>
__global__ void __launch_bounds__(PF2_NT)
k_predict_fwd2(const uint16_t* __restrict__ img, uint16_t* __restrict__ sym, int W, int H, int T, int video,
               uint32_t z0, int band, int hw, const __grid_constant__ CUtensorMap tmap, int use_tma)
{
	extern __shared__ __align__(128) uint8_t pf_smem[];
	__shared__ __align__(8) uint64_t tile_bar;
	uint16_t* sm = reinterpret_cast<uint16_t*>(pf_smem);
	const int tid = (int)threadIdx.x;
	const int cols = PF_NT - hw;                                 // output columns per CTA
	const int x0 = blockIdx.x * cols, y0 = blockIdx.y * band, y1 = min(H, y0 + band);
	const uint32_t z = z0 + blockIdx.z;
	const uint64_t fpx = (uint64_t)W * H;
	const uint16_t* cur = img + (uint64_t)z * fpx;
	uint16_t* out = sym + (uint64_t)z * fpx;
	const int ys = y0 - (T + 1), xs = x0 - hw;                   // image coordinates of smem element (0, 0); may be negative
	const int yc = max(0, ys);
	const int nrows = y1 - yc;
	if (use_tma) {
		// the box of PF_PITCH columns x (band + T + 1) rows at image coordinates (xs, ys) of frame blockIdx.z of this launch
		if (tid == 0) mbar_init(&tile_bar, 1);
		__syncthreads();
		if (tid == 0) {
			mbar_expect_tx(&tile_bar, (uint32_t)((band + T + 1) * PF_PITCH * 2));
			tma_load_3d(sm, &tmap, &tile_bar, xs, ys, (int)blockIdx.z);
		}
		mbar_wait(&tile_bar, 0);
	} else {
		const int cv = tid & 31, rr = tid >> 5;                    // 16-byte column cv (of 32) of rows rr, rr+4, ...
		const int xv = xs + cv * 8;
		if (xv >= 0 && xv < W) {
			const uint32_t gstep = (uint32_t)(W >> 3);
			const uint4* gp = reinterpret_cast<const uint4*>(cur + (size_t)yc * W + xv) + (uint32_t)rr * gstep;
			uint32_t dsm = (uint32_t)__cvta_generic_to_shared(sm + (yc - ys) * PF_PITCH + cv * 8) + (uint32_t)rr * (PF_PITCH * 2);
			for (int r = rr; r < nrows; r += 4, dsm += 4 * PF_PITCH * 2, gp += 4 * gstep)
				asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(dsm), "l"(gp) : "memory");
		}
		asm volatile("cp.async.commit_group;" ::: "memory");
		asm volatile("cp.async.wait_group 0;" ::: "memory");
	}
	__syncthreads();
	const int sc = 2 * tid;                                      // my first tile column
	const int x = xs + sc;
	if (sc < hw || x >= W) return;                               // hw and W are even: a pair is inside or outside as a whole
	const int txa = x / T, ua = x - txa * T;
	const int txb = (ua + 1 == T) ? txa + 1 : txa, ub = (ua + 1 == T) ? 0 : ua + 1;
	int ty = y0 / T, v = y0 - ty * T;
	const bool zf = (video & (int)z & 1) != 0;
	const uint16_t* b = sm + (y0 - ys) * PF_PITCH + sc;
	uint16_t* op = out + (size_t)y0 * W + x;
	auto generic_row = [&](int y) {
		auto pxa = [&](int dx, int dy) -> int { return (int)b[dy * PF_PITCH + dx]; };
		auto pxb = [&](int dx, int dy) -> int { return (int)b[1 + dy * PF_PITCH + dx]; };
		int pa = predict0(pxa, T, WAY, K, txa, ty, ua, v), pb = predict0(pxb, T, WAY, K, txb, ty, ub, v);
		if (WAY == 0 && zf) {
			const uint32_t P2 = __ldg(reinterpret_cast<const uint32_t*>(cur + (size_t)y * W + x - fpx));
			const int Pa = (int)(P2 & 0xffffu), Pb = (int)(P2 >> 16);
			pa = (x == 0 && y == 0) ? Pa : ((pa + Pa) >> 1);
			pb = (pb + Pb) >> 1;
		}
		const uint32_t c2 = *reinterpret_cast<const uint32_t*>(b);
		*reinterpret_cast<uint32_t*>(op) = (uint32_t)symbolize16((int)(c2 & 0xffffu) - pa) | ((uint32_t)symbolize16((int)(c2 >> 16) - pb) << 16);
	};
	int y = y0;
	while (y < y1) {
		const int yend = min(y1, y + (T - v));                    // end of this tile row inside the band
		if (WAY != 2 && v == 0) {
			if (txa > 0 && ty > 0 && !(WAY == 0 && zf)) {           // first row of an interior tile: straight-line rule
				const uint32_t c2 = *reinterpret_cast<const uint32_t*>(b);
				const int c0 = (int)(c2 & 0xffffu), c1 = (int)(c2 >> 16);
				const int left0 = (int)b[-1];
				auto neara = [&](int dx, int dy) -> int { return dy == 0 ? left0 : (int)b[dy * PF_PITCH + dx]; };
				auto nearb = [&](int dx, int dy) -> int { return dy == 0 ? c0 : (int)b[1 + dy * PF_PITCH + dx]; };
				auto fara = [&](int dx, int dy) -> int { return (int)b[dy * PF_PITCH + dx]; };
				auto farb = [&](int dx, int dy) -> int { return (int)b[1 + dy * PF_PITCH + dx]; };
				const int pa = predict_interior_v0<WAY, K>(neara, fara, T, ua);
				const int pb = predict_interior_v0<WAY, K>(nearb, farb, T, ub);
				*reinterpret_cast<uint32_t*>(op) = (uint32_t)symbolize16(c0 - pa) | ((uint32_t)symbolize16(c1 - pb) << 16);
			} else generic_row(y);
			y++; v++; b += PF_PITCH; op += W;
		}
		if (txa > 0 && ty > 0 && !(WAY == 0 && zf)) {
			if (y < yend) {
				// the row above, carried in registers from here on
				const uint32_t u2 = *reinterpret_cast<const uint32_t*>(b - PF_PITCH);
				int up0 = (int)(u2 & 0xffffu), up1 = (int)(u2 >> 16), ul0 = (int)b[-PF_PITCH - 1];
				#pragma unroll 4
				for (; y < yend; y++, v++, b += PF_PITCH, op += W) {
					const uint32_t c2 = *reinterpret_cast<const uint32_t*>(b);
					const int c0 = (int)(c2 & 0xffffu), c1 = (int)(c2 >> 16);
					const int left0 = (int)b[-1];
					auto neara = [&](int dx, int dy) -> int { return dy == 0 ? left0 : (dx == 0 ? up0 : ul0); };
					auto nearb = [&](int dx, int dy) -> int { return dy == 0 ? c0 : (dx == 0 ? up1 : up0); };
					auto fara = [&](int dx, int dy) -> int { return (int)b[dy * PF_PITCH + dx]; };
					auto farb = [&](int dx, int dy) -> int { return (int)b[1 + dy * PF_PITCH + dx]; };
					const int pa = predict_interior<WAY, K>(neara, fara, T, ua, v);
					const int pb = predict_interior<WAY, K>(nearb, farb, T, ub, v);
					*reinterpret_cast<uint32_t*>(op) = (uint32_t)symbolize16(c0 - pa) | ((uint32_t)symbolize16(c1 - pb) << 16);
					ul0 = left0; up0 = c0; up1 = c1;
				}
			}
		} else {
			for (; y < yend; y++, v++, b += PF_PITCH, op += W) generic_row(y);
		}
		v = 0; ty++;
	}
}

// ---------------------------------------------------------------------------------------------------------
// Inverse predictor: one thread-block CLUSTER per frame (up to 8 CTAs, hardware cluster barrier between wavefront
// steps -- an order of magnitude cheaper than a grid-wide barrier), frames in parallel across clusters.
// Neighbours written by the other CTAs of the cluster are read with ld.global.cg (L2), never through the
// non-coherent L1; barrier.cluster arrive.release / wait.acquire orders the global writes.
constexpr int UP_NT = 512;

__global__ void __launch_bounds__(UP_NT, 2)
k_unpredict(const uint16_t* __restrict__ sym, uint16_t* out, int W, int H, int T, int way, int k, int video,
            uint32_t z_start, uint32_t z_step, uint32_t nframes, int rows_b)
{
	cg::cluster_group cluster = cg::this_cluster();
	__shared__ uint32_t pre[512];
	__shared__ uint32_t red[64];
	const uint32_t tid = threadIdx.x;
	const uint32_t csz = cluster.num_blocks();
	const uint32_t frame = blockIdx.x / csz;
	const uint32_t gtid = cluster.block_rank() * UP_NT + tid, gsize = csz * UP_NT;
	if (frame >= nframes) return;                            // whole clusters only: grid = nframes * csz
	const uint64_t fpx = (uint64_t)W * H;
	const int tilesX = (W + T - 1) / T, tilesY = (H + T - 1) / T;
	const int nr = 2 * T - 1;                                // pixel anti-diagonals inside a tile (<= 509)
	const int nsteps = tilesX + tilesY - 1 + nr - 1;
	const uint32_t z = z_start + frame * z_step;
	const uint16_t* s = sym + (uint64_t)z * fpx;
	uint16_t* o = out + (uint64_t)z * fpx;
	const bool zflag = (video & (int)z & 1) != 0;

	auto decode_px = [&](int x, int y, int tx, int ty, int u, int v) {
		auto px = [&](int dx, int dy) { return (int)__ldcg(o + (size_t)(y + dy) * W + (x + dx)); };
		int p = predict0(px, T, way, k, tx, ty, u, v);
		if (zflag) {
			int P = (int)__ldcg(o + (size_t)y * W + x - fpx);    // previous (even) frame, reconstructed by an earlier launch
			p = (x == 0 && y == 0) ? P : ((p + P) >> 1);
		}
		o[(size_t)y * W + x] = (uint16_t)(unsymbolize16(__ldg(s + (size_t)y * W + x)) + p);
	};

	if (k == 2 && way != 2) {
		// ---- schedule B: rows. Leading pixels with left-neighbour chains are walked by one thread.
		for (int y = 0; y < min(H, rows_b); y++) {               // rows_b < H: the column kernel below takes the rest
			const int ty = y / T, v = y - ty * T;
			const int seq = (y == 0) ? W : min(T, W);
			if (gtid == 0) for (int x = 0; x < seq; x++) decode_px(x, y, x / T, ty, x % T, v);
			for (int x = seq + (int)gtid - 1; x < W; x += (int)gsize - 1) if (gtid > 0) decode_px(x, y, x / T, ty, x % T, v);
			cluster.sync();
		}
		return;
	}

	// ---- schedule A: 4-D wavefront w = tx + ty + u + v
	for (int w = 0; w < nsteps; w++) {
		uint32_t c = 0;
		if ((int)tid < nr) {
			int r = (int)tid, sd = w - r;
			if (sd >= 0 && sd <= tilesX + tilesY - 2) {
				int lo = max(0, sd - (tilesY - 1)), hi = min(sd, tilesX - 1);
				int np = min(r, 2 * T - 2 - r) + 1;
				c = (uint32_t)((hi - lo + 1) * np);
			}
		}
		uint32_t total; uint32_t inc = block_scan_add<UP_NT>(c, red, &total);
		if ((int)tid < nr) pre[tid] = inc - c;
		__syncthreads();
		for (uint32_t i = gtid; i < total; i += gsize) {
			int lo_r = 0, hi_r = nr - 1;                 // last r with pre[r] <= i
			while (lo_r < hi_r) { int mid = (lo_r + hi_r + 1) >> 1; if (pre[mid] <= i) lo_r = mid; else hi_r = mid - 1; }
			const int r = lo_r, sd = w - r;
			const uint32_t j = i - pre[r];
			const int np = min(r, 2 * T - 2 - r) + 1;
			const int ti = (int)(j / (uint32_t)np), pi = (int)(j - (uint32_t)ti * (uint32_t)np);
			const int tx = max(0, sd - (tilesY - 1)) + ti, ty = sd - tx;
			const int u = max(0, r - (T - 1)) + pi, v = r - u;
			const int x = tx * T + u, y = ty * T + v;
			if (x < W && y < H) decode_px(x, y, tx, ty, u, v);
		}
		cluster.sync();
	}
}

// ---------------------------------------------------------------------------------------------------------
// Barrier-free inverse for the two ways whose dependency graph factorises (no cross-CTA synchronisation at all):
//   way "space": after the first tile, pixel (tx,ty,u,v) only depends on the SAME (u,v) of tiles (tx-1,ty), (tx,ty-1),
//     (tx-1,ty-1): T*T independent 2-D recurrences over the tile grid -> one warp per (frame, u, v) walks the tile
//     anti-diagonals with __syncwarp() only.
//   way "angle" (predictor != 2): only the tile DC looks at other tiles (their DCs) -> one warp per frame solves
//     the DC recurrence over tile anti-diagonals, then every tile is an independent intra-tile DPCM: one warp per tile.
// k_unpredict_first_tile decodes tile (0,0) (plain intra-tile DPCM in every way) / the DC grid.
constexpr int UF_NT = 128;

// mode 0: tile (0,0) of every frame (way space);  mode 1: the DC pixel of every tile (way angle).  One warp per frame.
__global__ void __launch_bounds__(UF_NT)
k_unpredict_seed(const uint16_t* __restrict__ sym, uint16_t* out, int W, int H, int T, int way, int k,
                 uint32_t z_start, uint32_t z_step, uint32_t nframes, int mode)
{
	const uint32_t lane = lane_id();
	const uint32_t f = blockIdx.x * (UF_NT / 32) + warp_id();
	if (f >= nframes) return;
	const uint64_t fpx = (uint64_t)W * H;
	const uint32_t z = z_start + f * z_step;
	const uint16_t* s = sym + (uint64_t)z * fpx;
	uint16_t* o = out + (uint64_t)z * fpx;
	auto decode_px = [&](int x, int y, int tx, int ty, int u, int v) {
		auto px = [&](int dx, int dy) { return (int)__ldcg(o + (size_t)(y + dy) * W + (x + dx)); };
		o[(size_t)y * W + x] = (uint16_t)(unsymbolize16(__ldg(s + (size_t)y * W + x)) + predict0(px, T, way, k, tx, ty, u, v));
	};
	if (mode == 0 && T <= 32) {
		// the tile stays in shared memory while its anti-diagonals are decoded (a step through global memory is an L2 round trip:
		// 29 steps = 22 us for a 15 x 15 tile, more than the two scan passes of a whole 2048^2 frame); the rule of tile (0,0) only
		// looks at its own left / upper pixels, a zero frame stands in for what lies outside the image
		__shared__ uint16_t tile_s[UF_NT / 32][34 * 34];
		uint16_t* tl = tile_s[warp_id()];
		const int tw = min(T, W), th = min(T, H);
		for (int i = (int)lane; i < 34 * 34; i += 32) tl[i] = 0;
		__syncwarp();
		for (int d = 0; d <= tw + th - 2; d++) {             // pixel anti-diagonals of the first tile
			for (int u = (int)lane; u <= d; u += 32) {
				const int v = d - u;
				if (u < tw && v < th) {
					auto px = [&](int dx, int dy) { return (int)tl[(v + dy + 1) * 34 + (u + dx + 1)]; };
					tl[(v + 1) * 34 + u + 1] = (uint16_t)(unsymbolize16(__ldg(s + (size_t)v * W + u)) + predict0(px, T, way, k, 0, 0, u, v));
				}
			}
			__syncwarp();
		}
		for (int i = (int)lane; i < tw * th; i += 32) { const int v = i / tw, u = i - v * tw; o[(size_t)v * W + u] = tl[(v + 1) * 34 + u + 1]; }
	} else if (mode == 0) {
		const int tw = min(T, W), th = min(T, H);
		for (int d = 0; d <= tw + th - 2; d++) {             // pixel anti-diagonals of the first tile
			for (int u = (int)lane; u <= d; u += 32) { int v = d - u; if (u < tw && v < th) decode_px(u, v, 0, 0, u, v); }
			__syncwarp();
		}
	} else {
		const int tilesX = (W + T - 1) / T, tilesY = (H + T - 1) / T;
		for (int d = 0; d <= tilesX + tilesY - 2; d++) {     // tile anti-diagonals, DC pixel only
			const int lo = max(0, d - (tilesY - 1)), hi = min(d, tilesX - 1);
			for (int tx = lo + (int)lane; tx <= hi; tx += 32) { int ty = d - tx; decode_px(tx * T, ty * T, tx, ty, 0, 0); }
			__syncwarp();
		}
	}
}

// way space: one warp per (frame, u, v)
__global__ void __launch_bounds__(UF_NT)
k_unpredict_space(const uint16_t* __restrict__ sym, uint16_t* out, int W, int H, int T, int k,
                  uint32_t z_start, uint32_t z_step, uint32_t nframes)
{
	const uint32_t lane = lane_id();
	const uint32_t wg = blockIdx.x * (UF_NT / 32) + warp_id();
	const uint32_t per_frame = (uint32_t)T * T;
	const uint32_t f = wg / per_frame;
	if (f >= nframes) return;
	const uint32_t uv = wg - f * per_frame;
	const int v = (int)(uv / (uint32_t)T), u = (int)(uv - (uint32_t)v * T);
	const uint64_t fpx = (uint64_t)W * H;
	const uint32_t z = z_start + f * z_step;
	const uint16_t* s = sym + (uint64_t)z * fpx;
	uint16_t* o = out + (uint64_t)z * fpx;
	const int tilesX = (W + T - 1) / T, tilesY = (H + T - 1) / T;
	for (int d = 1; d <= tilesX + tilesY - 2; d++) {         // tile (0,0) was decoded by k_unpredict_seed
		const int lo = max(0, d - (tilesY - 1)), hi = min(d, tilesX - 1);
		for (int tx = lo + (int)lane; tx <= hi; tx += 32) {
			const int ty = d - tx, x = tx * T + u, y = ty * T + v;
			if (x < W && y < H) {
				auto px = [&](int dx, int dy) { return (int)__ldcg(o + (size_t)(y + dy) * W + (x + dx)); };
				o[(size_t)y * W + x] = (uint16_t)(unsymbolize16(__ldg(s + (size_t)y * W + x)) + predict0(px, T, 2, k, tx, ty, u, v));
			}
		}
		__syncwarp();
	}
}

// way angle (predictor != 2): one warp per (frame, tile); the DC is already in place
__global__ void __launch_bounds__(UF_NT)
k_unpredict_angle(const uint16_t* __restrict__ sym, uint16_t* out, int W, int H, int T, int k,
                  uint32_t z_start, uint32_t z_step, uint32_t nframes)
{
	const uint32_t lane = lane_id();
	const int tilesX = (W + T - 1) / T, tilesY = (H + T - 1) / T;
	const uint64_t wg = (uint64_t)blockIdx.x * (UF_NT / 32) + warp_id();
	const uint64_t per_frame = (uint64_t)tilesX * tilesY;
	const uint32_t f = (uint32_t)(wg / per_frame);
	if (f >= nframes) return;
	const uint32_t tile = (uint32_t)(wg - (uint64_t)f * per_frame);
	const int ty = (int)(tile / (uint32_t)tilesX), tx = (int)(tile - (uint32_t)ty * tilesX);
	const uint64_t fpx = (uint64_t)W * H;
	const uint32_t z = z_start + f * z_step;
	const uint16_t* s = sym + (uint64_t)z * fpx;
	uint16_t* o = out + (uint64_t)z * fpx;
	const int x0 = tx * T, y0 = ty * T, tw = min(T, W - x0), th = min(T, H - y0);
	for (int d = 1; d <= tw + th - 2; d++) {
		for (int u = (int)lane; u <= d; u += 32) {
			const int v = d - u;
			if (u < tw && v < th) {
				const int x = x0 + u, y = y0 + v;
				auto px = [&](int dx, int dy) { return (int)__ldcg(o + (size_t)(y + dy) * W + (x + dx)); };
				o[(size_t)y * W + x] = (uint16_t)(unsymbolize16(__ldg(s + (size_t)y * W + x)) + predict0(px, T, 1, k, tx, ty, u, v));
			}
		}
		__syncwarp();
	}
}

// ---------------------------------------------------------------------------------------------------------
// Shared-memory inverse for the two ways whose dependency graph factorises.
//
// k_unpredict_grid: a 2-D recurrence over the TILE grid -- out(tx,ty) = res + f(out(tx-1,ty), out(tx,ty-1), out(tx-1,ty-1)).
//   way "space": one CTA per (frame, u, v): the sub-aperture image (pixel (u,v) of every microlens);
//   way "angle": one CTA per frame, (u,v) = (0,0): the grid of tile DC pixels.
//   The residuals of the sub-image are gathered into shared memory first (all loads in flight together), then
//   thread tx walks down column tx of the grid along the anti-diagonal wavefront d = tx + ty: `up` is the thread's own
//   previous output, `upleft` the value it read from its left neighbour one step earlier, `left` comes through a
//   double-buffered shared line -- one CTA barrier per wavefront step, no global-memory round trip on the chain.
// k_unpredict_tiles_angle: way "angle", predictor != 2: with the DCs in place every tile is an independent DPCM.
//   A CTA stages one tile row (T image rows x 128 tiles) in shared memory with coalesced loads, ONE THREAD decodes ONE
//   tile in place (raster order; its left / up / up-left neighbours are shared-memory reads of its own earlier
//   writes -- no synchronisation at all), then the strip is written back coalesced.
constexpr int UG_MAX_SMEM = 200 * 1024;

// One CTA decodes G sub-images that are neighbours in u (same v): a gathered 32-byte sector then carries G useful
// pixels instead of one, and the decoded pixels -- staged in shared memory, in place of the residuals -- leave as
// G-pixel runs: the sub-aperture gather / scatter is L2-sector bound.
template <int WAY, int K>
__global__ void __launch_bounds__(1024)
k_unpredict_grid(const uint16_t* __restrict__ sym, uint16_t* out, int W, int H, int T,
                 uint32_t z_start, uint32_t z_step, int G, int ugroups, int vcount, int nxr)
{
	extern __shared__ __align__(16) uint8_t ug_smem[];
	const uint32_t tid = threadIdx.x;
	uint32_t bq = blockIdx.x;
	const int ug = (int)(bq % (uint32_t)ugroups); bq /= (uint32_t)ugroups;
	const int v = (int)(bq % (uint32_t)vcount);                                              // (0,0) only for the DC grid
	const uint32_t f = bq / (uint32_t)vcount;
	const int u0 = ug * G;
	const int gcount = min(G, (WAY == 2 ? T : 1) - u0);                                      // sub-images of this CTA
	const int nx0 = (W - u0 + T - 1) / T, ny = (H - v + T - 1) / T;                          // grid points (widest sub-image)
	if (nx0 <= 0 || ny <= 0 || gcount <= 0) return;
	const uint64_t fpx = (uint64_t)W * H;
	const uint32_t z = z_start + f * z_step;
	const uint16_t* s = sym + (uint64_t)z * fpx + (size_t)v * W + u0;
	uint16_t* o = out + (uint64_t)z * fpx + (size_t)v * W + u0;
	const uint32_t plane = ((uint32_t)nx0 * (uint32_t)ny + 7u) & ~7u;
	int16_t* res = reinterpret_cast<int16_t*>(ug_smem);                                      // [G][ny][nx0] residuals, then pixels
	uint16_t* line = reinterpret_cast<uint16_t*>(ug_smem) + (size_t)G * plane;               // [G][2][nx0 + 1]
	const size_t rowstep = (size_t)T * W;

	// ---- gather (unsymbolize on the way in).  Work item = (grid row gy, element e of the row), e = gx * gcount + g:
	// neighbouring threads read neighbouring pixels of one tile, then the next tile
	const uint32_t rowlen = (uint32_t)nx0 * (uint32_t)gcount;
	const uint32_t rpp = max(1u, blockDim.x / rowlen);                                      // grid rows per pass
	const uint32_t er = tid / rowlen, ee = tid - er * rowlen;                               // my row slot, my element
	const uint32_t egx = ee / (uint32_t)gcount, eg = ee - egx * (uint32_t)gcount;
	const bool eok = er < rpp && egx * T + u0 + eg < (uint32_t)W;
	const size_t eoff = (size_t)egx * T + eg;
	int16_t* eres = res + eg * plane + egx;
	if (rowlen <= blockDim.x) {
		for (uint32_t gy0 = 0; gy0 < (uint32_t)ny; gy0 += rpp * 8) {
			uint16_t q[8];
			#pragma unroll
			for (int r = 0; r < 8; r++) { const uint32_t gy = gy0 + r * rpp + er; q[r] = 0; if (eok && gy < (uint32_t)ny) q[r] = __ldg(s + gy * rowstep + eoff); }
			#pragma unroll
			for (int r = 0; r < 8; r++) { const uint32_t gy = gy0 + r * rpp + er; if (er < rpp && gy < (uint32_t)ny) eres[gy * nx0] = (int16_t)unsymbolize16(q[r]); }
		}
	} else {
		for (uint32_t gy = 0; gy < (uint32_t)ny; gy++)
			for (uint32_t e = tid; e < rowlen; e += blockDim.x) {
				const uint32_t gx = e / (uint32_t)gcount, g = e - gx * (uint32_t)gcount;
				uint16_t qv = 0;
				if (gx * T + u0 + g < (uint32_t)W) qv = __ldg(s + gy * rowstep + (size_t)gx * T + g);
				res[g * plane + gy * nx0 + gx] = (int16_t)unsymbolize16(qv);
			}
	}
	// thread (g, tx)
	const int g = (int)(tid / (uint32_t)nxr), tx = (int)(tid - (uint32_t)g * (uint32_t)nxr);
	const int u = u0 + g;
	const int nx = (g < gcount) ? (W - u + T - 1) / T : 0;                                   // this sub-image's width
	// way space: tile (0,0) is an ordinary intra-tile DPCM decoded beforehand (k_unpredict_seed); DC grid: predictor 0
	int first = 0;
	if (tx == 0 && nx > 0 && WAY == 2) first = (int)__ldcg(o + g);
	__syncthreads();

	// ---- wavefront
	int16_t* myres = res + (size_t)g * plane;
	uint16_t* myline = line + (size_t)g * 2 * (nx0 + 1);
	int up = 0, upleft = 0;
	const int nsteps = nx0 + ny - 1;
	for (int d = 0; d < nsteps; d++) {
		const int ty = d - tx;
		const uint16_t* rd = myline + ((d + 1) & 1) * (nx0 + 1);        // written at step d-1
		uint16_t* wr = myline + (d & 1) * (nx0 + 1);
		if (tx < nx && ty >= 0 && ty < ny) {
			const int left = tx > 0 ? (int)rd[tx - 1] : 0;
			int16_t* cell = myres + (size_t)ty * nx0 + tx;
			int val;
			if (d == 0) val = (WAY == 2) ? first : (int)(uint16_t)*cell;
			else {
				auto px = [&](int dx, int dy) -> int { return dx == 0 ? up : (dy == 0 ? left : upleft); };
				const int p = predict0(px, T, WAY, K, tx, ty, u, v);
				val = (int)(uint16_t)((int)*cell + p);
			}
			wr[tx] = (uint16_t)val;
			*cell = (int16_t)val;
			upleft = left; up = val;
		}
		__syncthreads();
	}

	// ---- scatter the decoded sub-images, same traversal as the gather
	if (rowlen <= blockDim.x) {
		for (uint32_t gy = er; gy < (uint32_t)ny; gy += rpp)
			if (eok) o[gy * rowstep + eoff] = (uint16_t)eres[gy * nx0];
	} else {
		for (uint32_t gy = 0; gy < (uint32_t)ny; gy++)
			for (uint32_t e = tid; e < rowlen; e += blockDim.x) {
				const uint32_t gx = e / (uint32_t)gcount, g2 = e - gx * (uint32_t)gcount;
				if (gx * T + u0 + g2 < (uint32_t)W) o[gy * rowstep + (size_t)gx * T + g2] = (uint16_t)res[g2 * plane + gy * nx0 + gx];
			}
	}
}

template <int WAY>
static void launch_unpredict_grid(const uint16_t* sym, uint16_t* out, int W, int H, int T, int k, uint32_t z_start, uint32_t z_step,
                                  unsigned grid, unsigned block, size_t smem, int G, int ugroups, int vcount, int nxr, cudaStream_t st)
{
	#define LFM_UG(KK) do { cudaFuncSetAttribute(k_unpredict_grid<WAY, KK>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
		k_unpredict_grid<WAY, KK><<<grid, block, smem, st>>>(sym, out, W, H, T, z_start, z_step, G, ugroups, vcount, nxr); } while (0)
	switch (k) {
	case 1: LFM_UG(1); break; case 2: LFM_UG(2); break; case 3: LFM_UG(3); break; case 4: LFM_UG(4); break;
	case 5: LFM_UG(5); break; case 6: LFM_UG(6); break; default: LFM_UG(7); break;
	}
	#undef LFM_UG
}

constexpr int UT_NT = 128;       // tiles (= threads) per CTA

template <int K>
__global__ void __launch_bounds__(UT_NT)
k_unpredict_tiles_angle(const uint16_t* __restrict__ sym, uint16_t* out, int W, int H, int T,
                        uint32_t z_start, uint32_t z_step, int tilesX, int tilesY, int chunks)
{
	extern __shared__ __align__(16) uint8_t ut_smem[];
	uint16_t* sm = reinterpret_cast<uint16_t*>(ut_smem);
	const uint32_t tid = threadIdx.x;
	uint32_t b = blockIdx.x;
	const int chunk = (int)(b % (uint32_t)chunks); b /= (uint32_t)chunks;
	const int ty = (int)(b % (uint32_t)tilesY);
	const uint32_t f = b / (uint32_t)tilesY;
	const uint64_t fpx = (uint64_t)W * H;
	const uint32_t z = z_start + f * z_step;
	const int x0 = chunk * UT_NT * T, y0 = ty * T;
	const int sw = min(W - x0, UT_NT * T), th = min(T, H - y0);           // strip width / height in pixels
	const uint16_t* s = sym + (uint64_t)z * fpx + (size_t)y0 * W + x0;
	uint16_t* o = out + (uint64_t)z * fpx + (size_t)y0 * W + x0;
	const bool vec = ((W & 7) == 0) && ((sw & 7) == 0) && ((((uintptr_t)sym | (uintptr_t)out) & 15) == 0);   // x0 is a multiple of 128
	const int pitch = sw;

	// ---- stage the strip (residual symbols)
	if (vec) {
		const int wv = sw >> 3;                                   // asynchronous 16-byte copies: the whole strip in flight at once
		for (int r = 0; r < th; r++) {
			const uint4* gp = reinterpret_cast<const uint4*>(s + (size_t)r * W);
			const uint32_t dsm = (uint32_t)__cvta_generic_to_shared(sm + (size_t)r * pitch);
			for (int cx = (int)tid; cx < wv; cx += UT_NT)
				asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(dsm + (uint32_t)cx * 16u), "l"(gp + cx) : "memory");
		}
		asm volatile("cp.async.commit_group;" ::: "memory");
		asm volatile("cp.async.wait_group 0;" ::: "memory");
	} else {
		for (int i = (int)tid; i < sw * th; i += UT_NT) { const int r = i / sw, cx = i - r * sw; sm[(size_t)r * pitch + cx] = __ldg(s + (size_t)r * W + cx); }
	}
	__syncthreads();

	// ---- one thread, one tile
	const int tx = chunk * UT_NT + (int)tid;
	if (tx < tilesX) {
		const int tw = min(T, W - tx * T);
		uint16_t* t0 = sm + (size_t)tid * T;
		t0[0] = __ldcg(o + (size_t)tid * T);                              // the DC, decoded by k_unpredict_grid
		for (int v = 0; v < th; v++) {
			uint16_t* row = t0 + (size_t)v * pitch;
			if (v > 0 && tx > 0 && ty > 0) {
				// interior tile, v > 0: straight-line rule; left / up-left ride in registers, so the only value on the
				// pixel-to-pixel dependency chain is the previous result (the row above is an independent shared load)
				const uint16_t* above = row - pitch;
				int up = (int)above[0];
				int left = (int)(uint16_t)(unsymbolize16(row[0]) + up);           // u == 0: predicted from the pixel above
				row[0] = (uint16_t)left;
				int ul = up;
				for (int u = 1; u < tw; u++) {
					up = (int)above[u];
					auto near = [&](int dx, int dy) -> int { return dy == 0 ? left : (dx == 0 ? up : ul); };
					const int p = predict_interior<1, K>(near, near, T, u, v);
					left = (int)(uint16_t)(unsymbolize16(row[u]) + p);
					row[u] = (uint16_t)left;
					ul = up;
				}
			} else {
				for (int u = (v == 0) ? 1 : 0; u < tw; u++) {
					auto px = [&](int dx, int dy) -> int { return (int)row[u + dx + dy * pitch]; };
					const int p = predict0(px, T, 1, K, tx, ty, u, v);
					row[u] = (uint16_t)(unsymbolize16(row[u]) + p);
				}
			}
		}
	}
	__syncthreads();

	// ---- write the decoded strip back
	if (vec) {
		const int wv = sw >> 3;
		for (int i = (int)tid; i < wv * th; i += UT_NT) {
			const int r = i / wv, cx = i - r * wv;
			reinterpret_cast<uint4*>(o + (size_t)r * W)[cx] = reinterpret_cast<const uint4*>(sm + (size_t)r * pitch)[cx];
		}
	} else {
		for (int i = (int)tid; i < sw * th; i += UT_NT) { const int r = i / sw, cx = i - r * sw; o[(size_t)r * W + cx] = sm[(size_t)r * pitch + cx]; }
	}
}

template <int K>
static void launch_tiles_angle(const uint16_t* sym, uint16_t* out, int W, int H, int T, uint32_t z_start, uint32_t z_step,
                               uint32_t count, int tilesX, int tilesY, int chunks, size_t smem, cudaStream_t st)
{
	cudaFuncSetAttribute(k_unpredict_tiles_angle<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
	k_unpredict_tiles_angle<K><<<(unsigned)((uint64_t)count * tilesY * chunks), UT_NT, smem, st>>>(sym, out, W, H, T, z_start, z_step, tilesX, tilesY, chunks);
}

// ---------------------------------------------------------------------------------------------------------
// Universal shared-memory inverse (any way, predictor, video): one CTA per FRAME walks the frame block by block --
// a block = one tile row x up to 64 tiles -- in raster order.  Everything a block needs from earlier blocks (T+1 decoded
// rows above, T+1 decoded columns to the left, the previous frame for odd video frames) is re-read from the output in
// global memory (written by this CTA, or by the previous launch), so only the block and its halo live in shared memory.
// Inside a block the pixels are decoded along the wavefront  w = (tile index) + u + v  -- every operand of the rule
// function lies in an earlier block or has a smaller w -- with one CTA barrier per step.  Thread = (anti-diagonal r of a
// tile, position on it): at step w it decodes tile w - r.  Frames are independent CTAs: this is the throughput path for
// stacks and videos (hundreds of frames); a single frame is better served by the cluster kernel above.
constexpr int US_TILES = 64;             // tiles per block

template <int WAY, int K>
__global__ void __launch_bounds__(1024)
k_unpredict_strips(const uint16_t* __restrict__ sym, uint16_t* out, int W, int H, int T, int video,
                   uint32_t z_start, uint32_t z_step, int hw, int pitch)
{
	extern __shared__ __align__(16) uint8_t us_smem[];
	uint16_t* cur = reinterpret_cast<uint16_t*>(us_smem);                 // [T][pitch]      symbols -> pixels, column hw = block column 0
	uint16_t* prv = cur + (size_t)T * pitch;                               // [T + 1][pitch]  decoded rows y0-T-1 .. y0-1
	uint16_t* pfr = prv + (size_t)(T + 1) * pitch;                         // [T][pitch]      previous frame (odd video frames only)
	const int tid = (int)threadIdx.x, nt = (int)blockDim.x;
	const uint64_t fpx = (uint64_t)W * H;
	const uint32_t z = z_start + blockIdx.x * z_step;
	const uint16_t* s = sym + (uint64_t)z * fpx;
	uint16_t* o = out + (uint64_t)z * fpx;
	const bool zflag = (video & (int)z & 1) != 0;
	const int tilesX = (W + T - 1) / T, tilesY = (H + T - 1) / T;
	const int halo = T + 1;
	const int ncand = (2 * T - 1) * T;                                     // (anti-diagonal, position) pairs of a tile
	const int dr = nt / T, dl = nt - dr * T;                               // stride of the candidate loop in (r, l) form

	for (int ty = 0; ty < tilesY; ty++) {
		const int y0 = ty * T, th = min(T, H - y0);
		for (int tb0 = 0; tb0 < tilesX; tb0 += US_TILES) {
			const int ntb = min(US_TILES, tilesX - tb0);
			const int x0 = tb0 * T, cw = min(W - x0, ntb * T);             // block columns [x0, x0 + cw)
			const int xl = max(0, x0 - halo);                              // first halo column
			// ---- stage: symbols of the block, decoded halo (rows above incl. their left halo, columns to the left), previous frame
			if (((W & 7) == 0) && (((((uintptr_t)sym | (uintptr_t)out)) & 15) == 0)) {
				// rows are whole 16-byte vectors and block / halo starts are multiples of 8 pixels: asynchronous 16-byte copies,
				// everything in flight at once (.cg: served by L2, so this CTA's earlier stores are seen)
				auto copy_rows = [&](uint16_t* dst_row0, const uint16_t* src_row0, int rows, int xa, int xb) {   // columns [xa, xb) of `rows` rows
					const int nv = (xb - xa) >> 3;
					for (int i = tid; i < rows * nv; i += nt) {
						const int r = i / nv, cv = i - r * nv;
						const uint32_t d = (uint32_t)__cvta_generic_to_shared(dst_row0 + (size_t)r * pitch + hw + (xa - x0) + cv * 8);
						asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(d), "l"(src_row0 + (size_t)r * W + xa + cv * 8) : "memory");
					}
				};
				const int xh = max(0, x0 - hw);
				const int ya = max(0, y0 - halo);
				copy_rows(cur, s + (size_t)y0 * W, th, x0, x0 + cw);
				copy_rows(prv + (size_t)(ya - (y0 - halo)) * pitch, o + (size_t)ya * W, y0 - ya, xh, x0 + cw);
				copy_rows(cur, o + (size_t)y0 * W, th, xh, x0);
				if (zflag) copy_rows(pfr, o + (size_t)y0 * W - fpx, th, x0, x0 + cw);
				asm volatile("cp.async.commit_group;" ::: "memory");
				asm volatile("cp.async.wait_group 0;" ::: "memory");
			} else {
				for (int i = tid; i < th * cw; i += nt) { const int r = i / cw, c = i - r * cw; cur[r * pitch + hw + c] = __ldg(s + (size_t)(y0 + r) * W + x0 + c); }
				const int hwid = x0 + cw - xl;                             // halo rows span [xl, x0 + cw)
				const int ya = max(0, y0 - halo);
				for (int i = tid; i < (y0 - ya) * hwid; i += nt) {
					const int r = i / hwid, c = i - r * hwid;
					prv[(ya + r - (y0 - halo)) * pitch + hw + (xl + c - x0)] = __ldcg(o + (size_t)(ya + r) * W + xl + c);
				}
				const int lw = x0 - xl;
				for (int i = tid; i < th * lw; i += nt) { const int r = i / lw, c = i - r * lw; cur[r * pitch + hw + (xl + c - x0)] = __ldcg(o + (size_t)(y0 + r) * W + xl + c); }
				if (zflag) for (int i = tid; i < th * cw; i += nt) { const int r = i / cw, c = i - r * cw; pfr[r * pitch + hw + c] = __ldcg(o + (size_t)(y0 + r) * W + x0 + c - fpx); }
			}
			__syncthreads();
			// ---- wavefront over the block
			const int nsteps = ntb + 2 * T - 2;
			for (int w = 0; w < nsteps; w++) {
				int r = tid / T, l = tid - r * T;
				for (int i = tid; i < ncand; i += nt) {
					const int tb = w - r;
					const int u = max(0, r - (T - 1)) + l, v = r - u;
					if (tb >= 0 && tb < ntb && v >= 0 && u < T) {
						const int tx = tb0 + tb, xb = tb * T + u;          // xb: column inside the block
						if (x0 + xb < W && v < th) {
							uint16_t* c = cur + v * pitch + hw + xb;
							auto px = [&](int dx, int dy) -> int {
								const int yy = v + dy;
								return (int)(yy >= 0 ? c[dy * pitch + dx] : prv[(yy + halo) * pitch + hw + xb + dx]);
							};
							int p = predict0(px, T, WAY, K, tx, ty, u, v);
							if (zflag) { const int P = (int)pfr[v * pitch + hw + xb]; p = (x0 + xb == 0 && y0 + v == 0) ? P : ((p + P) >> 1); }
							*c = (uint16_t)(unsymbolize16(*c) + p);
						}
					}
					r += dr; l += dl; if (l >= T) { l -= T; r++; }
				}
				__syncthreads();
			}
			// ---- write the decoded block
			if (((W & 7) == 0) && ((((uintptr_t)out) & 15) == 0)) {
				const int nv = cw >> 3;
				for (int i = tid; i < th * nv; i += nt) {
					const int r = i / nv, cv = i - r * nv;
					*reinterpret_cast<uint4*>(o + (size_t)(y0 + r) * W + x0 + cv * 8) = *reinterpret_cast<const uint4*>(cur + (size_t)r * pitch + hw + cv * 8);
				}
			} else {
				for (int i = tid; i < th * cw; i += nt) { const int r = i / cw, c = i - r * cw; o[(size_t)(y0 + r) * W + x0 + c] = cur[r * pitch + hw + c]; }
			}
			__syncthreads();
		}
	}
}

template <int WAY>
static int launch_unpredict_strips(const uint16_t* sym, uint16_t* out, int W, int H, int T, int k, int video,
                                   uint32_t z_start, uint32_t z_step, uint32_t count, cudaStream_t st)
{
	const int hw = (T + 1 + 7) & ~7, pitch = hw + ((US_TILES * T + 7) & ~7);
	const size_t smem = (size_t)(3 * T + 1) * pitch * 2;
	if (smem > (size_t)UG_MAX_SMEM) return 2;                   // Nnum too large for this path
	const unsigned nt = (unsigned)std::min(1024, ((2 * T - 1) * T + 31) & ~31);
	#define LFM_US(KK) do { cudaFuncSetAttribute(k_unpredict_strips<WAY, KK>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
		k_unpredict_strips<WAY, KK><<<count, nt, smem, st>>>(sym, out, W, H, T, video, z_start, z_step, hw, pitch); } while (0)
	switch (k) {
	case 1: LFM_US(1); break; case 2: LFM_US(2); break; case 3: LFM_US(3); break; case 4: LFM_US(4); break;
	case 5: LFM_US(5); break; case 6: LFM_US(6); break; default: LFM_US(7); break;
	}
	#undef LFM_US
	return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

// ---------------------------------------------------------------------------------------------------------
// Predictor 2 of the ways "tiles" and "angle": below the first tile row the rules only look UP -- U = (x, y-1) and
// Ut = (x, y-T) -- so every image column is an independent chain of H - T steps (lfm_predict.cuh: way tiles
// (U + Ut) >> 1 / Ut, way angle U / Ut).  One thread per column walks down its column: U in a register, the last T
// decoded pixels of the column in a shared-memory ring (slot y mod T holds Ut when row y is decoded), symbols prefetched
// UC_D rows ahead into registers; loads and stores of a warp are 64 contiguous bytes of an image row.  The one
// horizontal dependency left -- way angle, first tile column, first row of a tile: pred = L -- is a chain of T - 1
// shuffles in the warp that owns columns 0..31.  In the first tile row the rules of rows 1..T-1 look up as well; only image
// ROW 0 is a chain along x (pred = L, or Lt for the first pixel of a tile): k_unpredict_row0 walks it, one warp per frame,
// with the symbols staged in shared memory.
// Replaces the row-by-row schedule (one cluster barrier per image row: 14.7 ms for a 2048^2 x 32 stack).
// image row 0 of every frame (predictor 2, ways tiles / angle): t00 pred = L (0 for the first pixel), later tiles Lt for
// u == 0 and L for u > 0.  One warp per frame: symbols (and the previous frame's row, video) staged in shared memory,
// lane 0 walks the W pixels with L in a register, the warp writes the row back.
template <int WAY>
__global__ void __launch_bounds__(32)
k_unpredict_row0(const uint16_t* __restrict__ sym, uint16_t* out, int W, int H, int T, int video, uint32_t z_start, uint32_t z_step)
{
	extern __shared__ __align__(16) uint8_t r0_smem[];
	uint16_t* srow = reinterpret_cast<uint16_t*>(r0_smem);        // symbols -> pixels, in place
	uint16_t* prow = srow + W;                                     // previous frame (odd video frames)
	const int lane = (int)threadIdx.x;
	const uint32_t z = z_start + blockIdx.x * z_step;
	const uint64_t fpx = (uint64_t)W * H;
	const bool zflag = (video & (int)z & 1) != 0;
	const uint16_t* s = sym + (uint64_t)z * fpx;
	uint16_t* o = out + (uint64_t)z * fpx;
	for (int x = lane; x < W; x += 32) { srow[x] = __ldg(s + x); if (zflag) prow[x] = __ldcg(o + x - fpx); }
	__syncwarp();
	if (lane == 0) {
		int left = 0, tx = 0, u = 0;
		for (int x = 0; x < W; x++) {
			// predict0 for k = 2, ty == 0, v == 0 written out (both ways): L inside a tile, Lt (already decoded, in place) for the
			// first pixel of a tile, 0 for the first pixel of the row
			int p = u ? left : (tx ? (int)srow[x - T] : 0);
			if (WAY == 0 && zflag) p = x == 0 ? (int)prow[0] : ((p + (int)prow[x]) >> 1);
			left = (unsymbolize16(srow[x]) + p) & 0xffff;
			srow[x] = (uint16_t)left;
			if (++u == T) { u = 0; tx++; }
		}
	}
	__syncwarp();
	for (int x = lane; x < W; x += 32) o[x] = srow[x];
}

constexpr int UC_NT = 128;
constexpr int UC_D = 8;

template <int WAY>
__global__ void __launch_bounds__(UC_NT)
k_unpredict_cols2(const uint16_t* __restrict__ sym, uint16_t* out, int W, int H, int T, int video,
                  uint32_t z_start, uint32_t z_step)
{
	extern __shared__ __align__(16) uint8_t uc_smem[];
	uint16_t* ring = reinterpret_cast<uint16_t*>(uc_smem);          // [T][UC_NT]
	const int tid = (int)threadIdx.x;
	const int x = (int)blockIdx.x * UC_NT + tid;
	const bool live = x < W;
	const int xc = live ? x : W - 1;                                // dead lanes shadow the last column and never store
	const uint32_t z = z_start + blockIdx.y * z_step;
	const uint64_t fpx = (uint64_t)W * H;
	const bool zflag = (video & (int)z & 1) != 0;
	const uint16_t* s = sym + (uint64_t)z * fpx + xc;
	uint16_t* o = out + (uint64_t)z * fpx + xc;
	const int tx = xc / T, u = xc - tx * T;
	const bool chain_warp = WAY == 1 && blockIdx.x == 0 && tid < 32;  // columns 0..31 hold the first tile (T <= 32)
	ring[tid] = __ldcg(o);                                          // row 0: decoded by k_unpredict_row0 before
	int up = (int)ring[tid];
	uint32_t q[UC_D];                                               // symbol | previous-frame pixel << 16
	auto fetch = [&](int y) -> uint32_t {
		if (y >= H) return 0u;
		uint32_t v2 = (uint32_t)__ldg(s + (size_t)y * W);
		if (zflag) v2 |= (uint32_t)__ldcg(o + (size_t)y * W - fpx) << 16;
		return v2;
	};
	#pragma unroll
	for (int d = 0; d < UC_D; d++) q[d] = fetch(1 + d);
	int v = T > 1 ? 1 : 0, slot = v, tyc = T > 1 ? 0 : 1;           // row y: v = y mod T = ring slot, tyc = (y >= T)
	for (int y0 = 1; y0 < H; y0 += UC_D) {
		#pragma unroll
		for (int d = 0; d < UC_D; d++) {
			const int y = y0 + d;
			if (y < H) {                                              // uniform
				const uint32_t qq = q[d];
				q[d] = fetch(y + UC_D);
				const int ut = (int)ring[slot * UC_NT + tid];
				// predict0 for k = 2 written out (lfm_predict.cuh): first tile row: U.  Below it -- way tiles: Ut where the rule
				// has no near neighbour (u == 0; in the first tile column v == 0), else (U + Ut) >> 1; way angle: Ut for the tile
				// DC, else U (the L of the first tile column is patched below).
				int p;
				if (!tyc) p = up;
				else if (WAY == 0) p = (tx == 0 ? v == 0 : u == 0) ? ut : ((up + ut) >> 1);
				else p = (u == 0 && v == 0) ? ut : up;
				if (WAY == 0 && zflag) p = (p + (int)(qq >> 16)) >> 1;  // (x, y) != (0, 0) here
				const int res = unsymbolize16((uint16_t)qq);
				int val = (res + p) & 0xffff;
				if (chain_warp && v == 0 && tyc) {                      // way angle, tile column 0, first row of a tile below the first: pred = L
					for (int uu = 1; uu < T; uu++) {
						const int l = __shfl_sync(0xffffffffu, val, uu - 1);
						if (tid == uu) val = (res + l) & 0xffff;
					}
				}
				if (live) o[(size_t)y * W] = (uint16_t)val;
				ring[slot * UC_NT + tid] = (uint16_t)val;
				up = val;
				if (++v == T) { v = 0; tyc = 1; }
				slot = v;
			}
		}
	}
}

// ---------------------------------------------------------------------------------------------------------
// Band-pipelined inverse (way "tiles" incl. video; any way whose rule only looks at the operands listed below; not
// predictor 2 of the ways tiles / angle, whose U crosses the tile border).
//
// A CTA owns a BAND of R tile rows of one frame; thread (j, u, v) owns in-tile position (u, v) of band row j and walks
// along its tile row: at wavefront step w it decodes tile  tx = w - (u + v + j + 1).  Every operand of the rule function
// is then the output of a thread of the same CTA one or two steps earlier:
//     (-1,0) (0,-1) (-T,0) (0,-T)                          step w-1     (left, up, same pixel of the left / upper tile)
//     (-1,-1) (-T,-T) (-1,-T) (0,-T-1) (-T,-1) (-T-1,0)    step w-2
// so the chain runs through a 4-deep shared-memory ring of "what every thread produced at step s" with ONE named
// barrier per step and all R*T*T threads busy in the steady state -- no fill / drain per block of tiles.  The row above
// the band (last tile row of the previous band, decoded by ANOTHER CTA) enters the ring as virtual row 0, fed by the
// threads of band row 0 from global memory.  Residual symbols, the row above and (video) the previous frame are
// prefetched UB_D steps ahead into registers, so no global latency sits on the chain; decoded pixels are stored as they
// are produced.
// Bands of a frame form a software pipeline through global progress flags (number of wavefront steps the band has
// completed: the band below may run R + UB_D + 1 steps behind, it never waits for whole tiles).  Three helper warps keep
// every fence off the compute threads:
//   signal    joins each step's barrier and releases the step count to the CTA (the barrier orders the pixel stores
//             of the compute threads before that release);
//   publisher free running: acquires the step count, gpu-scope fence, stores the progress flag -- the fence costs
//             microseconds while stores are in flight, and nobody inside the CTA waits for it;
//   poller    reads the flag of the band above, fences, and passes the count on through shared memory, where the threads
//             of band row 0 look before they prefetch from the row above (ld.global.cg, issued after the value was
//             seen: L2 already holds the data).
// The compute threads never execute a fence, so their register prefetch queues stay in flight across steps.  CTAs are
// numbered band-major (all frames' band b before any band b+1): a CTA only waits for a CTA with a smaller index, and
// the bands in flight belong to as many different frames as possible.
constexpr int UB_D = 4;                 // prefetch distance, wavefront steps
constexpr int UB_HELPERS = 96;          // three helper warps: signal, publisher, poller (one lane each is active)

__device__ __forceinline__ uint32_t ub_ld_acquire_cta(const uint32_t* p)
{
	uint32_t v; asm volatile("ld.acquire.cta.shared.u32 %0, [%1];" : "=r"(v) : "r"((uint32_t)__cvta_generic_to_shared(p)) : "memory"); return v;
}
__device__ __forceinline__ void ub_st_release_cta(uint32_t* p, uint32_t v)
{
	asm volatile("st.release.cta.shared.u32 [%0], %1;" :: "r"((uint32_t)__cvta_generic_to_shared(p)), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ub_ld_relaxed_gpu(const uint32_t* p)
{
	uint32_t v; asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v;
}
__device__ __forceinline__ void ub_st_relaxed_gpu(uint32_t* p, uint32_t v)
{
	asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void ub_fence_gpu() { asm volatile("fence.acq_rel.gpu;" ::: "memory"); }

template <int WAY, int K, int ZF>
__global__ void __launch_bounds__(1024, 1)   // at most 64 registers: two CTAs of <= 512 threads (or four of 256) share an SM
k_unpredict_bands(const uint16_t* __restrict__ sym, uint16_t* out, int W, int H, int T,
                  uint32_t z_start, uint32_t z_step, uint32_t count, int R, int ncomp, uint32_t* flags)
{
	extern __shared__ __align__(16) uint8_t ub_smem[];
	__shared__ uint32_t s_avail, s_step, s_ticket;
	__builtin_assume(T >= 2);
	const int tid = (int)threadIdx.x;
	const int TT = T * T;
	const int tilesX = (W + T - 1) / T, tilesY = (H + T - 1) / T;
	const int nbands = (tilesY + R - 1) / R;
	// a band waits for the band above it: the logical (band-major) id is a ticket taken when the CTA starts running, so a
	// CTA only ever waits for a CTA that is already resident -- whatever order the hardware dispatches blockIdx in
	if (tid == 0) s_ticket = atomicAdd(flags + (size_t)gridDim.x, 1u);
	__syncthreads();
	const uint32_t bid = s_ticket;
	const uint32_t fi = bid % count;
	const int band = (int)(bid / count);
	const uint32_t z = z_start + fi * z_step;
	const uint64_t fpx = (uint64_t)W * H;
	const int last_skew = 2 * T - 2 + R;                         // u + v + j + 1 of the band's last thread
	const int nsteps = tilesX + last_skew;
	uint32_t* f_mine = flags + (size_t)fi * nbands + band;
	const uint32_t* f_above = f_mine - 1;
	if (tid == 0) s_step = 0;
	if (tid == 0) s_avail = band == 0 ? 0x7fffffffu : 0u;     // wavefront steps the band above has completed
	const int RS = (R + 1) * TT + T + 2;                        // ring row: T+2 guard elements, virtual row 0, R band rows
	uint16_t* ring = reinterpret_cast<uint16_t*>(ub_smem);
	for (int i = tid; i < 4 * RS; i += (int)blockDim.x) ring[i] = 0;
	__syncthreads();

	const int nsteps_run = (nsteps + UB_D - 1) / UB_D * UB_D;    // the step loop is unrolled by UB_D
	if (tid >= ncomp) {
		// ---- helper warps: all global synchronisation
		if (tid < ncomp + 32) {
			// signal warp: joins EVERY compute barrier (it has no memory operations of its own in flight, so it never delays
			// one) and releases the count of complete steps to the CTA -- the barrier orders the compute threads' pixel
			// stores before this release
			for (int w = 0; w <= nsteps_run; w++) {
				asm volatile("bar.sync 1, %0;" :: "r"(ncomp + 32) : "memory");      // steps < w are complete
				if (tid == ncomp) ub_st_release_cta(&s_step, w >= nsteps_run ? 0x7fffffffu : (uint32_t)w);
			}
		} else if (tid == ncomp + 32) {
			// publisher lane, free running: acquire the step count, gpu-scope fence, store the progress flag.  The fence takes
			// microseconds under load; nothing waits for it except the band below.
			uint32_t published = 0;
			while (published < 0x7fffffffu) {
				const uint32_t sd = ub_ld_acquire_cta(&s_step);
				if (sd > published) { ub_fence_gpu(); ub_st_relaxed_gpu(f_mine, sd); published = sd; }
			}
		} else if (tid == ncomp + 64 && band > 0) {             // poller of the band above
			uint32_t avail = 0;
			while (avail < 0x7fffffffu) {
				const uint32_t f = ub_ld_relaxed_gpu(f_above);
				if (f > avail) { ub_fence_gpu(); avail = f; *(volatile uint32_t*)&s_avail = f; }
			}
		}
		return;
	}

	// ---- compute threads
	// thread -> (band row j, u, v), ordered by rule class so that (almost) every warp runs ONE branch of the rule function:
	// first the general pixels (u > 0, v > 0) of all band rows, then the first columns (u == 0), the first rows (v == 0), the DCs
	int j, u, v;
	{
		const int T1 = T - 1, G = T1 * T1, NG = R * G, NA = R * T1;
		if (tid < NG) { j = tid / G; const int i = tid - j * G; v = 1 + i / T1; u = 1 + i - (v - 1) * T1; }
		else if (tid < NG + NA) { const int i = tid - NG; j = i / T1; u = 0; v = 1 + i - j * T1; }
		else if (tid < NG + 2 * NA) { const int i = tid - NG - NA; j = i / T1; v = 0; u = 1 + i - j * T1; }
		else if (tid < R * TT) { j = tid - NG - 2 * NA; u = 0; v = 0; }
		else { j = R; u = 0; v = 0; }                               // padding threads of the last warp
	}
	const int p = v * T + u;
	const int ty = band * R + j, y = ty * T + v;
	const bool row_ok = j < R && ty < tilesY && y < H;
	const bool feeds_above = row_ok && j == 0 && band > 0;
	const int skew = u + v + j + 1;
	const int tyc = ty > 0 ? 1 : 0;                             // the rules only ask whether tx / ty are zero
	const unsigned ntx = row_ok ? (unsigned)((W - u + T - 1) / T) : 0u;     // tiles t of my row with t * T + u < W
	const int yy = row_ok ? y : 0;
	// ring: 4 rows (slot = step & 3, static inside the unrolled loop), my element first
	uint16_t* const rme = ring + T + 2 + (j + 1) * TT + p;
	// running pointers: tile tx + UB_D of the symbol row (and previous frame), tile tx + 1 + UB_D of the row above, tile tx of the output
	int tx = -skew;
	const int64_t rowoff = (int64_t)z * (int64_t)fpx + (int64_t)yy * W + u;
	const uint16_t* sp = sym + rowoff + (int64_t)(tx + UB_D) * T;
	const uint16_t* pp = out + rowoff - (int64_t)fpx + (int64_t)(tx + UB_D) * T;        // previous frame (odd video frames)
	const uint16_t* ap = out + rowoff - (int64_t)T * W + (int64_t)(tx + 1 + UB_D) * T;  // same (u, v) one tile row up
	uint16_t* op = out + rowoff + (int64_t)tx * T;
	// The pixel above my tile ta = w - u - v (entering the ring at step w) was produced by the last row of the band above
	// at ITS step ta + u + v + R = w + R: the prefetch for step w + UB_D needs w + UB_D + R + 1 complete steps up there.
	auto wait_above = [&](int w_use) {
		const uint32_t need = (uint32_t)(w_use + R + 1);
		while (*(volatile uint32_t*)&s_avail < need) { }          // written by the poller lane after its gpu-scope fence
	};

	uint32_t sq[UB_D], aq[UB_D];                                // sq: symbol | previous-frame pixel << 16
	#pragma unroll
	for (int d = 0; d < UB_D; d++) {
		const unsigned t = (unsigned)(d - skew);
		sq[d] = 0; aq[d] = 0;
		if (t < ntx) {
			sq[d] = (uint32_t)__ldg(sp + (int64_t)(d - UB_D) * T);
			if (ZF) sq[d] |= (uint32_t)__ldcg(pp + (int64_t)(d - UB_D) * T) << 16;
		}
		if (feeds_above && t + 1u < ntx) { wait_above(d); aq[d] = (uint32_t)__ldcg(ap + (int64_t)(d - UB_D) * T); }
	}
	int my_prev = 0, ut_prev = 0;                                // my pixel / the pixel above it, one tile to the left

	for (int w0 = 0; w0 < nsteps; w0 += UB_D) {
		#pragma unroll
		for (int d = 0; d < UB_D; d++) {
			uint16_t* const C = rme + (d & 3) * RS;                  // written this step
			const uint16_t* const P1 = rme + ((d + 3) & 3) * RS;     // one step ago
			const uint16_t* const P2 = rme + ((d + 2) & 3) * RS;     // two steps ago
			asm volatile("bar.sync 1, %0;" :: "r"(ncomp + 32) : "memory");    // compute threads + the signal warp
			const uint32_t q = sq[d];
			{	// refill the queue for step w + UB_D
				uint32_t nv = 0;
				if ((unsigned)(tx + UB_D) < ntx) {
					nv = (uint32_t)__ldg(sp);
					if (ZF) nv |= (uint32_t)__ldcg(pp) << 16;
				}
				sq[d] = nv;
				sp += T; if (ZF) pp += T;
			}
			if (feeds_above) {                                      // virtual row 0: the pixel above tile tx + 1
				C[-TT] = (uint16_t)aq[d];
				const unsigned t = (unsigned)(tx + 1 + UB_D);
				if (t < ntx) { wait_above(w0 + d + UB_D); aq[d] = (uint32_t)__ldcg(ap); }
				ap += T;
			}
			if ((unsigned)tx < ntx) {
				const int ut = (int)P1[-TT];
				auto px = [&](int dx, int dy) -> int {
					const bool fx = dx <= -T, fy = dy <= -T;
					const int nx = fx ? dx + T : dx, ny = fy ? dy + T : dy;          // near part: 0 or -1
					if (nx == 0 && ny == 0) return (fx && fy) ? ut_prev : fx ? my_prev : ut;
					const int back = (fx ? 1 : 0) + (fy ? 1 : 0) - nx - ny;          // 1 or 2 steps ago
					const uint16_t* base = back == 1 ? P1 : P2;
					return (int)base[(fy ? -TT : 0) + nx + ny * T];
				};
				int pr = tx == 0 ? predict0(px, T, WAY, K, 0, tyc, u, v) : predict0(px, T, WAY, K, 1, tyc, u, v);
				if (ZF) pr = (tx == 0 && ty == 0 && u == 0 && v == 0) ? (int)(q >> 16) : ((pr + (int)(q >> 16)) >> 1);
				const uint16_t val = (uint16_t)(unsymbolize16((uint16_t)q) + pr);
				C[0] = val;
				*op = val;
				my_prev = (int)val; ut_prev = ut;
			}
			op += T; tx++;
		}
	}
	asm volatile("bar.sync 1, %0;" :: "r"(ncomp + 32) : "memory");                            // w == nsteps_run: everything is stored
}

// =====================================================================================================
// Way "space", predictors 1, 2 and 4: the rule is LINEAR modulo 2^16 (the same sub-aperture pixel of the left / upper / both
// neighbouring microlenses, src/lfm_Predictors_space.cu), so the inverse is a strided prefix sum and needs no wavefront:
//   k = 4:  pixel = 2-D prefix sum, over the tile grid (tx, ty) of its sub-aperture image (u, v), of the residuals -- with
//           tile (0,0) (decoded by k_unpredict_seed) as the corner term: a column pass (stride T rows) and a row pass (stride T
//           pixels), the second one in place;
//   k = 1:  first tile column by a column pass (its rule looks up), then every row by a row pass seeded with that column;
//   k = 2:  first tile row by a row pass, then every column by a column pass seeded with that row.
// Both passes stream whole 128-byte lines; frames are processed in groups that fit L2, so the in-place second pass reads what
// the first one has just written.  Arithmetic is 2 x 16 bits per 32-bit word (__vadd2 wraps each half: exactly the int16
// truncation of the reference).
// element source rules for the heads of the chains: 0 = residual, 1 = from `out` inside tile (0,0) only (the seed),
// 2 = from `out` for the whole first tile column / row (already final)
// =====================================================================================================
__device__ __forceinline__ uint32_t unsymbolize16x2(uint32_t w)
{
	return ((w >> 1) & 0x7FFF7FFFu) ^ ((w & 0x00010001u) * 0xFFFFu);      // per half: (s >> 1) ^ -(s & 1)
}

template <bool SRC_OUT, int SC_ROWS_NT>
__global__ void __launch_bounds__(SC_ROWS_NT)
k_unscan_rows(const uint16_t* __restrict__ sym, uint16_t* out, int W, int H, int T, uint32_t z_start, uint32_t z_step,
              int rows_per_cta, int y_limit, int head_rule, int pitch)
{
	extern __shared__ __align__(16) uint16_t sc_rows[];                   // [rows_per_cta][pitch]
	const int tid = (int)threadIdx.x;
	const uint32_t z = z_start + blockIdx.y * z_step;
	const uint64_t fbase = (uint64_t)z * W * H;
	const int y0 = (int)blockIdx.x * rows_per_cta;
	const int nrows = min(rows_per_cta, min(H, y_limit) - y0);
	if (nrows <= 0) return;
	const uint16_t* src = (SRC_OUT ? (const uint16_t*)out : sym) + fbase;
	const uint16_t* o = out + fbase;
	// rows are whole 16-byte vectors of 16-byte aligned buffers (a view into a caller's tensor need not be)
	const bool vec = ((W & 7) == 0) && ((((uintptr_t)sym | (uintptr_t)out) & 15) == 0);
	if (vec) {
		const int vpr = W >> 3;
		for (int i = tid; i < nrows * vpr; i += SC_ROWS_NT) {
			const int r = i / vpr, xv = i - r * vpr;
			uint4 q = *reinterpret_cast<const uint4*>(src + (size_t)(y0 + r) * W + xv * 8);
			if (!SRC_OUT) { q.x = unsymbolize16x2(q.x); q.y = unsymbolize16x2(q.y); q.z = unsymbolize16x2(q.z); q.w = unsymbolize16x2(q.w); }
			*reinterpret_cast<uint4*>(sc_rows + (size_t)r * pitch + xv * 8) = q;
		}
	} else {
		for (int i = tid; i < nrows * W; i += SC_ROWS_NT) {
			const int r = i / W, x = i - r * W;
			const uint16_t sv = src[(size_t)(y0 + r) * W + x];
			sc_rows[(size_t)r * pitch + x] = SRC_OUT ? sv : (uint16_t)unsymbolize16(sv);
		}
	}
	__syncthreads();
	if (!SRC_OUT && head_rule) {                                          // heads of the chains that are already decoded
		const int tw = min(T, W);
		for (int i = tid; i < nrows * tw; i += SC_ROWS_NT) {
			const int r = i / tw, x = i - r * tw;
			if (head_rule == 2 || y0 + r < T) sc_rows[(size_t)r * pitch + x] = o[(size_t)(y0 + r) * W + x];
		}
		__syncthreads();
	}
	for (int g = tid; g < nrows * T; g += SC_ROWS_NT) {                   // thread = (row, u): the chain over tx
		const int r = g / T, u = g - r * T;
		uint16_t* row = sc_rows + (size_t)r * pitch;
		uint32_t acc = 0;
		for (int xb = u; xb < W; xb += 8 * T) {                             // eight loads first: the stores below may alias them
			uint32_t val[8];
			#pragma unroll
			for (int j = 0; j < 8; j++) { const int x = xb + j * T; val[j] = x < W ? row[x] : 0u; }
			#pragma unroll
			for (int j = 0; j < 8; j++) { const int x = xb + j * T; acc += val[j]; if (x < W) row[x] = (uint16_t)acc; }
		}
	}
	__syncthreads();
	uint16_t* dst = out + fbase;
	if (vec) {
		const int vpr = W >> 3;
		for (int i = tid; i < nrows * vpr; i += SC_ROWS_NT) {
			const int r = i / vpr, xv = i - r * vpr;
			*reinterpret_cast<uint4*>(dst + (size_t)(y0 + r) * W + xv * 8) = *reinterpret_cast<const uint4*>(sc_rows + (size_t)r * pitch + xv * 8);
		}
	} else {
		for (int i = tid; i < nrows * W; i += SC_ROWS_NT) { const int r = i / W, x = i - r * W; dst[(size_t)(y0 + r) * W + x] = sc_rows[(size_t)r * pitch + x]; }
	}
}

constexpr int SC_COLS_NT = 128;
constexpr int SC_COLS_B = 12;                                             // rows fetched ahead of the running sum
// thread = (VEC adjacent columns, v): the chain over ty.  VEC = 4 / 2 need W to be a multiple of 4 / 2 (64- / 32-bit accesses).
template <bool SRC_OUT, int VEC>
__global__ void __launch_bounds__(SC_COLS_NT)
k_unscan_cols(const uint16_t* __restrict__ sym, uint16_t* out, int W, int H, int T, uint32_t z_start, uint32_t z_step,
              int x_limit, int head_rule)
{
	const int x = VEC * (int)(blockIdx.x * SC_COLS_NT + threadIdx.x);
	if (x >= min(W, x_limit)) return;
	const int v = (int)blockIdx.y;
	if (v >= H) return;
	const uint32_t z = z_start + blockIdx.z * z_step;
	const uint64_t fbase = (uint64_t)z * W * H;
	const uint16_t* src = (SRC_OUT ? (const uint16_t*)out : sym) + fbase;
	uint16_t* o = out + fbase;
	constexpr int NW = VEC == 4 ? 2 : 1;                                    // 32-bit words per thread and row
	uint32_t acc[NW];
	#pragma unroll
	for (int w = 0; w < NW; w++) acc[w] = 0;
	for (int yb = v; yb < H; yb += T * SC_COLS_B) {
		uint32_t val[SC_COLS_B][NW];
		#pragma unroll
		for (int j = 0; j < SC_COLS_B; j++) {                               // independent loads first: the stores below may alias them
			const int y = yb + j * T;
			#pragma unroll
			for (int w = 0; w < NW; w++) val[j][w] = 0;
			if (y < H) {
				const size_t at = (size_t)y * W + x;
				if (VEC == 1) {
					uint32_t sv = src[at];
					if (!SRC_OUT) { sv = (uint32_t)unsymbolize16((uint16_t)sv) & 0xffffu; if (y < T && head_rule && (head_rule == 2 || x < T)) sv = o[at]; }
					val[j][0] = sv;
				} else {
					uint32_t wv[NW];
					if (VEC == 4) { const uint2 q = *reinterpret_cast<const uint2*>(src + at); wv[0] = q.x; wv[NW - 1] = q.y; }
					else wv[0] = *reinterpret_cast<const uint32_t*>(src + at);
					if (!SRC_OUT) {
						#pragma unroll
						for (int w = 0; w < NW; w++) {
							wv[w] = unsymbolize16x2(wv[w]);
							if (y < T && head_rule) {                           // heads that are already decoded (per half)
								const uint32_t ov = *reinterpret_cast<const uint32_t*>(o + at + 2 * w);
								const bool h0 = head_rule == 2 || x + 2 * w < T, h1 = head_rule == 2 || x + 2 * w + 1 < T;
								wv[w] = (h0 ? (ov & 0xffffu) : (wv[w] & 0xffffu)) | (h1 ? (ov & 0xffff0000u) : (wv[w] & 0xffff0000u));
							}
						}
					}
					#pragma unroll
					for (int w = 0; w < NW; w++) val[j][w] = wv[w];
				}
			}
		}
		#pragma unroll
		for (int j = 0; j < SC_COLS_B; j++) {
			const int y = yb + j * T;
			if (y < H) {
				const size_t at = (size_t)y * W + x;
				if (VEC == 1) { acc[0] = (acc[0] + val[j][0]) & 0xffffu; o[at] = (uint16_t)acc[0]; }
				else {
					#pragma unroll
					for (int w = 0; w < NW; w++) acc[w] = __vadd2(acc[w], val[j][w]);
					if (VEC == 4) *reinterpret_cast<uint2*>(o + at) = make_uint2(acc[0], acc[NW - 1]);
					else *reinterpret_cast<uint32_t*>(o + at) = acc[0];
				}
			}
		}
	}
}

// The column pass for whole frames with every load independent (the chain of k_unscan_cols waits a DRAM latency per batch of 12
// rows: ncu 72 % long-scoreboard stalls, 13 warps per SM): CTA = 32 column quads x SEG warps, one v; warp s owns Q consecutive
// tile rows of the chain, fetches its Q rows at once, sums them in registers, and the warps' totals are combined through shared
// memory (two levels: no serial dependence between loads).  Chains longer than SEG * Q rows take further rounds with a carry.
constexpr int SC_SEG = 16, SC_Q = 9;
__global__ void __launch_bounds__(32 * SC_SEG)
k_unscan_cols_seg(const uint16_t* __restrict__ sym, uint16_t* out, int W, int H, int T, uint32_t z_start, uint32_t z_step, int head_rule)
{
	__shared__ uint2 tot[SC_SEG][32];
	const int lane = (int)threadIdx.x, s = (int)threadIdx.y;
	const int x = 4 * (int)(blockIdx.x * 32 + lane);
	const int v = (int)blockIdx.y;
	const bool live = x < W;                                              // W is a multiple of 4 here
	const uint32_t z = z_start + blockIdx.z * z_step;
	const uint64_t fbase = (uint64_t)z * W * H;
	const uint16_t* src = sym + fbase;
	uint16_t* o = out + fbase;
	const int NR = (H - v + T - 1) / T;                                   // rows of this chain: y = v + T i
	uint2 carry = make_uint2(0u, 0u);
	for (int r0 = 0; r0 < NR; r0 += SC_SEG * SC_Q) {
		const int i0 = r0 + s * SC_Q;
		uint2 val[SC_Q];
		#pragma unroll
		for (int j = 0; j < SC_Q; j++) {
			const int i = i0 + j;
			val[j] = make_uint2(0u, 0u);
			if (live && i < NR) {
				const size_t at = (size_t)(v + T * i) * W + x;
				uint2 q = *reinterpret_cast<const uint2*>(src + at);
				q.x = unsymbolize16x2(q.x); q.y = unsymbolize16x2(q.y);
				if (i == 0 && head_rule) {                                    // heads that are already decoded (per half); row y = v < T
					const uint2 ov = *reinterpret_cast<const uint2*>(o + at);
					const bool h0 = head_rule == 2 || x < T, h1 = head_rule == 2 || x + 1 < T, h2 = head_rule == 2 || x + 2 < T, h3 = head_rule == 2 || x + 3 < T;
					q.x = (h0 ? (ov.x & 0xffffu) : (q.x & 0xffffu)) | (h1 ? (ov.x & 0xffff0000u) : (q.x & 0xffff0000u));
					q.y = (h2 ? (ov.y & 0xffffu) : (q.y & 0xffffu)) | (h3 ? (ov.y & 0xffff0000u) : (q.y & 0xffff0000u));
				}
				val[j] = q;
			}
		}
		#pragma unroll
		for (int j = 1; j < SC_Q; j++) { val[j].x = __vadd2(val[j].x, val[j - 1].x); val[j].y = __vadd2(val[j].y, val[j - 1].y); }
		tot[s][lane] = val[SC_Q - 1];
		__syncthreads();
		uint2 before = carry, all = carry;
		#pragma unroll
		for (int k = 0; k < SC_SEG; k++) {
			const uint2 t = tot[k][lane];
			all.x = __vadd2(all.x, t.x); all.y = __vadd2(all.y, t.y);
			if (k < s) { before.x = __vadd2(before.x, t.x); before.y = __vadd2(before.y, t.y); }
		}
		carry = all;
		#pragma unroll
		for (int j = 0; j < SC_Q; j++) {
			const int i = i0 + j;
			if (live && i < NR) {
				const size_t at = (size_t)(v + T * i) * W + x;
				*reinterpret_cast<uint2*>(o + at) = make_uint2(__vadd2(val[j].x, before.x), __vadd2(val[j].y, before.y));
			}
		}
		__syncthreads();
	}
}

// returns 0 ok, 1 launch error, 2 not applicable
static int launch_unpredict_space_scans(const uint16_t* sym, uint16_t* out, int W, int H, int T, int k,
                                        uint32_t z_start, uint32_t z_step, uint32_t count, cudaStream_t st)
{
	if (k != 1 && k != 2 && k != 4) return 2;
	const int vec = ((W & 3) == 0 && ((((uintptr_t)sym | (uintptr_t)out) & 7) == 0)) ? 4 : ((W & 1) == 0 && ((((uintptr_t)sym | (uintptr_t)out) & 3) == 0)) ? 2 : 1;
	const int pitch = ((W + 7) & ~7) + 16;                               // +8 words: the rows of a CTA start in different banks (the chain threads of one step touch R rows)
	// rows per CTA: R * T chain threads; small CTAs (R = 8, 128 threads) so that seven of them share an SM and the load, chain and
	// store phases of different CTAs overlap (R = 16 / 256 threads: 4 per SM, ncu 45 % of the warp slots, DRAM latency exposed)
	static const int r_forced = getenv("LFM_B200_SCAN_R") ? atoi(getenv("LFM_B200_SCAN_R")) : 0;
	int R = std::min(r_forced > 0 ? r_forced : 8, (int)((48 * 1024) / ((size_t)pitch * 2)));
	if (R < 1) return 2;                                                   // rows wider than 24 K pixels: the wavefront kernels
	while (R > 1 && (uint64_t)((H + R - 1) / R) * count < 592) R >>= 1;     // enough CTAs for a single frame
	const int rnt = R * T > 128 ? 256 : R * T > 64 ? 128 : 64;
	const size_t rsmem = (size_t)R * pitch * 2;
	const unsigned wpb = UF_NT / 32;
	k_unpredict_seed<<<(count + wpb - 1) / wpb, UF_NT, 0, st>>>(sym, out, W, H, T, 2, k, z_start, z_step, count, 0);
	// frames in groups whose symbols + pixels fit L2, so that the second pass finds the first one's output there
	const uint64_t fbytes = (uint64_t)W * H * 2;
	const uint32_t group = (uint32_t)std::min<uint64_t>(65535, std::max<uint64_t>(1, ((uint64_t)64 << 20) / fbytes));
	auto rows = [&](bool src_out, uint32_t zs, uint32_t n, int y_limit, int head) {
		const dim3 grid((unsigned)((std::min(H, y_limit) + R - 1) / R), n);
		#define LFM_ROWS(SO, NT) k_unscan_rows<SO, NT><<<grid, NT, rsmem, st>>>(sym, out, W, H, T, zs, z_step, R, y_limit, head, pitch)
		if (src_out) { if (rnt == 256) LFM_ROWS(true, 256); else if (rnt == 128) LFM_ROWS(true, 128); else LFM_ROWS(true, 64); }
		else { if (rnt == 256) LFM_ROWS(false, 256); else if (rnt == 128) LFM_ROWS(false, 128); else LFM_ROWS(false, 64); }
		#undef LFM_ROWS
	};
	auto cols = [&](uint32_t zs, uint32_t n, int x_limit, int head) {
		const int xl = std::min(W, x_limit);
		const int vc = x_limit >= W ? vec : 1;                              // the restricted pass stops at a column that need not be even
		const int nthr = (xl + vc - 1) / vc;
		const dim3 grid((unsigned)((nthr + SC_COLS_NT - 1) / SC_COLS_NT), (unsigned)std::min(T, H), n);
		static const int seg_on = getenv("LFM_B200_SCAN_SEG") ? atoi(getenv("LFM_B200_SCAN_SEG")) : 1;
		if (vc == 4 && seg_on) {
			const dim3 g2((unsigned)((W / 4 + 31) / 32), (unsigned)std::min(T, H), n);
			k_unscan_cols_seg<<<g2, dim3(32, SC_SEG), 0, st>>>(sym, out, W, H, T, zs, z_step, head);
		}
		else if (vc == 4) k_unscan_cols<false, 4><<<grid, SC_COLS_NT, 0, st>>>(sym, out, W, H, T, zs, z_step, x_limit, head);
		else if (vc == 2) k_unscan_cols<false, 2><<<grid, SC_COLS_NT, 0, st>>>(sym, out, W, H, T, zs, z_step, x_limit, head);
		else k_unscan_cols<false, 1><<<grid, SC_COLS_NT, 0, st>>>(sym, out, W, H, T, zs, z_step, x_limit, head);
	};
	const int ALL = 0x7fffffff;
	if (k == 4) {
		for (uint32_t f0 = 0; f0 < count; f0 += group) {
			const uint32_t n = std::min(group, count - f0), zs = z_start + f0 * z_step;
			cols(zs, n, ALL, 1); rows(true, zs, n, ALL, 0);
		}
	} else {
		// one restricted pass (first tile column / row: a short latency-bound launch, so ONE launch for all frames), then one
		// full pass straight from the symbols: nothing to keep in L2 between them
		for (uint32_t f0 = 0; f0 < count; f0 += 65535u) {
			const uint32_t n = std::min(65535u, count - f0), zs = z_start + f0 * z_step;
			if (k == 1) { cols(zs, n, T, 1); rows(false, zs, n, ALL, 2); }
			else { rows(false, zs, n, T, 1); cols(zs, n, ALL, 2); }
		}
	}
	return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

// per-device progress flags of the band pipeline (grown on demand; launches on one device are stream-ordered by the engine)
static uint32_t* ub_flags(size_t n)
{
	static uint32_t* buf[64] = { nullptr }; static size_t cap[64] = { 0 };
	int dev = 0; cudaGetDevice(&dev); dev &= 63;
	if (cap[dev] < n) {
		if (buf[dev]) cudaFree(buf[dev]);
		buf[dev] = nullptr; cap[dev] = 0;
		const size_t want = n + n / 2 + 1024;
		if (cudaMalloc(&buf[dev], want * 4) != cudaSuccess) { cudaGetLastError(); return nullptr; }
		cap[dev] = want;
	}
	return buf[dev];
}

// returns 0 ok, 1 launch error, 2 shape not supported by this path
template <int WAY>
static int launch_unpredict_bands(const uint16_t* sym, uint16_t* out, int W, int H, int T, int k, int zflag,
                                  uint32_t z_start, uint32_t z_step, uint32_t count, cudaStream_t st)
{
	const int TT = T * T;
	int R = 0;
	while ((((R + 1) * TT + 31) & ~31) + UB_HELPERS <= 1024) R++;
	if (R == 0) return 2;
	static const int r_max = getenv("LFM_B200_BANDS_R") ? atoi(getenv("LFM_B200_BANDS_R")) : 1024;
	const int tilesY = (H + T - 1) / T;
	R = std::max(1, std::min(std::min(R, r_max), tilesY));
	const int ncomp = (R * TT + 31) & ~31;
	const int nbands = (tilesY + R - 1) / R;
	const uint64_t nctas = (uint64_t)nbands * count;
	if (nctas > 0x7fffffffull) return 2;
	uint32_t* flags = ub_flags((size_t)nctas + 1);              // progress flag per CTA + the ticket counter
	if (!flags) return 2;
	cudaMemsetAsync(flags, 0, ((size_t)nctas + 1) * 4, st);
	const size_t smem = (size_t)4 * ((R + 1) * TT + T + 2) * 2;
	#define LFM_UB(KK) do { if (zflag) k_unpredict_bands<WAY, KK, 1><<<(unsigned)nctas, ncomp + UB_HELPERS, smem, st>>>(sym, out, W, H, T, z_start, z_step, count, R, ncomp, flags); \
		else k_unpredict_bands<WAY, KK, 0><<<(unsigned)nctas, ncomp + UB_HELPERS, smem, st>>>(sym, out, W, H, T, z_start, z_step, count, R, ncomp, flags); } while (0)
	switch (k) {
	case 1: LFM_UB(1); break; case 3: LFM_UB(3); break; case 4: LFM_UB(4); break;
	case 5: LFM_UB(5); break; case 6: LFM_UB(6); break; case 7: LFM_UB(7); break;
	case 2: if (WAY == 2) { LFM_UB(2); break; } return 2;
	default: return 2;
	}
	#undef LFM_UB
	return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link against libcuda)
typedef CUresult (*TensorMapEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                      const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static TensorMapEncodeFn tensor_map_encoder()
{
	static const TensorMapEncodeFn fn = [] {
		void* p = nullptr;
		cudaDriverEntryPointQueryResult q;
		if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) { cudaGetLastError(); p = nullptr; }
		return (TensorMapEncodeFn)p;
	}();
	return fn;
}

template <int WAY, int K>
static void launch_predict_fwd_wk(const uint16_t* img, uint16_t* sym, int W, int H, int T, int video, uint32_t z0, uint32_t nz,
                                  cudaStream_t st)
{
	const int hw = (T + 1 + 7) & ~7;
	const bool tile = hw <= PF_NT / 2;                          // halo of at most half the tile (Nnum <= 127)
	const int cols = tile ? PF_NT - hw : PF_NT;
	const int colchunks = (W + cols - 1) / cols;
	// band height: enough CTAs to fill the GPU for a single frame, tall tiles (less halo) for stacks; <= 48 KB of shared memory
	const bool pairs = tile && ((W & 7) == 0) && ((((uintptr_t)img | (uintptr_t)sym) & 15) == 0);   // rows are whole 16-byte vectors
	int band = pairs ? 32 : 64;                                 // 128-thread CTAs: smaller tiles keep ~36 warps per SM resident
	while (band > 16 && (uint64_t)colchunks * ((H + band - 1) / band) * nz < 1184) band >>= 1;
	while (band > 8 && (size_t)(band + T + 1) * PF_PITCH * 2 > 48 * 1024) band >>= 1;
	const size_t smem = (size_t)(band + T + 1) * PF_PITCH * 2;
	if (pairs) cudaFuncSetAttribute(k_predict_fwd2<WAY, K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
	else if (tile) cudaFuncSetAttribute(k_predict_fwd<WAY, K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
	static const int tma_on = getenv("LFM_B200_TMA") ? atoi(getenv("LFM_B200_TMA")) : 1;
	for (uint32_t zb = 0; zb < nz; zb += 65535) {            // gridDim.z limit
		const uint32_t cz = std::min<uint32_t>(65535, nz - zb);
		dim3 grid((unsigned)colchunks, (unsigned)((H + band - 1) / band), cz);
		if (pairs) {
			// tensor map of the cz frames of this launch: uint16 [cz][H][W], box = one tile + halo
			CUtensorMap tmap; memset(&tmap, 0, sizeof(tmap));
			int use_tma = 0;
			if (tma_on && tensor_map_encoder()) {
				const cuuint64_t gdim[3] = { (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)cz };
				const cuuint64_t gstr[2] = { (cuuint64_t)W * 2, (cuuint64_t)W * H * 2 };
				const cuuint32_t box[3] = { (cuuint32_t)PF_PITCH, (cuuint32_t)(band + T + 1), 1u };
				const cuuint32_t estr[3] = { 1u, 1u, 1u };
				void* base = const_cast<uint16_t*>(img + (uint64_t)(z0 + zb) * W * H);
				use_tma = tensor_map_encoder()(&tmap, CU_TENSOR_MAP_DATA_TYPE_UINT16, 3, base, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
				                               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
			}
			k_predict_fwd2<WAY, K><<<grid, PF2_NT, smem, st>>>(img, sym, W, H, T, video, z0 + zb, band, hw, tmap, use_tma);
		}
		else if (tile) k_predict_fwd<WAY, K><<<grid, PF_NT, smem, st>>>(img, sym, W, H, T, video, z0 + zb, band, hw);
		else k_predict_fwd_rows<WAY, K><<<grid, PF_NT, 0, st>>>(img, sym, W, H, T, video, z0 + zb, band);   // huge Nnum
	}
}

template <int WAY>
static void launch_predict_fwd_way(const uint16_t* img, uint16_t* sym, int W, int H, int T, int k, int video,
                                   uint32_t z0, uint32_t nz, cudaStream_t st)
{
	switch (k) {
	case 1: launch_predict_fwd_wk<WAY, 1>(img, sym, W, H, T, video, z0, nz, st); break;
	case 2: launch_predict_fwd_wk<WAY, 2>(img, sym, W, H, T, video, z0, nz, st); break;
	case 3: launch_predict_fwd_wk<WAY, 3>(img, sym, W, H, T, video, z0, nz, st); break;
	case 4: launch_predict_fwd_wk<WAY, 4>(img, sym, W, H, T, video, z0, nz, st); break;
	case 5: launch_predict_fwd_wk<WAY, 5>(img, sym, W, H, T, video, z0, nz, st); break;
	case 6: launch_predict_fwd_wk<WAY, 6>(img, sym, W, H, T, video, z0, nz, st); break;
	default: launch_predict_fwd_wk<WAY, 7>(img, sym, W, H, T, video, z0, nz, st); break;
	}
}

void launch_predict_fwd(const uint16_t* img, uint16_t* sym, int W, int H, int T, int way, int k, int video,
                        uint32_t z0, uint32_t nz, cudaStream_t st)
{
	if (nz == 0) return;
	if (way == 0) launch_predict_fwd_way<0>(img, sym, W, H, T, k, video, z0, nz, st);
	else if (way == 1) launch_predict_fwd_way<1>(img, sym, W, H, T, k, video, z0, nz, st);
	else launch_predict_fwd_way<2>(img, sym, W, H, T, k, video, z0, nz, st);
}

static int failed_launch(const char* kernel, const char** failed)
{
	if (failed) *failed = kernel;
	return 1;
}

// frames z_start, z_start+z_step, ... (count of them); video stacks: even frames first, then odd frames.
// Returns 0, or 1 if a launch fails; *failed then names the kernel(s) of the branch that failed.
int launch_unpredict(const uint16_t* sym, uint16_t* out, int W, int H, int T, int way, int k, int video,
                     uint32_t z_start, uint32_t z_step, uint32_t count, int sm_count, cudaStream_t st, const char** failed)
{
	(void)sm_count;
	if (count == 0) return 0;
	static const int bands_all = getenv("LFM_B200_BANDS") ? atoi(getenv("LFM_B200_BANDS")) : 1;
	if (bands_all >= 2 && !video && ((way == 1 && k != 2) || way == 2)) {      // measurement switch: every way through the band pipeline
		const int rcb = way == 1 ? launch_unpredict_bands<1>(sym, out, W, H, T, k, 0, z_start, z_step, count, st)
		                         : launch_unpredict_bands<2>(sym, out, W, H, T, k, 0, z_start, z_step, count, st);
		if (rcb != 2) return rcb ? failed_launch("k_unpredict_bands", failed) : 0;
	}
	const int tilesX = (W + T - 1) / T, tilesY = (H + T - 1) / T;
	const unsigned wpb = UF_NT / 32;
	// sub-images per CTA for the way "space" (neighbours in u share 32-byte sectors): as many as shared memory / 1024 threads allow
	const size_t plane_b = ((((size_t)tilesX * tilesY + 7) & ~(size_t)7) + 2 * ((size_t)tilesX + 1)) * 2;
	const int nxr = std::max(32, (tilesX + 31) & ~31);
	int G = std::min(4, T);
	while (G > 1 && ((size_t)G * plane_b + 16 > (size_t)UG_MAX_SMEM || G * nxr > 1024)) G--;
	const bool grid_ok = nxr <= 1024 && plane_b + 16 <= (size_t)UG_MAX_SMEM;
	static const int scans_on = getenv("LFM_B200_SCANS") ? atoi(getenv("LFM_B200_SCANS")) : 1;
	if (!video && way == 2 && scans_on) {                    // linear rules: strided prefix sums
		const int rcs = launch_unpredict_space_scans(sym, out, W, H, T, k, z_start, z_step, count, st);
		if (rcs != 2) return rcs ? failed_launch("k_unscan_rows / k_unscan_cols", failed) : 0;
	}
	if (!video && way == 2 && grid_ok) {                    // tile (0,0), then T*T sub-aperture recurrences per frame
		k_unpredict_seed<<<(count + wpb - 1) / wpb, UF_NT, 0, st>>>(sym, out, W, H, T, way, k, z_start, z_step, count, 0);
		const size_t smem = (size_t)G * plane_b + 16;
		const int ugroups = (T + G - 1) / G;
		launch_unpredict_grid<2>(sym, out, W, H, T, k, z_start, z_step, (unsigned)((uint64_t)count * T * ugroups), (unsigned)(G * nxr), smem, G, ugroups, T, nxr, st);
		return cudaGetLastError() == cudaSuccess ? 0 : failed_launch("k_unpredict_seed / k_unpredict_grid", failed);
	}
	const size_t strip_smem = (size_t)T * T * UT_NT * 2 + 16;
	if (!video && way == 1 && k != 2 && grid_ok && strip_smem <= (size_t)UG_MAX_SMEM) {   // DC grid, then every tile on its own
		launch_unpredict_grid<1>(sym, out, W, H, T, k, z_start, z_step, count, (unsigned)nxr, plane_b + 16, 1, 1, 1, nxr, st);
		const int chunks = (tilesX + UT_NT - 1) / UT_NT;
		switch (k) {
		case 1: launch_tiles_angle<1>(sym, out, W, H, T, z_start, z_step, count, tilesX, tilesY, chunks, strip_smem, st); break;
		case 3: launch_tiles_angle<3>(sym, out, W, H, T, z_start, z_step, count, tilesX, tilesY, chunks, strip_smem, st); break;
		case 4: launch_tiles_angle<4>(sym, out, W, H, T, z_start, z_step, count, tilesX, tilesY, chunks, strip_smem, st); break;
		case 5: launch_tiles_angle<5>(sym, out, W, H, T, z_start, z_step, count, tilesX, tilesY, chunks, strip_smem, st); break;
		case 6: launch_tiles_angle<6>(sym, out, W, H, T, z_start, z_step, count, tilesX, tilesY, chunks, strip_smem, st); break;
		default: launch_tiles_angle<7>(sym, out, W, H, T, z_start, z_step, count, tilesX, tilesY, chunks, strip_smem, st); break;
		}
		return cudaGetLastError() == cudaSuccess ? 0 : failed_launch("k_unpredict_grid / k_unpredict_tiles_angle", failed);
	}
	if (!video && way == 2) {                               // (fallback for tile grids that do not fit shared memory)
		k_unpredict_seed<<<(count + wpb - 1) / wpb, UF_NT, 0, st>>>(sym, out, W, H, T, way, k, z_start, z_step, count, 0);
		const uint64_t warps = (uint64_t)count * T * T;
		k_unpredict_space<<<(unsigned)((warps + wpb - 1) / wpb), UF_NT, 0, st>>>(sym, out, W, H, T, k, z_start, z_step, count);
		return cudaGetLastError() == cudaSuccess ? 0 : failed_launch("k_unpredict_seed / k_unpredict_space", failed);
	}
	if (!video && way == 1 && k != 2) {
		k_unpredict_seed<<<(count + wpb - 1) / wpb, UF_NT, 0, st>>>(sym, out, W, H, T, way, k, z_start, z_step, count, 1);
		const uint64_t warps = (uint64_t)count * tilesX * tilesY;
		k_unpredict_angle<<<(unsigned)((warps + wpb - 1) / wpb), UF_NT, 0, st>>>(sym, out, W, H, T, k, z_start, z_step, count);
		return cudaGetLastError() == cudaSuccess ? 0 : failed_launch("k_unpredict_seed / k_unpredict_angle", failed);
	}
	// way tiles (image stacks and video), every predictor but 2: the band pipeline
	static const int bands_on = getenv("LFM_B200_BANDS") ? atoi(getenv("LFM_B200_BANDS")) : 1;
	// (a single frame is a chain of tilesY / R bands, each ~R + UB_D + 10 steps behind the one above: one or two frames are
	// served faster by the cluster wavefront below, which puts 8 SMs on every frame)
	static const int bands_min = getenv("LFM_B200_BANDS_MIN") ? atoi(getenv("LFM_B200_BANDS_MIN")) : 3;
	if (bands_on && way == 0 && k != 2 && (int)count >= bands_min) {
		const int rcb = launch_unpredict_bands<0>(sym, out, W, H, T, k, (video && (z_start & 1u)) ? 1 : 0, z_start, z_step, count, st);
		if (rcb != 2) return rcb ? failed_launch("k_unpredict_bands", failed) : 0;
	}
	// remaining cases (way tiles, video, predictor 2 of tiles/angle): many frames -> one CTA per frame in shared memory;
	// few frames -> the cluster wavefront below (all SMs on one frame)
	// predictor 2 of the ways tiles / angle: below the first tile row every image column is an independent chain
	static const int cols_on = getenv("LFM_B200_COLS") ? atoi(getenv("LFM_B200_COLS")) : 1;
	const bool cols = cols_on && k == 2 && way != 2 && T <= 32 && H > 1 && (size_t)W * 4 <= (size_t)UG_MAX_SMEM;
	static const int strips_min = getenv("LFM_B200_STRIPS_MIN") ? atoi(getenv("LFM_B200_STRIPS_MIN")) : 128;
	if ((int)count >= strips_min && !cols) {
		const int rcs = way == 0 ? launch_unpredict_strips<0>(sym, out, W, H, T, k, video, z_start, z_step, count, st)
		              : way == 1 ? launch_unpredict_strips<1>(sym, out, W, H, T, k, video, z_start, z_step, count, st)
		                         : launch_unpredict_strips<2>(sym, out, W, H, T, k, video, z_start, z_step, count, st);
		if (rcs != 2) return rcs ? failed_launch("k_unpredict_strips", failed) : 0;
	}
	const uint64_t steps = (k == 2 && way != 2) ? (uint64_t)H : (uint64_t)(tilesX + tilesY + 2 * T);
	const uint64_t per_step = ((uint64_t)W * H + steps - 1) / steps;              // mean ready pixels per step and frame
	unsigned csz = 1;
	while (csz < 8 && (uint64_t)csz * UP_NT < per_step) csz <<= 1;                // about one pixel per thread per step
	cudaLaunchConfig_t cfg = {};
	cfg.gridDim = dim3(count * csz); cfg.blockDim = dim3(UP_NT); cfg.dynamicSmemBytes = 0; cfg.stream = st;
	cudaLaunchAttribute attr[1];
	attr[0].id = cudaLaunchAttributeClusterDimension;
	attr[0].val.clusterDim.x = csz; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
	cfg.attrs = attr; cfg.numAttrs = 1;
	if (cols) {
		const size_t smem0 = (size_t)W * 2 * 2;
		const size_t smem = (size_t)T * UC_NT * 2;
		if (way == 0) {
			cudaFuncSetAttribute(k_unpredict_row0<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem0);
			k_unpredict_row0<0><<<count, 32, smem0, st>>>(sym, out, W, H, T, video, z_start, z_step);
		} else {
			cudaFuncSetAttribute(k_unpredict_row0<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem0);
			k_unpredict_row0<1><<<count, 32, smem0, st>>>(sym, out, W, H, T, video, z_start, z_step);
		}
		if (cudaGetLastError() != cudaSuccess) return failed_launch("k_unpredict_row0", failed);
		for (uint32_t f0 = 0; f0 < count; f0 += 65535u) {          // frames in gridDim.y: at most 65535 per launch
			const dim3 grid((unsigned)((W + UC_NT - 1) / UC_NT), std::min(65535u, count - f0));
			if (way == 0) k_unpredict_cols2<0><<<grid, UC_NT, smem, st>>>(sym, out, W, H, T, video, z_start + f0 * z_step, z_step);
			else k_unpredict_cols2<1><<<grid, UC_NT, smem, st>>>(sym, out, W, H, T, video, z_start + f0 * z_step, z_step);
		}
		return cudaGetLastError() == cudaSuccess ? 0 : failed_launch("k_unpredict_cols2", failed);
	}
	return cudaLaunchKernelEx(&cfg, k_unpredict, sym, out, W, H, T, way, k, video, z_start, z_step, count, H) == cudaSuccess ? 0
	       : failed_launch("k_unpredict (cluster)", failed);
}

}  // namespace lfm
