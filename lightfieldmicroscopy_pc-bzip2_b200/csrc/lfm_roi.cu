// lfm_roi.cu -- k_roi_gather: the box lb..ub of decoded frames -> a dense [t][c][z][y][x] buffer in device memory.
//
// An ROI read into device memory ends here instead of in one 2-D copy per frame: an XZ or YZ plane through a few hundred frames
// would otherwise be a few hundred copies of a few rows each.  One launch covers every frame of the box.  The output rows (x
// runs of the box) are numbered y fastest, then z, c, t -- the order of the dense output -- and one warp copies one row: 16-byte
// loads and stores where the source row and its place in the output have the same offset modulo 16 bytes, 2-byte accesses for
// the head and tail around the vectors and for rows whose offsets differ.  HBM bound: 2 x box bytes of traffic.
#include <algorithm>
#include "kernels.h"

namespace lfm {

__device__ __forceinline__ void roi_copy_row(const uint16_t* __restrict__ s, uint16_t* __restrict__ d, uint32_t n, uint32_t lane)
{
	const uint32_t sa = (uint32_t)reinterpret_cast<uintptr_t>(s) & 15u, da = (uint32_t)reinterpret_cast<uintptr_t>(d) & 15u;
	const uint32_t head = sa == da ? min(n, ((16u - sa) & 15u) >> 1) : n;          // pixels before the first 16-byte boundary
	for (uint32_t i = lane; i < head; i += 32) d[i] = s[i];
	if (head == n) return;
	const uint32_t nv = (n - head) >> 3;
	const uint4* __restrict__ sv = reinterpret_cast<const uint4*>(s + head);
	uint4* __restrict__ dv = reinterpret_cast<uint4*>(d + head);
	for (uint32_t i = lane; i < nv; i += 32) dv[i] = sv[i];
	for (uint32_t i = head + nv * 8 + lane; i < n; i += 32) d[i] = s[i];
}

// frames: absolute frame indexing (frame f of the stack at frames + f * W * H); box origin x0..t0, extent rx x ny x nz x nc x nt
__global__ void __launch_bounds__(256) k_roi_gather(const uint16_t* __restrict__ frames, uint32_t W, uint32_t H, uint32_t Z, uint32_t Cn,
                                                    uint32_t x0, uint32_t y0, uint32_t z0, uint32_t c0, uint32_t t0,
                                                    uint32_t rx, uint32_t ny, uint32_t nz, uint32_t nc, uint64_t rows,
                                                    uint16_t* __restrict__ out)
{
	const uint32_t lane = threadIdx.x & 31u;
	const uint64_t fpx = (uint64_t)W * H, nwarps = (uint64_t)gridDim.x * (blockDim.x >> 5);
	for (uint64_t r = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < rows; r += nwarps) {
		uint64_t q = r;
		const uint32_t y = (uint32_t)(q % ny); q /= ny;
		const uint32_t z = (uint32_t)(q % nz); q /= nz;
		const uint32_t c = (uint32_t)(q % nc); q /= nc;
		const uint64_t f = (uint64_t)(z0 + z) + (uint64_t)Z * ((uint64_t)(c0 + c) + (uint64_t)Cn * (t0 + q));
		roi_copy_row(frames + f * fpx + (uint64_t)(y0 + y) * W + x0, out + r * rx, rx, lane);
	}
}

void launch_roi_gather(const uint16_t* frames, const uint32_t xyzct[5], const uint32_t lb[5], const uint32_t ub[5], uint16_t* out,
                       int sm_count, cudaStream_t st)
{
	const uint32_t rx = ub[0] - lb[0] + 1, ny = ub[1] - lb[1] + 1, nz = ub[2] - lb[2] + 1, nc = ub[3] - lb[3] + 1, nt = ub[4] - lb[4] + 1;
	const uint64_t rows = (uint64_t)ny * nz * nc * nt;
	// 8 warps a CTA, at most 8 CTAs per SM resident at a time: enough 16-byte loads in flight to keep HBM busy
	const uint64_t ctas = std::min<uint64_t>((rows + 7) / 8, (uint64_t)sm_count * 8);
	k_roi_gather<<<(unsigned)ctas, 256, 0, st>>>(frames, xyzct[0], xyzct[1], xyzct[2], xyzct[3], lb[0], lb[1], lb[2], lb[3], lb[4],
	                                              rx, ny, nz, nc, rows, out);
}

}  // namespace lfm
