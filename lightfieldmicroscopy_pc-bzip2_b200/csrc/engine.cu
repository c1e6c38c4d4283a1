// engine.cu -- per-GPU pipeline driver (see engine.h). Host code; all arithmetic runs in the kernels.
#include "engine.h"
#include "kernels.h"
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <map>
#include <mutex>
#include <memory>
#include <algorithm>

namespace lfm {

struct Totals { unsigned long long running; uint32_t err; uint32_t periodic; uint32_t overflow; uint32_t pad; };

// exclusive offsets of the batch's streams inside the payload (running base carried across batches); a stream is the
// bit-concatenation of the bzip2 blocks in its `nsub` records, padded to a byte
__global__ void k_offsets(const EncJob* __restrict__ jobs, uint32_t njobs, uint32_t nsub, Totals* tot, uint64_t* __restrict__ offs,
                          uint32_t* __restrict__ sizes, uint64_t payload_cap)
{
	__shared__ uint32_t red[64];
	__shared__ unsigned long long s_base;
	if (threadIdx.x == 0) s_base = tot->running;
	__syncthreads();
	uint32_t err = 0, per = 0;
	for (uint32_t j0 = 0; j0 < njobs; j0 += 1024) {
		uint32_t j = j0 + threadIdx.x;
		uint32_t v = 0;
		if (j < njobs) {
			uint32_t bits = 0;
			for (uint32_t k = 0; k < nsub; k++) {
				const EncJob& J = jobs[(size_t)j * nsub + k];
				err |= J.status; per += J.periodic;
				if (!(J.flags & kSubUnused)) bits += J.total_bits;
			}
			v = (bits + 7) / 8;
		}
		uint32_t total; uint32_t inc = block_scan_add<1024>(v, red, &total);
		unsigned long long base = s_base;
		if (j < njobs) { offs[j] = base + inc - v; sizes[j] = v; }
		__syncthreads();
		if (threadIdx.x == 0) s_base = base + total;
		__syncthreads();
	}
	if (err) atomicOr(&tot->err, err);
	if (per) atomicAdd(&tot->periodic, per);
	__syncthreads();
	if (threadIdx.x == 0) { tot->running = s_base; if (s_base > payload_cap) tot->overflow = 1; }
}

// copy each stream from its slot(s) to its final place (byte granular; destination is unaligned by nature)
__global__ void k_compact(const uint8_t* __restrict__ slots, uint32_t ocap, const EncJob* __restrict__ jobs, uint32_t nsub,
                          const uint64_t* __restrict__ offs, const uint32_t* __restrict__ sizes, uint8_t* __restrict__ payload,
                          uint64_t payload_cap)
{
	__shared__ uint32_t s_start[kMaxSub + 1];      // first stream bit of every bzip2 block
	const uint32_t job = blockIdx.x;
	const uint32_t n = sizes[job];
	const uint64_t o = offs[job];
	if (o + n > payload_cap) return;
	const uint8_t* src = slots + (size_t)job * nsub * ocap;
	uint8_t* dst = payload + o;
	uint32_t nu = 0;
	for (uint32_t k = 0; k < nsub; k++) nu += (jobs[(size_t)job * nsub + k].flags & kSubUnused) ? 0u : 1u;
	if (nu > 1) {
		// several bzip2 blocks: block k starts at stream bit s_start[k], anywhere inside a byte (bzip2 does not pad between
		// blocks, compress.c:603-676).  Every thread assembles whole output bytes from at most two blocks.
		if (threadIdx.x == 0) {
			uint32_t acc = 0;
			for (uint32_t k = 0; k < nu; k++) { s_start[k] = acc; acc += jobs[(size_t)job * nsub + k].total_bits; }
			s_start[nu] = acc;
		}
		__syncthreads();
		for (uint32_t P = threadIdx.x; P < n; P += blockDim.x) {
			const uint32_t bit = P * 8;
			uint32_t k = 0;
			while (k + 1 < nu && bit >= s_start[k + 1]) k++;
			uint32_t v = 0, have = 0;
			while (have < 8 && k < nu) {
				const uint32_t lb = bit + have - s_start[k], avail = s_start[k + 1] - (bit + have);      // unread bits of block k
				const uint8_t* sk = src + (size_t)k * ocap;
				const uint32_t two = ((uint32_t)sk[lb >> 3] << 8) | sk[(lb >> 3) + 1];
				const uint32_t take = min(8u - have, avail);
				const uint32_t bits = (two >> (16 - (lb & 7) - take)) & ((1u << take) - 1u);
				v |= bits << (8 - have - take);
				have += take; k++;
			}
			dst[P] = (uint8_t)v;
		}
		return;
	}
	// head bytes until dst is 4-aligned, then words assembled from the (4-aligned) source with a byte shift
	uint32_t head = (uint32_t)((4 - (o & 3)) & 3); if (head > n) head = n;
	if (threadIdx.x < head) dst[threadIdx.x] = src[threadIdx.x];
	const uint32_t nwords = (n - head) / 4;
	const uint32_t* s32 = reinterpret_cast<const uint32_t*>(src);
	uint32_t* d32 = reinterpret_cast<uint32_t*>(dst + head);
	const uint32_t sh = head * 8;
	for (uint32_t i = threadIdx.x; i < nwords; i += blockDim.x) {
		uint32_t a = s32[i], b = s32[i + 1];
		d32[i] = sh ? __funnelshift_r(a, b, sh) : a;
	}
	uint32_t done = head + nwords * 4;
	if (threadIdx.x < n - done) dst[done + threadIdx.x] = src[done + threadIdx.x];
}

__global__ void k_dec_status(const DecJob* __restrict__ jobs, uint32_t njobs, uint32_t* flag)
{
	uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
	if (j < njobs && jobs[j].status) atomicOr(flag, 1u << min(jobs[j].status, 31u));
}

// KLB_COMPRESSION_TYPE::NONE: a block's payload is its rows, x fastest, copied verbatim (src/klb_imageIO.cpp:146-183 gather,
// :207-210 "codec", :673-746 scatter).  One CTA per KLB block, one warp per row.  Payload positions come from the file on
// the read side and may be odd: bytes are moved one by one there.
__global__ void k_none_gather(const uint16_t* __restrict__ sym, Geom g, uint64_t first_block, const uint64_t* __restrict__ starts,
                              uint8_t* __restrict__ payload)
{
	uint32_t c0[5], ext[5];
	block_box(g, first_block + blockIdx.x, c0, ext);
	const uint32_t rows = ext[1] * ext[2] * ext[3] * ext[4], rowpx = ext[0];
	uint16_t* dst = reinterpret_cast<uint16_t*>(payload + starts[blockIdx.x]);       // starts are sums of even byte counts
	for (uint32_t r = warp_id(); r < rows; r += blockDim.x >> 5) {
		uint32_t y = r % ext[1], q = r / ext[1];
		uint32_t z = q % ext[2]; q /= ext[2];
		uint32_t c = q % ext[3], t = q / ext[3];
		const uint16_t* row = sym + (c0[0] + (uint64_t)(c0[1] + y) * g.stride[1] + (uint64_t)(c0[2] + z) * g.stride[2]
		                             + (uint64_t)(c0[3] + c) * g.stride[3] + (uint64_t)(c0[4] + t) * g.stride[4]);
		for (uint32_t x = lane_id(); x < rowpx; x += 32) dst[(size_t)r * rowpx + x] = row[x];
	}
}
__global__ void k_none_scatter(const uint8_t* __restrict__ payload, const uint64_t* __restrict__ begin, const uint64_t* __restrict__ block_ids,
                               uint16_t* __restrict__ sym, Geom g)
{
	uint32_t c0[5], ext[5];
	block_box(g, block_ids[blockIdx.x], c0, ext);
	const uint32_t rows = ext[1] * ext[2] * ext[3] * ext[4], rowpx = ext[0];
	const uint8_t* src = payload + begin[blockIdx.x];
	for (uint32_t r = warp_id(); r < rows; r += blockDim.x >> 5) {
		uint32_t y = r % ext[1], q = r / ext[1];
		uint32_t z = q % ext[2]; q /= ext[2];
		uint32_t c = q % ext[3], t = q / ext[3];
		uint16_t* row = sym + (c0[0] + (uint64_t)(c0[1] + y) * g.stride[1] + (uint64_t)(c0[2] + z) * g.stride[2]
		                       + (uint64_t)(c0[3] + c) * g.stride[3] + (uint64_t)(c0[4] + t) * g.stride[4]);
		const uint8_t* s2 = src + ((size_t)r * rowpx) * 2;
		for (uint32_t x = lane_id(); x < rowpx; x += 32) row[x] = (uint16_t)(s2[2 * x] | ((uint32_t)s2[2 * x + 1] << 8));
	}
}

// ------------------------------------------------------------------------------------------------
static std::mutex g_mu;
static std::map<int, std::unique_ptr<Engine>> g_engines;

Engine& Engine::for_device(int device)
{
	std::lock_guard<std::mutex> lk(g_mu);
	auto it = g_engines.find(device);
	if (it == g_engines.end()) it = g_engines.emplace(device, std::unique_ptr<Engine>(new Engine(device))).first;
	return *it->second;
}

Engine::Engine(int device) : device_(device)
{
	cudaSetDevice(device_);
	cudaDeviceProp p;
	if (cudaGetDeviceProperties(&p, device_) == cudaSuccess) sm_count_ = p.multiProcessorCount;
	cudaStream_t st; cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking);
	stream_ = st;
	for (int i = 0; i < 5 + kMaxGroups; i++) { cudaEvent_t e; cudaEventCreateWithFlags(&e, i < 4 ? cudaEventDefault : cudaEventDisableTiming); ev_[i] = e; }
}

void* Engine::aux_stream(int i)
{
	while ((int)aux_.size() <= i) { cudaStream_t s2; cudaStreamCreateWithFlags(&s2, cudaStreamNonBlocking); aux_.push_back(s2); }
	return aux_[i];
}

// Groups a batch of nj KLB blocks is cut into, each running its kernel pipeline on a forked stream so that the stages of
// different groups overlap.  Measured on B200 (profiles/r1_07): compress +5 % on one 2048^2 frame (484 blocks, 3 groups),
// +13 % on 968 blocks of 147 KB (4 groups), nothing on decode -- k_bwt's 1024-thread CTAs own a whole SM, so little can
// run beside them -- and the per-stage event times stop being separable.  Off unless LFM_B200_GROUPS=n asks for it.
int Engine::groups_for(uint32_t nj) const
{
	static const int forced = getenv("LFM_B200_GROUPS") ? atoi(getenv("LFM_B200_GROUPS")) : 0;
	if (forced <= 1) return 1;
	return std::min<int>(std::min<int>(forced, kMaxGroups), (int)std::max<uint32_t>(1, nj / (uint32_t)sm_count_));
}

void* Engine::pooled_event(size_t i)
{
	while (ev_pool_.size() <= i) { cudaEvent_t e; cudaEventCreate(&e); ev_pool_.push_back(e); }
	return ev_pool_[i];
}

static double elapsed_or_zero(void* a, void* b)
{
	float ms = 0.f;
	if (cudaEventElapsedTime(&ms, (cudaEvent_t)a, (cudaEvent_t)b) != cudaSuccess) { cudaGetLastError(); return 0.0; }
	return ms;
}
double Engine::last_predict_ms() { return elapsed_or_zero(ev_[0], ev_[1]); }
double Engine::last_unpredict_ms() { return elapsed_or_zero(ev_[2], ev_[3]); }

int Engine::check(const char* what)
{
	cudaError_t e = cudaGetLastError();
	if (e != cudaSuccess) {
		err_ = std::string(what) + ": " + cudaGetErrorString(e);
		fprintf(stderr, "lfm_b200: CUDA error in %s\n", err_.c_str());
		return LFM_ERR_CUDA;
	}
	return LFM_OK;
}

int Engine::reserve(Buf& b, size_t bytes)
{
	if (b.cap >= bytes) return LFM_OK;
	if (b.p) cudaFree(b.p);
	b.p = nullptr; b.cap = 0;
	size_t want = bytes + bytes / 8 + 256;
	if (cudaMalloc(&b.p, want) != cudaSuccess) {
		cudaGetLastError();
		if (cudaMalloc(&b.p, bytes) != cudaSuccess) { err_ = "cudaMalloc failed"; cudaGetLastError(); return LFM_ERR_CUDA; }
		want = bytes;
	}
	b.cap = want;
	return LFM_OK;
}

void* Engine::pinned(size_t bytes, int slot)
{
	slot &= 1;
	if (pin_cap_[slot] >= bytes) return pin_[slot];
	if (pin_[slot]) cudaFreeHost(pin_[slot]);
	pin_[slot] = nullptr; pin_cap_[slot] = 0;
	size_t want = bytes + bytes / 4 + 4096;
	if (cudaHostAlloc(&pin_[slot], want, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); pin_[slot] = nullptr; return nullptr; }
	pin_cap_[slot] = want;
	return pin_[slot];
}

static inline uint32_t round16(uint64_t v) { return (uint32_t)((v + 15) & ~(uint64_t)15); }

static Geom make_geom(const StackDesc& s)
{
	Geom g;
	uint64_t st = 1;
	for (int i = 0; i < 5; i++) {
		g.xyzct[i] = s.xyzct[i]; g.bs[i] = s.blockSize[i];
		g.nb[i] = (uint32_t)std::ceil((float)s.xyzct[i] / (float)s.blockSize[i]);   // klb_imageHeader.cpp:77-85
		g.stride[i] = st; st *= s.xyzct[i];
	}
	return g;
}

// Slot geometry.  A KLB block is one bzip2 stream of `nsub` bzip2 blocks at most: every block but the last holds
// nblockMAX .. nblockMAX + 4 run-length coded bytes (bzlib.c: nblockMAX = 100000 * level - 19, a block is closed by the
// record that reaches it), so nsub = floor(maxn / nblockMAX) + 1 and a sub-slot holds nblockMAX + 10 bytes.
struct EncSizes { uint32_t cap, mcap, selcap, ocap, nsub, nblock_max; int level; int text_in_smem; };
static void slot_sizes(uint64_t subn, EncSizes& z)         // subn: most run-length coded bytes one block can hold
{
	z.cap = round16(subn + 8) + 16;
	z.mcap = round16((uint64_t)z.cap + 2);
	z.selcap = round16((uint64_t)z.mcap / kGSize + 2);
	z.ocap = round16(subn + subn / 8 + subn / 16 + 8192);
	z.text_in_smem = bwt_smem_bytes(z.cap, 1) <= 227 * 1024;
}
static int enc_sizes(const StackDesc& s, EncSizes& z)
{
	uint64_t blockBytes = 2;
	for (int i = 0; i < 5; i++) blockBytes *= s.blockSize[i];
	z.level = (int)std::min<uint64_t>(9, (blockBytes + 99999) / 100000);     // klb_imageIO.cpp:108
	const uint64_t maxn = blockBytes + blockBytes / 4 + 1;                     // RLE1 worst case: 4 -> 5 bytes
	z.nblock_max = (uint32_t)(100000 * z.level - 19);
	const uint64_t nsub = maxn / z.nblock_max + 1;
	if (nsub > (uint64_t)kMaxSub || blockBytes > 0x7fffffffull / 2) return LFM_ERR_UNSUPPORTED;
	z.nsub = (uint32_t)nsub;
	slot_sizes(std::min<uint64_t>(maxn, (uint64_t)z.nblock_max + 10), z);
	return LFM_OK;
}
// a standalone stream (bz2_compress): any number of blocks at the caller's level, one record per block
static void stream_sizes(int level, EncSizes& z)
{
	z.level = level; z.nsub = 1;
	z.nblock_max = (uint32_t)(100000 * level - 19);
	slot_sizes((uint64_t)z.nblock_max + 10, z);
}

// ------------------------------------------------------------------------------------------------ selection
int Engine::select_mode(const uint16_t* d_frame0, const StackDesc& s, float entropy[8], int* winner)
{
	cudaSetDevice(device_);
	cudaStream_t st = (cudaStream_t)stream_;
	const int W = (int)s.xyzct[0], H = (int)s.xyzct[1];
	const uint64_t fpx = (uint64_t)W * H;
	const uint32_t chunk_px = 450000;                                          // klb_imageIO.cpp:2032
	const uint32_t nchunks = (uint32_t)((fpx + chunk_px - 1) / chunk_px);
	const uint32_t sstride = round16((uint64_t)chunk_px * 2 + 2);
	int rc;
	if ((rc = reserve(sel_cand_, 7 * fpx * 2))) return rc;
	if ((rc = reserve(sel_sorted_, (size_t)8 * nchunks * sstride))) return rc;
	if ((rc = reserve(sel_hist_, (size_t)8 * nchunks * 65536 * 4))) return rc;
	const size_t e_words = ((size_t)8 * nchunks + 63) & ~(size_t)63;                 // entropies, then the sort's per-part digit counts
	if ((rc = reserve(sel_e_, (e_words + select_scratch_words(8, nchunks)) * 4))) return rc;
	const uint16_t* cands[8];
	cands[0] = d_frame0;
	for (int k = 1; k < 8; k++) {
		uint16_t* c = (uint16_t*)sel_cand_.p + (size_t)(k - 1) * fpx;
		launch_predict_fwd(d_frame0, c, W, H, s.Nnum, s.way, k, 0, 0, 1, st);
		cands[k] = c;
	}
	launch_select(cands, 8, fpx, chunk_px, nchunks, (uint8_t*)sel_sorted_.p, sstride, (uint32_t*)sel_hist_.p, (float*)sel_e_.p, (uint32_t*)sel_e_.p + e_words, st);
	std::vector<float> e((size_t)8 * nchunks);
	cudaMemcpyAsync(e.data(), sel_e_.p, e.size() * 4, cudaMemcpyDeviceToHost, st);
	cudaStreamSynchronize(st);
	if ((rc = check("select_mode"))) return rc;
	int best = 0;
	for (int id = 0; id < 8; id++) {
		float acc = 0.f;
		for (uint32_t c = 0; c < nchunks; c++) acc += e[(size_t)id * nchunks + c];     // `*entropy += ...` per chunk
		entropy[id] = id ? acc : (float)(acc * 0.96);                                  // klb_imageIO.cpp:2087-2090
		if (id && entropy[id] <= entropy[best]) best = id;                             // std::map: equal keys -> last wins
	}
	*winner = best;
	return LFM_OK;
}

int Engine::predict(const uint16_t* d_img, uint16_t* d_sym, const StackDesc& s, int predictor, int video, uint32_t z0, uint32_t nz)
{
	cudaSetDevice(device_);
	if (predictor < 1 || predictor > 7 || s.way < 0 || s.way > 2) return LFM_ERR_UNSUPPORTED;
	if (video && s.way != 0) return LFM_ERR_UNSUPPORTED;     // the reference's z!=0 angle/space kernels are not invertible
	cudaEventRecord((cudaEvent_t)ev_[0], (cudaStream_t)stream_);
	launch_predict_fwd(d_img, d_sym, (int)s.xyzct[0], (int)s.xyzct[1], s.Nnum, s.way, predictor, video, z0, nz, (cudaStream_t)stream_);
	cudaEventRecord((cudaEvent_t)ev_[1], (cudaStream_t)stream_);
	return check("predict");
}

int Engine::unpredict(const uint16_t* d_sym, uint16_t* d_out, const StackDesc& s, int predictor, int video, uint32_t z0, uint32_t nz)
{
	cudaSetDevice(device_);
	if (predictor < 1 || predictor > 7 || s.way < 0 || s.way > 2) return LFM_ERR_UNSUPPORTED;
	if (video && s.way != 0) return LFM_ERR_UNSUPPORTED;
	cudaStream_t st = (cudaStream_t)stream_;
	const int W = (int)s.xyzct[0], H = (int)s.xyzct[1];
	// test aid: a wrong wavefront order must not be masked by stale, accidentally correct data in a recycled buffer
	static const bool poison = getenv("LFM_B200_DEBUG_POISON") != nullptr;
	if (poison) cudaMemsetAsync(d_out + (size_t)z0 * W * H, 0xAB, (size_t)nz * W * H * 2, st);
	int bad = 0;
	const char* failed = "?";
	cudaEventRecord((cudaEvent_t)ev_[2], st);
	if (!video) bad |= launch_unpredict(d_sym, d_out, W, H, s.Nnum, s.way, predictor, 0, z0, 1, nz, sm_count_, st, &failed);
	else {
		// odd frames need the decoded even frame before them: evens first, then odds (z0 must be even)
		uint32_t first_even = z0 + (z0 & 1), first_odd = z0 + 1 - (z0 & 1);
		uint32_t n_even = first_even < z0 + nz ? (z0 + nz - first_even + 1) / 2 : 0;
		uint32_t n_odd = first_odd < z0 + nz ? (z0 + nz - first_odd + 1) / 2 : 0;
		bad |= launch_unpredict(d_sym, d_out, W, H, s.Nnum, s.way, predictor, 1, first_even, 2, n_even, sm_count_, st, &failed);
		if (!bad) bad |= launch_unpredict(d_sym, d_out, W, H, s.Nnum, s.way, predictor, 1, first_odd, 2, n_odd, sm_count_, st, &failed);
	}
	cudaEventRecord((cudaEvent_t)ev_[3], st);
	if (bad) { cudaGetLastError(); err_ = std::string("inverse predictor: launch of ") + failed + " failed"; return LFM_ERR_CUDA; }
	return check("unpredict");
}

int Engine::roi_gather(const uint16_t* d_frames, const StackDesc& s, const uint32_t lb[5], const uint32_t ub[5], uint16_t* d_out)
{
	cudaSetDevice(device_);
	launch_roi_gather(d_frames, s.xyzct, lb, ub, d_out, sm_count_, (cudaStream_t)stream_);
	return check("roi_gather");
}

// ------------------------------------------------------------------------------------------------ codec NONE
static uint64_t host_block_bytes(const Geom& g, uint64_t id)
{
	uint64_t n = 2;
	for (int i = 0; i < 5; i++) {
		const uint64_t c = id % g.nb[i]; id /= g.nb[i];
		n *= std::min<uint64_t>(g.bs[i], g.xyzct[i] - c * g.bs[i]);
	}
	return n;
}

int Engine::compress_blocks_none(const uint16_t* d_sym, const StackDesc& s, uint64_t first, uint64_t count,
                                 uint32_t* sizes_out, const uint8_t** d_payload, uint64_t* payload_bytes, CompressStats* stt)
{
	cudaStream_t st = (cudaStream_t)stream_;
	const Geom g = make_geom(s);
	if (count == 0) { *d_payload = nullptr; *payload_bytes = 0; return LFM_OK; }
	std::vector<uint64_t> starts(count);
	uint64_t acc = 0;
	for (uint64_t i = 0; i < count; i++) {
		const uint64_t n = host_block_bytes(g, first + i);
		if (n > 0xffffffffull) { err_ = "KLB block larger than 4 GB"; return LFM_ERR_UNSUPPORTED; }
		starts[i] = acc; sizes_out[i] = (uint32_t)n; acc += n;
	}
	int rc;
	if ((rc = reserve(payload2_[pay_sel_], acc + 16))) return rc;
	if ((rc = reserve(offs_, count * 8))) return rc;
	cudaMemcpyAsync(offs_.p, starts.data(), count * 8, cudaMemcpyHostToDevice, st);
	for (uint64_t b0 = 0; b0 < count; b0 += 0x40000000ull) {
		const uint32_t nj = (uint32_t)std::min<uint64_t>(0x40000000ull, count - b0);
		k_none_gather<<<nj, 256, 0, st>>>(d_sym, g, first + b0, (const uint64_t*)offs_.p + b0, (uint8_t*)payload2_[pay_sel_].p);
		if (stt) stt->launches++;
	}
	cudaStreamSynchronize(st);                                  // `starts` is pageable host memory
	if ((rc = check("compress_blocks_none"))) return rc;
	*d_payload = (const uint8_t*)payload2_[pay_sel_].p; *payload_bytes = acc;
	return LFM_OK;
}

int Engine::decompress_blocks_none(const uint8_t* d_payload, const uint64_t* begin, const uint64_t* end, const uint64_t* block_ids,
                                   uint64_t count, uint16_t* d_sym, const StackDesc& s, DecompressStats* stt)
{
	cudaStream_t st = (cudaStream_t)stream_;
	const Geom g = make_geom(s);
	if (count == 0) return LFM_OK;
	for (uint64_t i = 0; i < count; i++)
		if (end[i] - begin[i] != host_block_bytes(g, block_ids[i])) { err_ = "uncompressed block has the wrong size"; return LFM_ERR_BZIP; }
	int rc;
	if ((rc = reserve(dbegin_, count * 8))) return rc;
	if ((rc = reserve(dids_, count * 8))) return rc;
	cudaMemcpyAsync(dbegin_.p, begin, count * 8, cudaMemcpyHostToDevice, st);
	cudaMemcpyAsync(dids_.p, block_ids, count * 8, cudaMemcpyHostToDevice, st);
	for (uint64_t b0 = 0; b0 < count; b0 += 0x40000000ull) {
		const uint32_t nj = (uint32_t)std::min<uint64_t>(0x40000000ull, count - b0);
		k_none_scatter<<<nj, 256, 0, st>>>(d_payload, (const uint64_t*)dbegin_.p + b0, (const uint64_t*)dids_.p + b0, d_sym, g);
		if (stt) stt->launches++;
	}
	cudaStreamSynchronize(st);
	return check("decompress_blocks_none");
}

// ------------------------------------------------------------------------------------------------ compress
int Engine::compress_blocks(const uint16_t* d_sym, const StackDesc& s, uint64_t first, uint64_t count,
                            uint32_t* sizes_out, const uint8_t** d_payload, uint64_t* payload_bytes, CompressStats* stt)
{
	cudaSetDevice(device_);
	if (s.codec == 0) return compress_blocks_none(d_sym, s, first, count, sizes_out, d_payload, payload_bytes, stt);
	cudaStream_t st = (cudaStream_t)stream_;
	const Geom g = make_geom(s);
	EncSizes z;
	if (enc_sizes(s, z)) { err_ = "KLB block too large: more than kMaxSub bzip2 blocks per stream"; return LFM_ERR_UNSUPPORTED; }
	if (count == 0) { *d_payload = nullptr; *payload_bytes = 0; return LFM_OK; }
	// per KLB block: nsub records / sub-slots (one per possible bzip2 block of its stream; 1 for the default block shapes)
	const size_t per_job = ((size_t)z.cap * 3 + (size_t)z.mcap * 2 + (size_t)z.selcap * 2 + z.ocap + sizeof(EncJob)) * z.nsub;
	uint64_t B = std::min<uint64_t>(count, std::max<uint64_t>(1, ((size_t)6 << 30) / per_job));
	B = std::min<uint64_t>(B, 16384);
	const uint64_t BS = B * z.nsub;                                            // job records per batch
	const int grid = (int)std::min<uint64_t>(BS, (uint64_t)sm_count_ * bwt_ctas_per_sm(z.cap, z.text_in_smem));   // resident k_bwt CTAs
	uint64_t blockBytes = 2; for (int i = 0; i < 5; i++) blockBytes *= s.blockSize[i];
	uint64_t pcap = std::min<uint64_t>(count * (uint64_t)z.ocap * z.nsub, count * blockBytes + count * blockBytes / 3 + count * 1024 * z.nsub + (1 << 20));
	int rc;
	if ((rc = reserve(jobs_, BS * sizeof(EncJob)))) return rc;
	if ((rc = reserve(txt_, BS * z.cap))) return rc;
	if ((rc = reserve(bwt_, BS * z.cap))) return rc;
	if ((rc = reserve(rank_, BS * z.cap))) return rc;
	if ((rc = reserve(mtfv_, BS * (size_t)z.mcap * 2))) return rc;
	if ((rc = reserve(sel_, BS * (size_t)z.selcap * 2))) return rc;
	if ((rc = reserve(out_, BS * (size_t)z.ocap + 16))) return rc;
	const int Gres = groups_for((uint32_t)B);                                  // forked groups need a scratch region each
	if ((rc = reserve(scratch_, (size_t)Gres * grid * bwt_scratch_elems_per_cta(z.cap) * 4))) return rc;
	if ((rc = reserve(payload2_[pay_sel_], pcap + 16))) return rc;
	if ((rc = reserve(sizes_, count * 4))) return rc;
	if ((rc = reserve(offs_, B * 8 + sizeof(Totals)))) return rc;
	Totals* tot = (Totals*)((uint8_t*)offs_.p + B * 8);
	cudaMemsetAsync(tot, 0, sizeof(Totals), st);

	std::vector<cudaEvent_t> evs;
	uint64_t launches = 0;
	for (uint64_t b0 = 0; b0 < count; b0 += B) {
		const uint32_t nj = (uint32_t)std::min<uint64_t>(B, count - b0);
		const uint32_t ns = nj * z.nsub;                                       // job records of this batch
		// optional (groups_for): the batch cut into G groups whose four-kernel pipelines run on forked streams
		const int G = groups_for(nj);
		if (G > 1) cudaEventRecord((cudaEvent_t)ev_[4], st);
		for (int gi = 0; gi < G; gi++) {
			const uint32_t j0 = (uint32_t)((uint64_t)nj * gi / G), j1 = (uint32_t)((uint64_t)nj * (gi + 1) / G);
			const uint32_t gj = j1 - j0, gs = gj * z.nsub;
			const size_t r0 = (size_t)j0 * z.nsub;                                // first job record of the group
			cudaStream_t sg = G > 1 ? (cudaStream_t)aux_stream(gi) : st;
			if (G > 1) cudaStreamWaitEvent(sg, (cudaEvent_t)ev_[4], 0);
			auto markg = [&]() { if (stt) { cudaEvent_t e = (cudaEvent_t)pooled_event(evs.size()); cudaEventRecord(e, sg); evs.push_back(e); } };
			EncJob* gjobs = (EncJob*)jobs_.p + r0;
			uint8_t* gtxt = (uint8_t*)txt_.p + r0 * z.cap; uint8_t* gbwt = (uint8_t*)bwt_.p + r0 * z.cap; uint8_t* grank = (uint8_t*)rank_.p + r0 * z.cap;
			uint16_t* gmtfv = (uint16_t*)mtfv_.p + r0 * z.mcap;
			markg();
			launch_rle1(d_sym, g, first + b0 + j0, gj, gtxt, gbwt, z.cap, z.nsub, (uint32_t)blockBytes, z.nblock_max, gjobs, sg);
			markg();
			launch_bwt(gtxt, z.cap, gjobs, gs, gbwt, (uint32_t*)scratch_.p + (size_t)gi * grid * bwt_scratch_elems_per_cta(z.cap),
			           (int)std::min<uint32_t>(gs, (uint32_t)grid), z.text_in_smem, sg);
			markg();
			launch_mtf(gbwt, grank, z.cap, gjobs, gs, gmtfv, z.mcap, sg);
			markg();
			launch_huff_pack(gmtfv, z.mcap, gjobs, gs, (uint8_t*)sel_.p + r0 * (size_t)z.selcap * 2, z.selcap, (uint8_t*)out_.p + r0 * z.ocap, z.ocap, z.level, sg);
			markg();
			if (G > 1) { cudaEvent_t je = (cudaEvent_t)ev_[5 + gi]; cudaEventRecord(je, sg); cudaStreamWaitEvent(st, je, 0); }
		}
		k_offsets<<<1, 1024, 0, st>>>((EncJob*)jobs_.p, nj, z.nsub, tot, (uint64_t*)offs_.p, (uint32_t*)sizes_.p + b0, pcap);
		k_compact<<<nj, 256, 0, st>>>((uint8_t*)out_.p, z.ocap, (EncJob*)jobs_.p, z.nsub, (uint64_t*)offs_.p, (uint32_t*)sizes_.p + b0, (uint8_t*)payload2_[pay_sel_].p, pcap);
		launches += 4 * G + 2;
		last_njobs_ = ns;
	}
	last_cap_ = z.cap; last_mcap_ = z.mcap;
	Totals h;
	cudaMemcpyAsync(&h, tot, sizeof(Totals), cudaMemcpyDeviceToHost, st);
	cudaMemcpyAsync(sizes_out, sizes_.p, count * 4, cudaMemcpyDeviceToHost, st);
	cudaStreamSynchronize(st);
	if ((rc = check("compress_blocks"))) return rc;
	if (stt) {
		for (size_t i = 0; i + 4 < evs.size(); i += 5) {
			float ms;
			cudaEventElapsedTime(&ms, evs[i], evs[i + 1]); stt->ms_rle += ms;
			cudaEventElapsedTime(&ms, evs[i + 1], evs[i + 2]); stt->ms_bwt += ms;
			cudaEventElapsedTime(&ms, evs[i + 2], evs[i + 3]); stt->ms_mtf += ms;
			cudaEventElapsedTime(&ms, evs[i + 3], evs[i + 4]); stt->ms_huff += ms;
		}
		stt->launches += launches;
		stt->periodic_blocks += h.periodic;
	}
	if (h.overflow) { err_ = "payload buffer overflow"; return LFM_ERR_BZIP; }
	if (h.err & 4u) { err_ = "a KLB block needs more bzip2 blocks than the engine reserves per stream"; return LFM_ERR_UNSUPPORTED; }
	if (h.err) { err_ = "block encoder reported an error"; return LFM_ERR_BZIP; }
	*d_payload = (const uint8_t*)payload2_[pay_sel_].p;
	*payload_bytes = h.running;
	return LFM_OK;
}

int Engine::fetch_encode_trace(EncodeTrace& t)
{
	cudaSetDevice(device_);
	cudaStream_t st = (cudaStream_t)stream_;
	t.cap = last_cap_; t.mcap = last_mcap_; t.njobs = last_njobs_;
	t.jobs.resize((size_t)t.njobs * sizeof(EncJob));
	t.txt.resize((size_t)t.njobs * t.cap); t.bwt.resize((size_t)t.njobs * t.cap); t.mtfv.resize((size_t)t.njobs * t.mcap);
	cudaMemcpyAsync(t.jobs.data(), jobs_.p, t.jobs.size(), cudaMemcpyDeviceToHost, st);
	cudaMemcpyAsync(t.txt.data(), txt_.p, t.txt.size(), cudaMemcpyDeviceToHost, st);
	cudaMemcpyAsync(t.bwt.data(), bwt_.p, t.bwt.size(), cudaMemcpyDeviceToHost, st);
	cudaMemcpyAsync(t.mtfv.data(), mtfv_.p, t.mtfv.size() * 2, cudaMemcpyDeviceToHost, st);
	cudaStreamSynchronize(st);
	return check("fetch_encode_trace");
}

// ------------------------------------------------------------------------------------------------ standalone bzip2 stream
uint8_t* Engine::bz2_staging(size_t bytes)
{
	cudaSetDevice(device_);
	return reserve(sz_in_, bytes + 16) ? nullptr : (uint8_t*)sz_in_.p;
}

// One stream of any number of bzip2 blocks (bz_stream.cu): the RLE1 structure of the whole input and the block boundaries first,
// then the blocks in batches through the stages of the KLB path, each batch's bits assembled into the stream before the next one
// reuses the slots.  Workspace beyond the input and the stream: the slots of one batch (as compress_blocks), a record per tile of
// kSzTile input bytes, a record per block and the record-end bitmap (one bit per run-length coded byte).
int Engine::bz2_compress(const uint8_t* d_src, uint64_t n, int level, const uint8_t** d_out, uint64_t* out_size, CompressStats* stt)
{
	cudaSetDevice(device_);
	cudaStream_t st = (cudaStream_t)stream_;
	if (level < 1 || level > 9) { err_ = "level must be 1..9"; return LFM_ERR_OPEN; }
	if (n >= (1ull << 32)) { err_ = "input of 2^32 bytes or more"; return LFM_ERR_UNSUPPORTED; }
	EncSizes z; stream_sizes(level, z);
	const uint32_t n32 = (uint32_t)n, nt = sz_tiles(n);
	const uint64_t max_rle = n + n / 4 + 1;                                    // RLE1 worst case: 4 -> 5 bytes
	const uint32_t max_blocks = (uint32_t)(max_rle / z.nblock_max + 2);
	const uint64_t bitmap_words = (max_rle + 31) / 32 + 2;
	const uint64_t out_cap = (n + n / 64 + 1024ull * max_blocks + 4096) & ~3ull;
	const size_t per_job = (size_t)z.cap * 3 + (size_t)z.mcap * 2 + (size_t)z.selcap * 2 + z.ocap + sizeof(EncJob);
	uint32_t B = (uint32_t)std::min<uint64_t>(max_blocks, std::max<uint64_t>(1, ((size_t)6 << 30) / per_job));
	B = std::min<uint32_t>(B, 16384);
	const int grid = (int)std::min<uint64_t>(B, (uint64_t)sm_count_ * bwt_ctas_per_sm(z.cap, z.text_in_smem));
	int rc;
	if ((rc = reserve(sz_tiles_, (size_t)nt * 5 * 4 + ((size_t)nt + 1) * 8 + 64))) return rc;
	if ((rc = reserve(sz_bits_, bitmap_words * 4))) return rc;
	if ((rc = reserve(sz_blocks_, ((size_t)max_blocks + 1) * 12 + ((size_t)B + 1) * 8 + 64))) return rc;
	if ((rc = reserve(sz_out_, out_cap + 16))) return rc;
	if ((rc = reserve(jobs_, (size_t)B * sizeof(EncJob)))) return rc;
	if ((rc = reserve(txt_, (size_t)B * z.cap))) return rc;
	if ((rc = reserve(bwt_, (size_t)B * z.cap))) return rc;
	if ((rc = reserve(rank_, (size_t)B * z.cap))) return rc;
	if ((rc = reserve(mtfv_, (size_t)B * z.mcap * 2))) return rc;
	if ((rc = reserve(sel_, (size_t)B * z.selcap * 2))) return rc;
	if ((rc = reserve(out_, (size_t)B * z.ocap + 16))) return rc;
	if ((rc = reserve(scratch_, (size_t)grid * bwt_scratch_elems_per_cta(z.cap) * 4))) return rc;
	uint64_t* tobase = (uint64_t*)sz_tiles_.p;                                 // [nt + 1]
	uint32_t* t32 = (uint32_t*)(tobase + nt + 1);
	uint32_t *tfirst = t32, *tlast = t32 + nt, *topen = t32 + 2 * (size_t)nt, *tnext = t32 + 3 * (size_t)nt, *tcount = t32 + 4 * (size_t)nt;
	uint64_t* bout = (uint64_t*)sz_blocks_.p;                                  // [max_blocks + 1]
	uint64_t* bitoff = bout + max_blocks + 1;                                  // [B + 1]
	SzRun* run = (SzRun*)(bitoff + B + 1);
	uint32_t* nbp = (uint32_t*)(run + 1);
	uint32_t* combined = nbp + 1;
	uint32_t* bin = combined + 1;                                              // [max_blocks + 1]
	cudaMemsetAsync(run, 0, sizeof(SzRun) + 8 + ((size_t)max_blocks + 1) * 4, st);
	cudaMemsetAsync(sz_out_.p, 0, out_cap, st);

	std::vector<cudaEvent_t> evs;
	auto mark = [&]() { if (stt) { cudaEvent_t e = (cudaEvent_t)pooled_event(evs.size()); cudaEventRecord(e, st); evs.push_back(e); } };
	uint64_t launches = 0;
	mark();
	uint32_t nb = 1;
	if (n > 0) {
		launch_sz_runs(d_src, n32, tfirst, tlast, topen, tnext, st);
		launch_sz_count(d_src, n32, topen, tnext, tcount, tobase, st);
		launch_sz_chain(d_src, n32, topen, tnext, tobase, (uint32_t*)sz_bits_.p, bitmap_words, z.nblock_max, max_blocks, bout, nbp, st);
		launches += 6;
		cudaMemcpyAsync(&nb, nbp, 4, cudaMemcpyDeviceToHost, st);
		cudaStreamSynchronize(st);
		if ((rc = check("bz2_compress structure"))) return rc;
		cudaMemcpyAsync(bin + nb, &n32, 4, cudaMemcpyHostToDevice, st);          // bin[0] = 0 from the memset
		launch_sz_locate(d_src, n32, topen, tnext, tobase, bout, bin, nb, st);
		launches += nb > 1 ? 1 : 0;
	} else {
		cudaMemsetAsync(bout, 0, 16, st);                                      // one empty block: header and trailer only
	}
	mark();
	for (uint32_t k0 = 0; k0 < nb; k0 += B) {
		const uint32_t nj = std::min<uint32_t>(B, nb - k0);
		EncJob* jobs = (EncJob*)jobs_.p;
		mark();
		launch_sz_emit(d_src, bin, bout, k0, nj, nb, (uint8_t*)txt_.p, z.cap, jobs, combined, st);
		mark();
		launch_bwt((uint8_t*)txt_.p, z.cap, jobs, nj, (uint8_t*)bwt_.p, (uint32_t*)scratch_.p, (int)std::min<uint32_t>(nj, (uint32_t)grid), z.text_in_smem, st);
		mark();
		launch_mtf((uint8_t*)bwt_.p, (uint8_t*)rank_.p, z.cap, jobs, nj, (uint16_t*)mtfv_.p, z.mcap, st);
		mark();
		launch_huff_pack((uint16_t*)mtfv_.p, z.mcap, jobs, nj, (uint8_t*)sel_.p, z.selcap, (uint8_t*)out_.p, z.ocap, level, st);
		launch_sz_assemble(jobs, nj, (uint8_t*)out_.p, z.ocap, bitoff, run, (uint8_t*)sz_out_.p, out_cap, sm_count_, st);
		mark();
		launches += 6 + (k0 + nj == nb ? 1 : 0);
	}
	SzRun h;
	cudaMemcpyAsync(&h, run, sizeof(h), cudaMemcpyDeviceToHost, st);
	cudaStreamSynchronize(st);
	if ((rc = check("bz2_compress"))) return rc;
	if (stt) {
		stt->ms_rle += elapsed_or_zero(evs[0], evs[1]);
		for (size_t i = 2; i + 4 < evs.size(); i += 5) {
			stt->ms_rle += elapsed_or_zero(evs[i], evs[i + 1]);
			stt->ms_bwt += elapsed_or_zero(evs[i + 1], evs[i + 2]);
			stt->ms_mtf += elapsed_or_zero(evs[i + 2], evs[i + 3]);
			stt->ms_huff += elapsed_or_zero(evs[i + 3], evs[i + 4]);          // Huffman coding + stream assembly
		}
		stt->launches += launches;
	}
	if (h.err) { err_ = "block encoder reported an error"; return LFM_ERR_BZIP; }
	const uint64_t bytes = (h.bits + 7) / 8;
	if (bytes > out_cap) { err_ = "stream buffer overflow"; return LFM_ERR_BZIP; }
	if (bytes >= (1ull << 32)) { err_ = "compressed stream of 2^32 bytes or more"; return LFM_ERR_UNSUPPORTED; }
	*d_out = (const uint8_t*)sz_out_.p;
	*out_size = bytes;
	return LFM_OK;
}

// Any .bz2 data (bz_stream.cu): candidate magics at every bit, every candidate decoded speculatively as a block (Huffman stage
// only, in batches) to learn where it ends, the chain walk keeps the real blocks; then the real blocks in batches through
// k_huff_decode / k_imtf / k_inv_bwt and the un-RLE1 length pass, a prefix sum of the lengths, the capacity check, and the replay
// into the flat output (the batches are decoded again when there is more than one).
int Engine::bz2_decompress(const void* src, uint64_t n, bool src_on_host, uint8_t* d_dst, uint64_t capacity, const uint8_t** d_out,
                           uint64_t* out_size, DecompressStats* stt)
{
	cudaSetDevice(device_);
	cudaStream_t st = (cudaStream_t)stream_;
	if (n == 0) { err_ = "empty input"; return LFM_ERR_BZIP; }
	if (n >= (1ull << 32)) { err_ = "input of 2^32 bytes or more"; return LFM_ERR_UNSUPPORTED; }
	EncSizes z; stream_sizes(9, z);                                            // slots for the largest block
	const uint32_t nt = sz_tiles(n);
	const size_t per_job = (size_t)z.cap * 2 + (size_t)z.mcap * 2 + sizeof(DecJob) + 24;
	const uint32_t B = (uint32_t)std::min<uint64_t>(16384, std::max<uint64_t>(1, ((size_t)6 << 30) / per_job));
	int rc;
	if ((rc = reserve(dz_in_, n + 64))) return rc;
	if ((rc = reserve(sz_tiles_, (size_t)nt * 4 + ((size_t)nt + 1) * 8 + 64))) return rc;
	uint8_t* in = (uint8_t*)dz_in_.p;
	cudaMemcpyAsync(in, src, n, src_on_host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, st);
	cudaMemsetAsync(in + n, 0, 64, st);
	uint64_t* tbase = (uint64_t*)sz_tiles_.p;
	uint32_t* tcount = (uint32_t*)(tbase + nt + 1);
	std::vector<cudaEvent_t> evs;
	auto mark = [&]() { if (stt) { cudaEvent_t e = (cudaEvent_t)pooled_event(evs.size()); cudaEventRecord(e, st); evs.push_back(e); } };
	mark();
	launch_bz_magic(in, n, 0, tcount, tbase, nullptr, nullptr, st);
	uint64_t nc64 = 0;
	cudaMemcpyAsync(&nc64, tbase + nt, 8, cudaMemcpyDeviceToHost, st);
	cudaStreamSynchronize(st);
	if ((rc = check("bz2_decompress magic scan"))) return rc;
	if (nc64 == 0) { err_ = "no bzip2 block or end-of-stream magic"; return LFM_ERR_BZIP; }
	const uint32_t nc = (uint32_t)nc64;
	// candidate records: cbit, cend, bbit (u64); ccrc, succ, blev, blen (u32); ceos (u8); boff (u64, nc + 1); dn, res
	if ((rc = reserve(dz_cand_, (size_t)nc * (3 * 8 + 4 * 4 + 1) + ((size_t)nc + 1) * 8 + 256))) return rc;
	uint64_t* cbit = (uint64_t*)dz_cand_.p; uint64_t* cend = cbit + nc; uint64_t* bbit = cend + nc; uint64_t* boff = bbit + nc;
	uint64_t* dn = boff + nc + 1;
	uint32_t* res = (uint32_t*)(dn + 1);
	uint32_t* ccrc = res + 4; uint32_t* succ = ccrc + nc; uint32_t* blev = succ + nc; uint32_t* blen = blev + nc;
	uint8_t* ceos = (uint8_t*)(blen + nc);
	cudaMemcpyAsync(dn, &n, 8, cudaMemcpyHostToDevice, st);
	launch_bz_magic(in, n, 1, tcount, tbase, cbit, ceos, st);
	const uint32_t grid = (uint32_t)std::min<uint64_t>(B, (uint64_t)sm_count_ * inv_bwt_ctas_per_sm(z.cap));
	if ((rc = reserve(djobs_, (size_t)B * sizeof(DecJob) + 16))) return rc;
	if ((rc = reserve(bwt_, (size_t)B * z.cap))) return rc;
	if ((rc = reserve(txt_, (size_t)B * z.cap))) return rc;
	if ((rc = reserve(mtfv_, (size_t)B * z.mcap * 2))) return rc;
	if ((rc = reserve(tt_, inv_bwt_scratch_elems(grid, z.cap) * 4))) return rc;
	DecJob* jobs = (DecJob*)djobs_.p;
	uint32_t* flag = (uint32_t*)(jobs + B);
	cudaMemsetAsync(flag, 0, 4, st);
	uint64_t launches = 2;
	mark();
	// ---- speculative pass: where does every candidate block end
	for (uint32_t c0 = 0; c0 < nc; c0 += B) {
		const uint32_t nj = std::min(B, nc - c0);
		if (launch_decode(in, cbit + c0, dn, nj, 1, jobs, (uint16_t*)mtfv_.p, z.mcap, (uint8_t*)txt_.p, (uint8_t*)bwt_.p, z.cap, z.selcap, st,
		                  nullptr, cend + c0, ccrc + c0, nullptr, false)) { err_ = "decoder launch failed"; return LFM_ERR_UNSUPPORTED; }
		launches++;
	}
	launch_bz_chain(in, n, cbit, ceos, nc, cend, ccrc, succ, bbit, blev, res, st);
	launches += 2;
	uint32_t hres[2] = { 0, 0 };
	cudaMemcpyAsync(hres, res, 8, cudaMemcpyDeviceToHost, st);
	cudaStreamSynchronize(st);
	if ((rc = check("bz2_decompress chain"))) return rc;
	mark();
	if (hres[1]) { err_ = "corrupt bzip2 data: the blocks do not chain from the stream header to the end of the input"; return LFM_ERR_BZIP; }
	const uint32_t nb = hres[0];
	const uint32_t nbatch = (nb + B - 1) / B;
	auto decode_batch = [&](uint32_t k0, uint32_t nj) -> int {
		if (launch_decode(in, bbit + k0, dn, nj, 1, jobs, (uint16_t*)mtfv_.p, z.mcap, (uint8_t*)txt_.p, (uint8_t*)bwt_.p, z.cap, z.selcap, st,
		                  nullptr, cend + k0, ccrc + k0, blev + k0, true)) { err_ = "decoder launch failed"; return LFM_ERR_UNSUPPORTED; }
		launch_inv_bwt((uint8_t*)bwt_.p, z.cap, jobs, nj, (uint32_t*)tt_.p, (uint8_t*)txt_.p, (int)std::min(nj, grid), st);
		launches += 3;
		return LFM_OK;
	};
	// ---- blocks: decode, lengths
	for (uint32_t k0 = 0; k0 < nb; k0 += B) {
		const uint32_t nj = std::min(B, nb - k0);
		if ((rc = decode_batch(k0, nj))) return rc;
		launch_unrle_len((uint8_t*)txt_.p, z.cap, jobs, nj, blen + k0, st);
		k_dec_status<<<(nj + 255) / 256, 256, 0, st>>>(jobs, nj, flag);
		launches += 2;
	}
	launch_scan_u32(nb, blen, boff, st);
	launches++;
	uint64_t total = 0; uint32_t hflag = 0;
	cudaMemcpyAsync(&total, boff + nb, 8, cudaMemcpyDeviceToHost, st);
	cudaMemcpyAsync(&hflag, flag, 4, cudaMemcpyDeviceToHost, st);
	cudaStreamSynchronize(st);
	if ((rc = check("bz2_decompress blocks"))) return rc;
	if (hflag) { char m[96]; snprintf(m, sizeof(m), "corrupt bzip2 block (decoder status mask 0x%x)", hflag); err_ = m; return LFM_ERR_BZIP; }
	*out_size = total;
	if (total >= (1ull << 32)) { err_ = "decompressed data of 2^32 bytes or more"; return LFM_ERR_UNSUPPORTED; }
	if (total > capacity) { err_ = "destination buffer too small"; return LFM_ERR_CREATE; }
	uint8_t* out = d_dst;
	if (!out) { if ((rc = reserve(dz_out_, total + 16))) return rc; out = (uint8_t*)dz_out_.p; }
	// ---- replay into the flat output, block CRCs checked
	for (uint32_t k0 = 0; k0 < nb; k0 += B) {
		const uint32_t nj = std::min(B, nb - k0);
		if (nbatch > 1 && (rc = decode_batch(k0, nj))) return rc;
		launch_unrle_flat((uint8_t*)txt_.p, z.cap, jobs, nj, boff + k0, out, st);
		k_dec_status<<<(nj + 255) / 256, 256, 0, st>>>(jobs, nj, flag);
		launches += 2;
	}
	mark();
	cudaMemcpyAsync(&hflag, flag, 4, cudaMemcpyDeviceToHost, st);
	cudaStreamSynchronize(st);
	if ((rc = check("bz2_decompress"))) return rc;
	if (stt) {
		stt->ms_decode += elapsed_or_zero(evs[0], evs[2]);                    // magic scan, speculative decode, chain walk
		stt->ms_unrle += elapsed_or_zero(evs[2], evs[3]);                     // blocks: decode, inverse BWT, un-RLE1, CRCs
		stt->launches += launches;
	}
	if (hflag) { char m[96]; snprintf(m, sizeof(m), "block CRC mismatch (decoder status mask 0x%x)", hflag); err_ = m; return LFM_ERR_BZIP; }
	*d_out = out;
	return LFM_OK;
}

// ------------------------------------------------------------------------------------------------ decompress
int Engine::decompress_blocks(const uint8_t* d_payload, const uint64_t* begin, const uint64_t* end, const uint64_t* block_ids,
                              uint64_t count, uint16_t* d_sym, const StackDesc& s, DecompressStats* stt)
{
	cudaSetDevice(device_);
	if (s.codec == 0) return decompress_blocks_none(d_payload, begin, end, block_ids, count, d_sym, s, stt);
	cudaStream_t st = (cudaStream_t)stream_;
	if (count == 0) return LFM_OK;
	const Geom g = make_geom(s);
	EncSizes z;
	if (enc_sizes(s, z)) { err_ = "KLB block too large: more than kMaxSub bzip2 blocks per stream"; return LFM_ERR_UNSUPPORTED; }
	uint64_t blockBytes = 2; for (int i = 0; i < 5; i++) blockBytes *= s.blockSize[i];
	const size_t per_job = ((size_t)z.cap * 2 + (size_t)z.mcap * 2 + sizeof(DecJob) + 24) * z.nsub;
	uint64_t B = std::min<uint64_t>(count, std::max<uint64_t>(1, ((size_t)6 << 30) / per_job));
	B = std::min<uint64_t>(B, 32768);
	const uint64_t BS = B * z.nsub;                                            // job records per batch
	const int grid = (int)std::min<uint64_t>(BS, (uint64_t)sm_count_ * inv_bwt_ctas_per_sm(z.cap));   // resident k_inv_bwt CTAs
	int rc;
	if ((rc = reserve(djobs_, BS * sizeof(DecJob) + 16))) return rc;
	if ((rc = reserve(bwt_, BS * z.cap))) return rc;
	if ((rc = reserve(txt_, BS * z.cap))) return rc;
	if ((rc = reserve(mtfv_, BS * (size_t)z.mcap * 2))) return rc;
	if ((rc = reserve(tt_, (size_t)groups_for((uint32_t)B) * inv_bwt_scratch_elems(grid, z.cap) * 4))) return rc;
	if ((rc = reserve(dbegin_, count * 8))) return rc;
	if ((rc = reserve(dend_, count * 8))) return rc;
	if ((rc = reserve(dids_, count * 8))) return rc;
	uint32_t* flag = (uint32_t*)((uint8_t*)djobs_.p + BS * sizeof(DecJob));
	cudaMemsetAsync(flag, 0, 4, st);
	cudaMemcpyAsync(dbegin_.p, begin, count * 8, cudaMemcpyHostToDevice, st);
	cudaMemcpyAsync(dend_.p, end, count * 8, cudaMemcpyHostToDevice, st);
	cudaMemcpyAsync(dids_.p, block_ids, count * 8, cudaMemcpyHostToDevice, st);
	std::vector<cudaEvent_t> evs;
	uint64_t launches = 0;
	for (uint64_t b0 = 0; b0 < count; b0 += B) {
		const uint32_t nj = (uint32_t)std::min<uint64_t>(B, count - b0);
		const int G = groups_for(nj);                                          // see compress_blocks
		if (G > 1) cudaEventRecord((cudaEvent_t)ev_[4], st);
		for (int gi = 0; gi < G; gi++) {
			const uint32_t j0 = (uint32_t)((uint64_t)nj * gi / G), j1 = (uint32_t)((uint64_t)nj * (gi + 1) / G);
			const uint32_t gj = j1 - j0, gs = gj * z.nsub;
			const size_t r0 = (size_t)j0 * z.nsub;
			cudaStream_t sg = G > 1 ? (cudaStream_t)aux_stream(gi) : st;
			if (G > 1) cudaStreamWaitEvent(sg, (cudaEvent_t)ev_[4], 0);
			auto markg = [&]() { if (stt) { cudaEvent_t e = (cudaEvent_t)pooled_event(evs.size()); cudaEventRecord(e, sg); evs.push_back(e); } };
			DecJob* gjobs = (DecJob*)djobs_.p + r0;
			uint8_t* gtxt = (uint8_t*)txt_.p + r0 * z.cap; uint8_t* gbwt = (uint8_t*)bwt_.p + r0 * z.cap;
			uint16_t* gmtfv = (uint16_t*)mtfv_.p + r0 * z.mcap;
			markg();
			cudaEvent_t mid = nullptr;
			if (stt) { mid = (cudaEvent_t)pooled_event(evs.size()); evs.push_back(mid); }      // recorded between k_huff_decode and k_imtf
			if (launch_decode(d_payload, (uint64_t*)dbegin_.p + b0 + j0, (uint64_t*)dend_.p + b0 + j0, gj, z.nsub, gjobs, gmtfv, z.mcap,
			                  gtxt, gbwt, z.cap, z.selcap, sg, mid)) { err_ = "decoder launch failed"; return LFM_ERR_UNSUPPORTED; }
			markg();
			const int ggrid = (int)std::min<uint32_t>(gs, (uint32_t)grid);
			launch_inv_bwt(gbwt, z.cap, gjobs, gs, (uint32_t*)tt_.p + (size_t)gi * inv_bwt_scratch_elems(grid, z.cap), gtxt, ggrid, sg);
			markg();
			launch_unrle(gtxt, gbwt, z.cap, z.nsub, (uint32_t)blockBytes, gjobs, gj, d_sym, g, (uint64_t*)dids_.p + b0 + j0, sg);
			k_dec_status<<<(gs + 255) / 256, 256, 0, sg>>>(gjobs, gs, flag);
			markg();
			if (G > 1) { cudaEvent_t je = (cudaEvent_t)ev_[5 + gi]; cudaEventRecord(je, sg); cudaStreamWaitEvent(st, je, 0); }
		}
		launches += 5 * G;
	}
	uint32_t hflag = 0;
	cudaMemcpyAsync(&hflag, flag, 4, cudaMemcpyDeviceToHost, st);
	cudaStreamSynchronize(st);
	if ((rc = check("decompress_blocks"))) return rc;
	if (stt) {
		for (size_t i = 0; i + 4 < evs.size(); i += 5) {
			float ms;
			cudaEventElapsedTime(&ms, evs[i], evs[i + 1]); stt->ms_decode += ms;
			cudaEventElapsedTime(&ms, evs[i + 1], evs[i + 2]); stt->ms_imtf += ms;
			cudaEventElapsedTime(&ms, evs[i + 2], evs[i + 3]); stt->ms_ibwt += ms;
			cudaEventElapsedTime(&ms, evs[i + 3], evs[i + 4]); stt->ms_unrle += ms;
		}
		stt->launches += launches;
	}
	if (hflag) {
		char m[96]; snprintf(m, sizeof(m), "block decoder status mask 0x%x", hflag); err_ = m;
		return (hflag & (1u << 4)) ? LFM_ERR_UNSUPPORTED : LFM_ERR_BZIP;
	}
	return LFM_OK;
}

}  // namespace lfm
