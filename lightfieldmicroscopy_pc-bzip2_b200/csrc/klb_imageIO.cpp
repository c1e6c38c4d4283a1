// klb_imageIO.cpp -- host orchestration of the .lfm compress / decompress path on B200 GPUs.
//
// Mirrors the observable behaviour of the reference's klb_imageIO::writeImage / readImage / readImageFull
// (src/klb_imageIO.cpp:2248-2492, :2614-2782): same header handling, same predictor request rules, same block
// partition and blockOffset table, same return codes.  What differs is where the work runs:
//   * predictor, mode selection and the whole bzip2 block codec run as CUDA kernels (csrc/*.cu) instead of
//     CUDA predictor + std::thread bzip2;
//   * KLB blocks are sharded over the configured GPUs by contiguous z-slabs (block ids are x fastest, so a slab is a
//     contiguous block-id range and a contiguous payload range); no collective on the data path -- the host does the
//     inclusive prefix sum of the block sizes that becomes header.blockOffset[] (cf. blockWriter, :1145-1225);
//   * there is no CPU fallback: without a CUDA device every call fails with code 6.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <fcntl.h>
#include <unistd.h>
#include <sys/stat.h>
#include <sys/mman.h>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <new>
#include <thread>
#include <vector>
#include <cuda_runtime.h>
#include "klb_imageIO.h"
#include "lfm_b200.h"
#include "engine.h"

using namespace lfm;

// ------------------------------------------------------------------------------------------------ settings / stats
namespace {
struct Settings {
	int way = -1;            // -1: not initialised yet
	int first_device = 0;
	int ndev = -1;
} g_set;
// statistics / error text of the last call are per calling thread; the shard worker threads of a call report through their
// ShardOut / per-shard slots and the calling thread merges them after the join.
thread_local lfm_stats g_stats;
thread_local std::string g_err;
// The engines (one per GPU: stream, workspace, pinned staging) are shared by every klb_imageIO object of the process, so the
// compute entry points of the library are serialised; calls stay synchronous as in the reference (SURVEY 8b "Threading").
std::recursive_mutex g_api_mu;
#define LFM_API_LOCK() std::lock_guard<std::recursive_mutex> lfm_api_lock_(g_api_mu); DeviceGuard lfm_device_guard_
// the caller's current CUDA device is restored when a call returns (a framework above us keeps its own notion of it)
#define LFM_CATCH catch (const std::bad_alloc&) { g_err = "out of host memory"; return LFM_ERR_CREATE; } \
                  catch (const std::exception& ex_) { g_err = ex_.what(); return LFM_ERR_BZIP; }
struct DeviceGuard {
	int prev = -1;
	DeviceGuard() { if (cudaGetDevice(&prev) != cudaSuccess) { cudaGetLastError(); prev = -1; } }
	~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

int env_int(const char* name, int dflt) { const char* v = getenv(name); return v && *v ? atoi(v) : dflt; }
int current_way() { if (g_set.way < 0) { int w = env_int("LFM_PREDICTOR_WAY", LFM_PREDICTOR_WAY_DEFAULT); g_set.way = (w >= 0 && w <= 2) ? w : 0; } return g_set.way; }
int visible_devices() { int n = 0; if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; } return n; }
int current_ndev()
{
	if (g_set.ndev < 0) g_set.ndev = std::max(1, env_int("LFM_B200_GPUS", 1));
	int vis = visible_devices();
	return std::max(0, std::min(g_set.ndev, vis - g_set.first_device));
}
double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

struct FrameSource {              // contiguous stack or one pointer per XY slice
	const uint16_t* base = nullptr;
	const uint16_t* const* slices = nullptr;
	bool device = false;          // base is a contiguous stack in device memory of the first device: nothing is uploaded
	const uint16_t* frame(uint64_t f, uint64_t fpx) const { return slices ? slices[f] : base + f * fpx; }
};
// Where decoded pixels go when they stay on the GPU: the caller's device buffer of `capacity` bytes (dense box of the read)
struct DeviceSink {
	void* d_out = nullptr;
	uint64_t capacity = 0;
	uint64_t* out_bytes = nullptr;
};

struct Layout {                   // derived block / frame geometry
	uint32_t nb[5];
	uint64_t Nb, blocksPerSlab, nSlabs, F, fpx;
};
Layout make_layout(const klb_image_header& h)
{
	Layout L;
	L.Nb = 1;
	for (int d = 0; d < 5; d++) { L.nb[d] = (uint32_t)std::ceil((float)h.xyzct[d] / (float)h.blockSize[d]); L.Nb *= L.nb[d]; }
	L.blocksPerSlab = (uint64_t)L.nb[0] * L.nb[1];
	L.nSlabs = (uint64_t)L.nb[2] * L.nb[3] * L.nb[4];
	L.F = (uint64_t)h.xyzct[2] * h.xyzct[3] * h.xyzct[4];
	L.fpx = (uint64_t)h.xyzct[0] * h.xyzct[1];
	return L;
}
// flattened frame range [f0, f1] touched by slabs [s0, s1)
void slab_frames(const klb_image_header& h, const Layout& L, uint64_t s0, uint64_t s1, uint64_t& f0, uint64_t& f1)
{
	f0 = ~0ull; f1 = 0;
	for (uint64_t s = s0; s < s1; s++) {
		uint64_t bz = s % L.nb[2], r = s / L.nb[2], bc = r % L.nb[3], bt = r / L.nb[3];
		uint64_t z0 = bz * h.blockSize[2], z1 = std::min<uint64_t>(h.xyzct[2], z0 + h.blockSize[2]) - 1;
		uint64_t c0 = bc * h.blockSize[3], c1 = std::min<uint64_t>(h.xyzct[3], c0 + h.blockSize[3]) - 1;
		uint64_t t0 = bt * h.blockSize[4], t1 = std::min<uint64_t>(h.xyzct[4], t0 + h.blockSize[4]) - 1;
		f0 = std::min(f0, z0 + h.xyzct[2] * (c0 + (uint64_t)h.xyzct[3] * t0));
		f1 = std::max(f1, z1 + h.xyzct[2] * (c1 + (uint64_t)h.xyzct[3] * t1));
	}
}
// Slab boundaries of D shards: shard d owns slabs [cut[d], cut[d+1]) -- a contiguous block-id and payload range.  With
// pair_frames (video stack + predictor: an odd frame is predicted from the even frame before it, `video_bit & z`) a shard
// never starts on an odd frame, so the writer and the reader of a shard have everything they need inside it.
std::vector<uint64_t> shard_cuts(const klb_image_header& h, const Layout& L, int D, bool pair_frames)
{
	std::vector<uint64_t> cut(D + 1);
	for (int d = 0; d <= D; d++) {
		uint64_t s = L.nSlabs * (uint64_t)d / (uint64_t)D;
		if (d > 0) s = std::max(s, cut[d - 1]);
		if (pair_frames && d < D) {
			for (; s < L.nSlabs; s++) { uint64_t f0, f1; slab_frames(h, L, s, s + 1, f0, f1); if (!(f0 & 1)) break; }
		}
		cut[d] = d == D ? L.nSlabs : s;
	}
	return cut;
}
StackDesc make_desc(const klb_image_header& h, int way)
{
	StackDesc s;
	for (int d = 0; d < 5; d++) { s.xyzct[d] = h.xyzct[d]; s.blockSize[d] = h.blockSize[d]; }
	s.Nnum = h.Nnum ? h.Nnum : 1; s.way = way;
	s.codec = h.compressionType == KLB_COMPRESSION_TYPE::NONE ? 0 : 1;
	return s;
}
int validate(const klb_image_header& h, bool writing)
{
	if (h.compressionType != KLB_COMPRESSION_TYPE::BZIP2 && h.compressionType != KLB_COMPRESSION_TYPE::NONE) {
		if (h.compressionType == KLB_COMPRESSION_TYPE::ZLIB) {
			std::cout << "ERROR: lfm_b200: ZLIB block payloads (src/klb_imageIO.cpp:222-252) are not " << (writing ? "written" : "decoded")
			          << " by the GPU engine; supported KLB_COMPRESSION_TYPE values: BZIP2 (1) and NONE (0)" << std::endl;
			return LFM_ERR_UNSUPPORTED;
		}
		std::cout << "ERROR: workerfunc: compression type not implemented" << std::endl;
		return writing ? LFM_ERR_CREATE : LFM_ERR_OPEN;
	}
	if (h.getBytesPerPixel() != 2) {
		std::cout << "ERROR: lfm_b200: only 16-bit pixels are supported (the reference's predictor path reinterprets everything as uint16)" << std::endl;
		return LFM_ERR_UNSUPPORTED;
	}
	for (int d = 0; d < 5; d++) if (h.xyzct[d] == 0 || h.blockSize[d] == 0) return LFM_ERR_BZIP;
	return LFM_OK;
}

// a caller's buffer for the device-resident file calls: device or managed memory on the first device of lfmSetDevices, holding
// whole 16-bit pixels (code 3 otherwise)
int check_device_ptr(const void* p, const char* what)
{
	const int dev = Engine::for_device(g_set.first_device).device();
	cudaPointerAttributes a;
	if (!p || ((uintptr_t)p & 1) || cudaPointerGetAttributes(&a, p) != cudaSuccess) {
		cudaGetLastError(); g_err = std::string(what) + " is not a CUDA pointer to 16-bit pixels"; return LFM_ERR_OPEN;
	}
	if (a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) { g_err = std::string(what) + " is not device memory"; return LFM_ERR_OPEN; }
	if (a.device != dev) { g_err = std::string(what) + " is not on the first device of lfmSetDevices"; return LFM_ERR_OPEN; }
	return LFM_OK;
}

struct DevMem {                   // RAII device allocation
	void* p = nullptr;
	~DevMem() { if (p) cudaFree(p); }
	int alloc(size_t n) { if (cudaMalloc(&p, n ? n : 1) != cudaSuccess) { cudaGetLastError(); p = nullptr; return LFM_ERR_CUDA; } return 0; }
};

// ------------------------------------------------------------------------------------------------ pageable host memory
// Callers of the reference API hand in malloc'ed (pageable) stacks.  A plain cudaMemcpy of such memory runs at ~5 GB/s (the
// driver stages it through small internal buffers); here large copies go through four pinned staging buffers of the engine,
// filled / drained by a few host threads while the previous chunk crosses PCIe.  Pinned or registered memory (bench.py's e2e
// buffers) takes the direct path.
bool is_pageable(const void* p)
{
	cudaPointerAttributes a;
	if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return true; }
	return a.type == cudaMemoryTypeUnregistered;
}
// a few persistent host threads for the staging copies (thread start-up per call would cost more than a small copy)
class CopyPool {
public:
	// never destroyed: the workers wait on the condition variables for the life of the process (destroying a condition
	// variable with waiters blocks in pthread_cond_destroy at exit)
	static CopyPool& get() { static CopyPool* p = new CopyPool; return *p; }
	// workers beside the calling thread: the host cores this process may count on (one rank per GPU under torchrun: the
	// box's cores divided by LOCAL_WORLD_SIZE), at least 3, at most 7
	static int workers()
	{
		static const int n = [] {
			const int hw = (int)std::thread::hardware_concurrency();
			const int ranks = std::max(1, env_int("LOCAL_WORLD_SIZE", 1));
			const int forced = env_int("LFM_B200_COPY_THREADS", 0);
			return forced > 0 ? std::min(forced, 32) - 1 : std::min(7, std::max(3, hw / ranks - 1));
		}();
		return n;
	}
	// run f(0..parts-1): part 0 on the calling thread, the others on the workers; returns when all are done
	template <class F> void run(int parts, F f)
	{
		std::unique_lock<std::mutex> lk(mu_);
		// one batch at a time.  The pool is busy until its caller has finished part 0 as well: "no part pending" alone would let a
		// second caller (the upload, download and file threads of the slab pipelines run side by side) install its batch while
		// the first one is still inside f(0), and the first caller's clean-up would then drop parts of the second batch
		caller_.wait(lk, [&] { return !busy_; });
		busy_ = true;
		task_ = [&f](int i) { f(i); };
		nparts_ = parts; next_ = 1; pending_ = parts - 1;
		lk.unlock();
		work_.notify_all();
		f(0);
		lk.lock();
		caller_.wait(lk, [&] { return pending_ == 0; });
		nparts_ = 0; next_ = 0; busy_ = false;
		lk.unlock();
		caller_.notify_all();
	}
private:
	CopyPool() { for (int i = 0; i < workers(); i++) std::thread([this] { loop(); }).detach(); }
	void loop()
	{
		std::unique_lock<std::mutex> lk(mu_);
		for (;;) {
			work_.wait(lk, [&] { return next_ < nparts_; });
			const int i = next_++;
			lk.unlock();
			task_(i);
			lk.lock();
			if (--pending_ == 0) caller_.notify_all();
		}
	}
	std::mutex mu_;
	std::condition_variable work_, caller_;
	std::function<void(int)> task_;
	int nparts_ = 0, next_ = 0, pending_ = 0;
	bool busy_ = false;
};
void par_memcpy(void* dst, const void* src, size_t n)
{
	const int nt = CopyPool::workers() + 1;
	if (n < ((size_t)512 << 10)) { memcpy(dst, src, n); return; }
	const size_t part = ((n + nt - 1) / nt + 63) & ~(size_t)63;          // ceil: floor(n / nt) rounded to 64 can leave the last n mod nt bytes uncopied
	CopyPool::get().run(nt, [=](int i) {
		const size_t o = std::min(n, part * (size_t)i), len = std::min(n, part * (size_t)(i + 1)) - o;
		if (len) memcpy((uint8_t*)dst + o, (const uint8_t*)src + o, len);
	});
}
// file I/O of a staging buffer split over the copy pool (a single pwrite / pread of a tmpfs or page-cache file is a
// single-threaded memcpy: ~13 GB/s measured on the B200 box, tools/pcie_probe.py)
static int write_all(int fd, const void* p, size_t n, uint64_t at)
{
	size_t done = 0;
	while (done < n) {
		const ssize_t w = pwrite(fd, (const uint8_t*)p + done, n - done, (off_t)(at + done));
		if (w <= 0) return LFM_ERR_CREATE;
		done += (size_t)w;
	}
	return LFM_OK;
}
static int read_all(int fd, void* p, size_t n, uint64_t at)
{
	size_t done = 0;
	while (done < n) {
		const ssize_t got = pread(fd, (uint8_t*)p + done, n - done, (off_t)(at + done));
		if (got <= 0) return LFM_ERR_BZIP;
		done += (size_t)got;
	}
	return LFM_OK;
}
template <class IO> static int par_io(size_t n, IO io)          // io(offset, length) -> rc, on 4 KB aligned parts
{
	const int nt = CopyPool::workers() + 1;
	if (n < ((size_t)1 << 20)) return io((size_t)0, n);
	const size_t part = ((n + nt - 1) / nt + 4095) & ~(size_t)4095;
	std::atomic<int> rc(LFM_OK);
	CopyPool::get().run(nt, [&](int i) {
		const size_t o = std::min(n, part * (size_t)i), len = std::min(n, part * (size_t)(i + 1)) - o;
		if (len) { const int r = io(o, len); if (r) rc.store(r); }
	});
	return rc.load();
}
static int par_pread(int fd, uint8_t* buf, size_t n, uint64_t at) { return par_io(n, [=](size_t o, size_t len) { return read_all(fd, buf + o, len, at + o); }); }
constexpr size_t kStageChunk = (size_t)8 << 20;
constexpr int kStageBufs = 4;
// pageable <-> device copies of at least 2 MB are staged: big ones in 8 MB chunks, a single frame in 2 MB chunks so that the
// host copy of chunk i+1 overlaps the DMA of chunk i
constexpr size_t kStageMin = (size_t)2 << 20;
inline size_t stage_chunk(size_t bytes)
{
	static const size_t small = (size_t)std::min(8 << 10, std::max(256, env_int("LFM_B200_STAGE_KB", 2 << 10))) << 10;     // test knob
	return bytes >= ((size_t)64 << 20) ? kStageChunk : small;
}

void h2d_staged(Engine& e, void* dst, const void* src, size_t bytes, cudaStream_t st)
{
	uint8_t* pin = (bytes >= kStageMin && is_pageable(src)) ? (uint8_t*)e.pinned(kStageBufs * kStageChunk, 0) : nullptr;
	if (!pin) { cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st); return; }
	const size_t CH = stage_chunk(bytes);
	cudaEvent_t ev[kStageBufs];
	for (auto& x : ev) cudaEventCreateWithFlags(&x, cudaEventDisableTiming);
	size_t i = 0;
	for (size_t off = 0; off < bytes; off += CH, i++) {
		const size_t len = std::min(CH, bytes - off);
		uint8_t* buf = pin + (i % kStageBufs) * CH;
		if (i >= (size_t)kStageBufs) cudaEventSynchronize(ev[i % kStageBufs]);
		par_memcpy(buf, (const uint8_t*)src + off, len);
		cudaMemcpyAsync((uint8_t*)dst + off, buf, len, cudaMemcpyHostToDevice, st);
		cudaEventRecord(ev[i % kStageBufs], st);
	}
	cudaStreamSynchronize(st);                                   // the staging buffers are shared: free them before anyone else asks
	for (auto& x : ev) cudaEventDestroy(x);
}

void d2h_staged(Engine& e, void* dst, const void* src, size_t bytes, cudaStream_t st)
{
	uint8_t* pin = (bytes >= kStageMin && is_pageable(dst)) ? (uint8_t*)e.pinned(kStageBufs * kStageChunk, 1) : nullptr;
	if (!pin) { cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st); return; }
	const size_t CH = stage_chunk(bytes);
	cudaEvent_t ev[kStageBufs];
	for (auto& x : ev) cudaEventCreateWithFlags(&x, cudaEventDisableTiming);
	const size_t nch = (bytes + CH - 1) / CH;
	auto issue = [&](size_t i) {
		const size_t off = i * CH, len = std::min(CH, bytes - off);
		cudaMemcpyAsync(pin + (i % kStageBufs) * CH, (const uint8_t*)src + off, len, cudaMemcpyDeviceToHost, st);
		cudaEventRecord(ev[i % kStageBufs], st);
	};
	for (size_t i = 0; i < std::min<size_t>(nch, kStageBufs - 1); i++) issue(i);
	for (size_t i = 0; i < nch; i++) {
		if (i + kStageBufs - 1 < nch) issue(i + kStageBufs - 1);   // its buffer was drained in the previous iteration
		cudaEventSynchronize(ev[i % kStageBufs]);
		const size_t off = i * CH, len = std::min(CH, bytes - off);
		par_memcpy((uint8_t*)dst + off, pin + (i % kStageBufs) * CH, len);
	}
	for (auto& x : ev) cudaEventDestroy(x);
}

// ------------------------------------------------------------------------------------------------ compress core
struct ShardOut {
	std::vector<uint32_t> sizes; int rc = 0; CompressStats st; double ms_h2d = 0, ms_d2h = 0; std::string err;
	const uint8_t* d_payload = nullptr; uint64_t payload_bytes = 0; int device = 0;      // streams stay on the GPU until fetched
};
enum { UB_IMG = 0, UB_SYM = 1, UB_PAY = 2, UB_F0 = 3, UB_IMG2 = 4, UB_PAY2 = 5 };

// ------------------------------------------------------------------------------------------------ slab pipeline (one GPU)
// Large stacks written to a file go through the GPU in batches of whole z-slabs: while batch b is predicted and compressed, batch
// b + 1 is on its way to the GPU (pinned staging + copy stream 0, own host thread) and the streams of batch b - 1 are on their
// way to the file (copy stream 1 + pwrite at the final offset, own host thread) -- the counterpart of the reference's block
// threads feeding blockWriter through a staging queue (src/klb_imageIO.cpp:1152-1217, :2446).  Two image and two payload buffers.
struct FileSink { int fd = -1; uint64_t base = 0; };               // payload byte 0 lives at file offset `base`
constexpr uint64_t kBatchBytes = (uint64_t)96 << 20;               // raw bytes per batch (at least one slab)
constexpr uint64_t kBatchBlocks = 2048;                            // ... and at least this many KLB blocks

static int payload_to_fd(Engine& e, const uint8_t* d_payload, uint64_t bytes, int fd, uint64_t file_off, cudaStream_t st)
{
	uint8_t* pin = (uint8_t*)e.pinned(kStageBufs * kStageChunk, 1);
	if (!pin) return LFM_ERR_CUDA;
	cudaEvent_t ev[kStageBufs];
	for (auto& x : ev) cudaEventCreateWithFlags(&x, cudaEventDisableTiming);
	const size_t nch = (size_t)((bytes + kStageChunk - 1) / kStageChunk);
	auto issue = [&](size_t i) {
		const uint64_t o = (uint64_t)i * kStageChunk; const size_t len = (size_t)std::min<uint64_t>(kStageChunk, bytes - o);
		cudaMemcpyAsync(pin + (i % kStageBufs) * kStageChunk, d_payload + o, len, cudaMemcpyDeviceToHost, st);
		cudaEventRecord(ev[i % kStageBufs], st);
	};
	int rc = LFM_OK;
	for (size_t i = 0; i < std::min<size_t>(nch, kStageBufs - 1); i++) issue(i);
	for (size_t i = 0; i < nch && rc == LFM_OK; i++) {
		if (i + kStageBufs - 1 < nch) issue(i + kStageBufs - 1);           // its buffer was written out in the previous iteration
		if (cudaEventSynchronize(ev[i % kStageBufs]) != cudaSuccess) { cudaGetLastError(); rc = LFM_ERR_CUDA; break; }
		const uint64_t o = (uint64_t)i * kStageChunk; const size_t len = (size_t)std::min<uint64_t>(kStageChunk, bytes - o);
		const uint8_t* buf = pin + (i % kStageBufs) * kStageChunk;
		size_t done = 0;
		while (done < len) {
			const ssize_t w = pwrite(fd, buf + done, len - done, (off_t)(file_off + o + done));
			if (w <= 0) { rc = LFM_ERR_CREATE; break; }
			done += (size_t)w;
		}
	}
	cudaStreamSynchronize(st);
	for (auto& x : ev) cudaEventDestroy(x);
	return rc;
}

// slabs per batch; 0 when the stack is not worth / not fit for batching (few slabs, c or t blocked)
static uint64_t slabs_per_batch(const klb_image_header& h, const Layout& L, bool pair_frames)
{
	if (env_int("LFM_B200_NO_PIPELINE", 0) || h.blockSize[3] != 1 || h.blockSize[4] != 1) return 0;
	const uint64_t batch_bytes = env_int("LFM_B200_BATCH_KB", 0) > 0 ? (uint64_t)env_int("LFM_B200_BATCH_KB", 0) << 10 : kBatchBytes;   // test knob
	const uint64_t slab_bytes = (uint64_t)h.blockSize[2] * L.fpx * 2;
	uint64_t n = std::max<uint64_t>(1, batch_bytes / std::max<uint64_t>(1, slab_bytes));
	// the block codec kernels are latency bound: a batch needs a few thousand KLB blocks to fill the GPU (k_huff_decode alone keeps
	// ~1500 streams in flight), or the overlap won is lost again in half-empty kernels
	if (env_int("LFM_B200_BATCH_KB", 0) <= 0) n = std::max<uint64_t>(n, (kBatchBlocks + L.blocksPerSlab - 1) / L.blocksPerSlab);
	if (pair_frames && (h.blockSize[2] & 1)) n = (n + 1) & ~(uint64_t)1;         // batches start on even frames
	return L.nSlabs >= 2 * n ? n : 0;
}

static int compress_pipelined(const FrameSource& src, klb_image_header& h, const Layout& L, const StackDesc& desc, int k, int video,
                              const FileSink& sink, uint64_t per)
{
	Engine& e = Engine::for_device(g_set.first_device);
	cudaSetDevice(e.device());
	const int dev = e.device();
	cudaStream_t up_st = (cudaStream_t)e.copy_stream(0), down_st = (cudaStream_t)e.copy_stream(1);   // created on this thread
	const uint64_t nbatch = (L.nSlabs + per - 1) / per;
	struct Batch { uint64_t s0, s1, f0, nf; };
	std::vector<Batch> B(nbatch);
	uint64_t max_nf = 0;
	for (uint64_t b = 0; b < nbatch; b++) {
		B[b].s0 = b * per; B[b].s1 = std::min(L.nSlabs, (b + 1) * per);
		uint64_t f0, f1; slab_frames(h, L, B[b].s0, B[b].s1, f0, f1);
		B[b].f0 = f0; B[b].nf = f1 - f0 + 1;
		max_nf = std::max(max_nf, B[b].nf);
	}
	const size_t img_bytes = (size_t)max_nf * L.fpx * 2;
	if ((!src.device && (e.reserve(e.user[UB_IMG], img_bytes) || e.reserve(e.user[UB_IMG2], img_bytes))) ||
	    (k != 0 && e.reserve(e.user[UB_SYM], img_bytes))) return LFM_ERR_CUDA;
	if (!e.pinned(kStageBufs * kStageChunk, 0) || !e.pinned(kStageBufs * kStageChunk, 1)) return LFM_ERR_CUDA;
	uint16_t* dimg[2] = { (uint16_t*)e.user[UB_IMG].p, (uint16_t*)e.user[UB_IMG2].p };
	uint16_t* dsym = (uint16_t*)e.user[UB_SYM].p;
	std::thread up_th[2], wr_th[2];
	int up_rc[2] = { 0, 0 }, wr_rc[2] = { 0, 0 };
	auto upload = [&](uint64_t b, int slot) {
		if (src.device) return;                                        // the kernels read the caller's device stack
		cudaSetDevice(dev);
		const Batch& bt = B[b];
		if (src.base) h2d_staged(e, dimg[slot], src.frame(bt.f0, L.fpx), (size_t)bt.nf * L.fpx * 2, up_st);
		else for (uint64_t f = 0; f < bt.nf; f++) h2d_staged(e, dimg[slot] + f * L.fpx, src.frame(bt.f0 + f, L.fpx), (size_t)L.fpx * 2, up_st);
		if (cudaStreamSynchronize(up_st) != cudaSuccess) { cudaGetLastError(); up_rc[slot] = LFM_ERR_CUDA; }
	};
	auto join_all = [&]() { for (auto& t : up_th) if (t.joinable()) t.join(); for (auto& t : wr_th) if (t.joinable()) t.join(); };
	int rc = LFM_OK;
	uint64_t pay_off = 0, blk = 0;
	std::vector<uint32_t> sizes;
	const double t0 = now_ms();
	up_th[0] = std::thread(upload, 0, 0);
	for (uint64_t b = 0; b < nbatch && rc == LFM_OK; b++) {
		const int slot = (int)(b & 1);
		up_th[slot].join();                                            // batch b is resident
		if ((rc = up_rc[slot])) break;
		if (b + 1 < nbatch) up_th[slot ^ 1] = std::thread(upload, b + 1, slot ^ 1);   // its image buffer was last read by batch b - 1 (done)
		if (wr_th[slot].joinable()) { wr_th[slot].join(); if ((rc = wr_rc[slot])) break; }   // payload buffer `slot` (batch b - 2) is on disk
		const Batch& bt = B[b];
		const uint16_t* img_base = src.device ? src.base : dimg[slot] - bt.f0 * L.fpx;   // virtual base: absolute frame indexing
		const uint16_t* sym_base = img_base;
		CompressStats st;
		if (k != 0) {
			rc = e.predict(img_base, dsym - bt.f0 * L.fpx, desc, k, video, (uint32_t)bt.f0, (uint32_t)bt.nf);
			st.launches++;
			if (rc) break;
			sym_base = dsym - bt.f0 * L.fpx;
		}
		const uint64_t first = bt.s0 * L.blocksPerSlab, count = (bt.s1 - bt.s0) * L.blocksPerSlab;
		sizes.resize(count);
		const uint8_t* dpay = nullptr; uint64_t pbytes = 0;
		e.use_payload_buffer(slot);
		rc = e.compress_blocks(sym_base, desc, first, count, sizes.data(), &dpay, &pbytes, &st);
		if (rc) { g_err = e.last_error(); break; }
		if (k != 0) g_stats.ms_predict += e.last_predict_ms();
		uint64_t acc = blk ? h.blockOffset[blk - 1] : 0;
		for (uint64_t i = 0; i < count; i++) { acc += sizes[i]; h.blockOffset[blk + i] = acc; }
		blk += count;
		g_stats.ms_rle += st.ms_rle; g_stats.ms_bwt += st.ms_bwt; g_stats.ms_mtf += st.ms_mtf; g_stats.ms_huff += st.ms_huff;
		g_stats.gpu_launches += st.launches; g_stats.periodic_blocks += st.periodic_blocks;
		const uint64_t at = sink.base + pay_off;
		// one writer at a time (they share the pinned ring and copy stream 1): batch b - 1 had all of this batch's kernels to finish
		if (wr_th[slot ^ 1].joinable()) { wr_th[slot ^ 1].join(); if ((rc = wr_rc[slot ^ 1])) break; }
		wr_th[slot] = std::thread([&, slot, dpay, pbytes, at]() { cudaSetDevice(dev); wr_rc[slot] = pbytes ? payload_to_fd(e, dpay, pbytes, sink.fd, at, down_st) : LFM_OK; });
		pay_off += pbytes;
	}
	join_all();
	e.use_payload_buffer(0);
	for (int i = 0; i < 2; i++) { if (!rc && up_rc[i]) rc = up_rc[i]; if (!rc && wr_rc[i]) rc = wr_rc[i]; }
	g_stats.payload_bytes = pay_off;
	g_stats.ms_total += now_ms() - t0;
	return rc;
}

// Phase 1: everything up to the compacted streams in device memory + header.blockOffset[].
// With a FileSink and one GPU, large stacks take the slab pipeline: the payload is then already in the file when this returns
// (shards stays empty) and only the header + table are left to write.
int compress_core(const FrameSource& src, klb_image_header& h, std::vector<ShardOut>& shards, std::vector<uint64_t>& shardFirstBlock,
                  const FileSink* sink = nullptr)
{
	memset(&g_stats, 0, sizeof(g_stats));
	int rc = validate(h, true);
	if (rc) return rc;
	const int ndev = current_ndev();
	if (ndev <= 0) { std::cout << "ERROR: lfm_b200: no CUDA device available (this engine has no CPU fallback)" << std::endl; return LFM_ERR_CUDA; }
	if (src.device && (rc = check_device_ptr(src.base, "d_im"))) return rc;
	const int way = current_way();
	for (int d = 0; d < 5; d++) h.blockSize[d] = std::min(h.blockSize[d], h.xyzct[d]);     // src/klb_imageIO.cpp:2407-2408
	const Layout L = make_layout(h);
	h.resizeBlockOffset(L.Nb);
	const StackDesc desc = make_desc(h, way);
	const uint8_t hv_in = h.headerVersion;
	const int video = (hv_in & 0x80) ? 1 : 0;
	int k;
	const double t_start = now_ms();
	if ((hv_in & 0x7F) < NUM_PREDICTORS) {
		// auto-select on frame 0 (branches A and B of writeImage, src/klb_imageIO.cpp:2273-2377)
		Engine& e = Engine::for_device(g_set.first_device);
		cudaSetDevice(e.device());
		const uint16_t* f0 = src.base;
		if (!src.device) {
			if (e.reserve(e.user[UB_F0], L.fpx * 2)) return LFM_ERR_CUDA;
			// stream-ordered copy: a default-stream cudaMemcpy from pageable memory may return before the DMA has landed,
			// and the engine's non-blocking stream does not wait for the default stream
			cudaMemcpyAsync(e.user[UB_F0].p, src.frame(0, L.fpx), L.fpx * 2, cudaMemcpyHostToDevice, (cudaStream_t)e.stream());
			f0 = (const uint16_t*)e.user[UB_F0].p;
		}
		double t0 = now_ms();
		rc = e.select_mode(f0, desc, g_stats.entropy, &k);
		if (rc) { g_err = e.last_error(); return rc; }
		g_stats.ms_select = now_ms() - t0;
		g_stats.selected = 1; g_stats.gpu_launches += 7 + 5;       // 7 candidate predictions + count, starts, sort, histogram, entropy
	} else {
		k = hv_in & 0x77 & 0x7F;                       // `hv & 0x7F - 8` parses as hv & 0x77 (src/klb_imageIO.cpp:2380)
		if (k > 7) { std::cout << "ERROR: The predictors hava not selected!" << std::endl; return LFM_ERR_UNSUPPORTED; }
	}
	if (k != 0 && video && way != 0) {
		std::cout << "ERROR: lfm_b200: video stacks are only invertible with predictor way 0 (tiles); refusing to write" << std::endl;
		return LFM_ERR_UNSUPPORTED;
	}
	h.headerVersion = (uint8_t)((hv_in & 0x80) | k);
	g_stats.predictor = k;

	// a device stack lives on the first device: it is compressed there alone
	const int D = src.device ? 1 : (int)std::min<uint64_t>((uint64_t)ndev, L.nSlabs);
	if (sink && D == 1) {
		const uint64_t per = slabs_per_batch(h, L, k != 0 && video);
		if (per) {
			FileSink fs = *sink; fs.base = sizeof(uint8_t) * 320 + L.Nb * sizeof(uint64_t);
			shards.clear(); shardFirstBlock.clear();
			return compress_pipelined(src, h, L, desc, k, video, fs, per);
		}
	}
	const std::vector<uint64_t> cut = shard_cuts(h, L, D, k != 0 && video);
	shards.assign(D, ShardOut());
	shardFirstBlock.assign(D, 0);
	auto work = [&](int d) {
		ShardOut& out = shards[d];
		const uint64_t s0 = cut[d], s1 = cut[d + 1];
		shardFirstBlock[d] = s0 * L.blocksPerSlab;
		if (s0 == s1) return;                               // fewer indivisible slab groups than GPUs
		uint64_t f0, f1; slab_frames(h, L, s0, s1, f0, f1);
		if (k != 0 && video && (f0 & 1)) f0--;              // an odd first frame is predicted from the even one before it
		const uint64_t nf = f1 - f0 + 1;
		Engine& e = Engine::for_device(g_set.first_device + d);
		out.device = e.device();
		cudaSetDevice(e.device());
		cudaStream_t st = (cudaStream_t)e.stream();
		if ((!src.device && e.reserve(e.user[UB_IMG], nf * L.fpx * 2)) || (k != 0 && e.reserve(e.user[UB_SYM], nf * L.fpx * 2))) { out.rc = LFM_ERR_CUDA; return; }
		uint16_t* dimg = (uint16_t*)e.user[UB_IMG].p; uint16_t* dsym = (uint16_t*)e.user[UB_SYM].p;
		double t0 = now_ms();
		if (src.device) { /* the kernels read the caller's device stack */ }
		else if (src.base) h2d_staged(e, dimg, src.frame(f0, L.fpx), nf * L.fpx * 2, st);
		else for (uint64_t f = 0; f < nf; f++) cudaMemcpyAsync(dimg + f * L.fpx, src.frame(f0 + f, L.fpx), L.fpx * 2, cudaMemcpyHostToDevice, st);
		const uint16_t* img_base = src.device ? src.base : dimg - f0 * L.fpx;       // virtual base: absolute frame indexing
		const uint16_t* sym_base = img_base;
		if (k != 0) {
			out.rc = e.predict(img_base, dsym - f0 * L.fpx, desc, k, video, (uint32_t)f0, (uint32_t)nf);
			out.st.launches++;
			if (out.rc) return;
			sym_base = dsym - f0 * L.fpx;
		}
		const uint64_t first = s0 * L.blocksPerSlab, count = (s1 - s0) * L.blocksPerSlab;
		shardFirstBlock[d] = first;
		out.sizes.resize(count);
		out.rc = e.compress_blocks(sym_base, desc, first, count, out.sizes.data(), &out.d_payload, &out.payload_bytes, &out.st);
		if (k != 0 && out.rc == 0) out.st.ms_predict = e.last_predict_ms();
		out.ms_h2d = src.device ? 0 : now_ms() - t0;        // H2D + kernels (the copy is asynchronous and overlaps nothing yet)
		if (out.rc) { out.err = e.last_error(); return; }
	};
	if (D == 1) work(0);
	else {
		std::vector<std::thread> th;
		for (int d = 0; d < D; d++) th.emplace_back(work, d);
		for (auto& t : th) t.join();
	}
	for (auto& s : shards) if (s.rc) { g_err = s.err; return s.rc; }
	// host-side inclusive prefix sum of the block sizes -> blockOffset[] (END offsets)
	uint64_t acc = 0;
	for (int d = 0; d < D; d++) {
		const ShardOut& s = shards[d];
		for (size_t i = 0; i < s.sizes.size(); i++) { acc += s.sizes[i]; h.blockOffset[shardFirstBlock[d] + i] = acc; }
		g_stats.ms_predict = std::max(g_stats.ms_predict, s.st.ms_predict);
		g_stats.ms_rle = std::max(g_stats.ms_rle, s.st.ms_rle); g_stats.ms_bwt = std::max(g_stats.ms_bwt, s.st.ms_bwt);
		g_stats.ms_mtf = std::max(g_stats.ms_mtf, s.st.ms_mtf); g_stats.ms_huff = std::max(g_stats.ms_huff, s.st.ms_huff);
		g_stats.ms_h2d = std::max(g_stats.ms_h2d, s.ms_h2d);
		g_stats.gpu_launches += s.st.launches; g_stats.periodic_blocks += s.st.periodic_blocks;
	}
	g_stats.payload_bytes = acc;
	g_stats.ms_total = now_ms() - t_start;
	return LFM_OK;
}

// Phase 2: bring the shards' streams to the host, in block order, at dst (payload_bytes total)
int fetch_payload(std::vector<ShardOut>& shards, uint8_t* dst)
{
	const double t0 = now_ms();
	uint64_t off = 0;
	for (auto& s : shards) {
		cudaSetDevice(s.device);
		Engine& e = Engine::for_device(s.device);
		if (s.payload_bytes) cudaMemcpyAsync(dst + off, s.d_payload, s.payload_bytes, cudaMemcpyDeviceToHost, (cudaStream_t)e.stream());
		off += s.payload_bytes;
	}
	int rc = LFM_OK;
	for (auto& s : shards) {
		cudaSetDevice(s.device);
		if (cudaStreamSynchronize((cudaStream_t)Engine::for_device(s.device).stream()) != cudaSuccess) { cudaGetLastError(); rc = LFM_ERR_CUDA; }
	}
	g_stats.ms_d2h = now_ms() - t0;
	g_stats.ms_total += g_stats.ms_d2h;
	return rc;
}

// ------------------------------------------------------------------------------------------------ decompress core
// Where the block streams come from: a payload resident in HOST memory (first byte after the blockOffset table), or an open
// file of which only the byte ranges a shard needs are read (pread) -- an ROI that touches a few slabs of a multi-GB file
// costs the I/O of those slabs (the random-access use case of the KLB layout, src/klb_imageIO.cpp:524-763).
struct PayloadSource {
	const uint8_t* base = nullptr;      // memory-resident payload
	int fd = -1; uint64_t file_off = 0; // or: file descriptor + offset of the payload inside the file
	uint64_t size = 0;                  // payload bytes available
	// the payload byte ranges [r.first, r.second) -> device memory, packed one after the other at dst, on stream st.  File sources
	// go through two pinned staging buffers of the engine: chunk i+1 is read from the file while chunk i crosses PCIe.
	// Returns 0, or LFM_ERR_BZIP on a short read.
	int to_device(Engine& e, void* dst, const std::vector<std::pair<uint64_t, uint64_t>>& ranges, cudaStream_t st) const
	{
		uint64_t dpos = 0;
		if (base) {
			for (const auto& r : ranges) { cudaMemcpyAsync((uint8_t*)dst + dpos, base + r.first, r.second - r.first, cudaMemcpyHostToDevice, st); dpos += r.second - r.first; }
			return LFM_OK;
		}
		uint64_t total = 0;
		for (const auto& r : ranges) total += r.second - r.first;
		const uint64_t CH = total >= ((uint64_t)64 << 20) ? (uint64_t)16 << 20 : (uint64_t)2 << 20;      // two buffers: 16 MB chunks fit the 32 MB ring
		uint8_t* pin = (uint8_t*)e.pinned(kStageBufs * kStageChunk, 0);
		if (!pin) return LFM_ERR_CUDA;
		cudaEvent_t ev[2]; cudaEventCreateWithFlags(&ev[0], cudaEventDisableTiming); cudaEventCreateWithFlags(&ev[1], cudaEventDisableTiming);
		int rc = LFM_OK;
		uint64_t i = 0;
		for (const auto& r : ranges) {
			for (uint64_t off = r.first; off < r.second && rc == LFM_OK; off += CH, i++) {
				const uint64_t len = std::min<uint64_t>(CH, r.second - off);
				uint8_t* buf = pin + (i & 1) * CH;
				if (i >= 2) cudaEventSynchronize(ev[i & 1]);          // the copy that last used this buffer has finished
				rc = par_pread(fd, buf, (size_t)len, file_off + off);
				if (rc) break;
				cudaMemcpyAsync((uint8_t*)dst + dpos, buf, len, cudaMemcpyHostToDevice, st);
				cudaEventRecord(ev[i & 1], st);
				dpos += len;
			}
			if (rc) break;
		}
		cudaStreamSynchronize(st);                                // the staging buffers are free again (they are shared with the write path)
		cudaEventDestroy(ev[0]); cudaEventDestroy(ev[1]);
		return rc;
	}
};

// Full reads of large stacks on one GPU, the mirror image of compress_pipelined: while batch b (whole z-slabs) is decoded and
// un-predicted, the streams of batch b + 1 are read from the file / host memory into the second payload buffer (pinned staging,
// copy stream 0, own host thread) and the pixels of batch b - 1 travel to the caller's buffer (copy stream 1, own host thread).
// With out_on_device, `out` is the caller's device buffer: the batches decode straight into it and there is no download stage.
static int decompress_pipelined(const klb_image_header& h, const Layout& L, const StackDesc& desc, int k, int video,
                                const PayloadSource& psrc, uint16_t* out, bool out_on_device, uint64_t per)
{
	Engine& e = Engine::for_device(g_set.first_device);
	cudaSetDevice(e.device());
	const int dev = e.device();
	cudaStream_t up_st = (cudaStream_t)e.copy_stream(0), down_st = (cudaStream_t)e.copy_stream(1);
	const uint64_t nbatch = (L.nSlabs + per - 1) / per;
	struct Batch { uint64_t s0, s1, f0, nf, beg, end; };
	std::vector<Batch> B(nbatch);
	uint64_t max_nf = 0, max_pay = 0;
	for (uint64_t b = 0; b < nbatch; b++) {
		Batch& bt = B[b];
		bt.s0 = b * per; bt.s1 = std::min(L.nSlabs, (b + 1) * per);
		uint64_t f0, f1; slab_frames(h, L, bt.s0, bt.s1, f0, f1);
		bt.f0 = f0; bt.nf = f1 - f0 + 1;
		const uint64_t id0 = bt.s0 * L.blocksPerSlab, id1 = bt.s1 * L.blocksPerSlab;
		bt.beg = id0 ? h.blockOffset[id0 - 1] : 0; bt.end = h.blockOffset[id1 - 1];
		max_nf = std::max(max_nf, bt.nf); max_pay = std::max(max_pay, bt.end - bt.beg);
	}
	const size_t img_bytes = (size_t)max_nf * L.fpx * 2;
	if (e.reserve(e.user[UB_PAY], max_pay + 16) || e.reserve(e.user[UB_PAY2], max_pay + 16) ||
	    (!out_on_device && (e.reserve(e.user[UB_IMG], img_bytes) || e.reserve(e.user[UB_IMG2], img_bytes))) ||
	    (k != 0 && e.reserve(e.user[UB_SYM], img_bytes))) return LFM_ERR_CUDA;
	if (!e.pinned(kStageBufs * kStageChunk, 0) || !e.pinned(kStageBufs * kStageChunk, 1)) return LFM_ERR_CUDA;
	uint8_t* dpay[2] = { (uint8_t*)e.user[UB_PAY].p, (uint8_t*)e.user[UB_PAY2].p };
	uint16_t* dimg[2] = { (uint16_t*)e.user[UB_IMG].p, (uint16_t*)e.user[UB_IMG2].p };
	uint16_t* dsym = (uint16_t*)e.user[UB_SYM].p;
	std::thread up_th[2], dn_th[2];
	int up_rc[2] = { 0, 0 }, dn_rc[2] = { 0, 0 };
	auto fetch = [&](uint64_t b, int slot) {
		cudaSetDevice(dev);
		std::vector<std::pair<uint64_t, uint64_t>> ranges(1, std::make_pair(B[b].beg, B[b].end));
		up_rc[slot] = psrc.to_device(e, dpay[slot], ranges, up_st);
		if (cudaStreamSynchronize(up_st) != cudaSuccess) { cudaGetLastError(); up_rc[slot] = LFM_ERR_CUDA; }
	};
	auto join_all = [&]() { for (auto& t : up_th) if (t.joinable()) t.join(); for (auto& t : dn_th) if (t.joinable()) t.join(); };
	int rc = LFM_OK;
	std::vector<uint64_t> ids, beg, end;
	const double t0 = now_ms();
	up_th[0] = std::thread(fetch, 0, 0);
	for (uint64_t b = 0; b < nbatch && rc == LFM_OK; b++) {
		const int slot = (int)(b & 1);
		up_th[slot].join();
		if ((rc = up_rc[slot])) { if (rc == LFM_ERR_BZIP) std::cerr << "ERROR: lfm_b200: file is truncated" << std::endl; break; }
		if (b + 1 < nbatch) up_th[slot ^ 1] = std::thread(fetch, b + 1, slot ^ 1);    // its payload buffer was decoded by batch b - 1 (done)
		if (dn_th[slot].joinable()) { dn_th[slot].join(); if ((rc = dn_rc[slot])) break; }   // image buffer `slot` (batch b - 2) has left
		const Batch& bt = B[b];
		const uint64_t id0 = bt.s0 * L.blocksPerSlab, cnt = (bt.s1 - bt.s0) * L.blocksPerSlab;
		ids.resize(cnt); beg.resize(cnt); end.resize(cnt);
		for (uint64_t i = 0; i < cnt; i++) {
			ids[i] = id0 + i;
			beg[i] = ((id0 + i) ? h.blockOffset[id0 + i - 1] : 0) - bt.beg; end[i] = h.blockOffset[id0 + i] - bt.beg;
		}
		uint16_t* res = out_on_device ? out : dimg[slot] - bt.f0 * L.fpx;   // virtual base: absolute frame indexing
		uint16_t* sym_base = k != 0 ? dsym - bt.f0 * L.fpx : res;
		DecompressStats st;
		rc = e.decompress_blocks(dpay[slot], beg.data(), end.data(), ids.data(), cnt, sym_base, desc, &st);
		if (rc) { g_err = e.last_error(); break; }
		if (k != 0) {
			rc = e.unpredict(sym_base, res, desc, k, video, (uint32_t)bt.f0, (uint32_t)bt.nf);
			st.launches += video ? 2 : 1;
			if (rc) break;
			if (cudaStreamSynchronize((cudaStream_t)e.stream()) != cudaSuccess) { cudaGetLastError(); rc = LFM_ERR_CUDA; break; }
			g_stats.ms_unpredict += e.last_unpredict_ms();
		}
		g_stats.ms_decode += st.ms_decode; g_stats.ms_imtf += st.ms_imtf; g_stats.ms_ibwt += st.ms_ibwt; g_stats.ms_unrle += st.ms_unrle;
		g_stats.gpu_launches += st.launches;
		if (out_on_device) continue;                                   // the pixels are in place and the engine stream is synchronised
		const uint16_t* srcp = dimg[slot]; uint16_t* dstp = out + bt.f0 * L.fpx; const size_t nbytes = (size_t)bt.nf * L.fpx * 2;
		// one download at a time (they share the pinned ring and copy stream 1): batch b - 1 had all of this batch's kernels to finish
		if (dn_th[slot ^ 1].joinable()) { dn_th[slot ^ 1].join(); if ((rc = dn_rc[slot ^ 1])) break; }
		dn_th[slot] = std::thread([&, slot, srcp, dstp, nbytes]() {
			cudaSetDevice(dev);
			d2h_staged(e, dstp, srcp, nbytes, down_st);
			if (cudaStreamSynchronize(down_st) != cudaSuccess) { cudaGetLastError(); dn_rc[slot] = LFM_ERR_CUDA; }
		});
	}
	join_all();
	for (int i = 0; i < 2; i++) { if (!rc && up_rc[i]) rc = up_rc[i]; if (!rc && dn_rc[i]) rc = dn_rc[i]; }
	g_stats.ms_total = now_ms() - t0;
	return rc;
}

// Pixels go to the host buffer `out`, or with a DeviceSink to its device buffer (then `out` is ignored): full reads into a
// 16-byte aligned buffer decode straight into it; ROI reads, and full reads into any other buffer, decode into the engine's
// frame buffers and k_roi_gather copies the box out.
int decompress_core(const klb_image_header& h, const PayloadSource& psrc, uint16_t* out, const klb_ROI* roi, const DeviceSink* dsink = nullptr)
{
	const uint64_t payload_size = psrc.size;
	memset(&g_stats, 0, sizeof(g_stats));
	int rc = validate(h, false);
	if (rc) return rc;
	const int ndev = current_ndev();
	if (ndev <= 0) { std::cout << "ERROR: lfm_b200: no CUDA device available (this engine has no CPU fallback)" << std::endl; return LFM_ERR_CUDA; }
	if (h.Nb == 0) { std::cerr << "ERROR: Image to read has not blocks" << std::endl; return LFM_ERR_BZIP; }
	const int way = current_way();
	const Layout L = make_layout(h);
	if (L.Nb != h.Nb) return LFM_ERR_BZIP;
	if (h.blockOffset[L.Nb - 1] > payload_size) { std::cerr << "ERROR: lfm_b200: file is truncated" << std::endl; return LFM_ERR_BZIP; }
	// the table comes from an untrusted file: END offsets must not decrease and none may point past the payload (an ROI read
	// skips blocks, so checking only the last one is not enough)
	for (uint64_t i = 1; i < L.Nb; i++)
		if (h.blockOffset[i] < h.blockOffset[i - 1]) { std::cerr << "ERROR: lfm_b200: corrupt blockOffset table" << std::endl; return LFM_ERR_BZIP; }
	const StackDesc desc = make_desc(h, way);
	const int k = h.headerVersion & 0x7F, video = (h.headerVersion & 0x80) ? 1 : 0;
	if (k > 7) return LFM_ERR_UNSUPPORTED;
	if (k != 0 && video && way != 0) {
		std::cout << "ERROR: lfm_b200: video stack written with predictor way != 0 cannot be inverted (reference defect, see DESIGN.md)" << std::endl;
		return LFM_ERR_UNSUPPORTED;
	}
	const double t_start = now_ms();
	g_stats.predictor = k;

	// which slabs / blocks are needed
	uint32_t lb[5], ub[5];
	bool full = true;
	for (int d = 0; d < 5; d++) {
		lb[d] = roi ? roi->xyzctLB[d] : 0; ub[d] = roi ? roi->xyzctUB[d] : h.xyzct[d] - 1;
		if (ub[d] >= h.xyzct[d] || lb[d] > ub[d]) return LFM_ERR_OPEN;
		if (lb[d] != 0 || ub[d] != h.xyzct[d] - 1) full = false;
	}
	if (dsink) {
		// the caller's buffer is checked before any kernel runs: nothing is written to it unless the whole box fits
		uint64_t bytes = 2;
		for (int d = 0; d < 5; d++) bytes *= (uint64_t)(ub[d] - lb[d] + 1);
		if (dsink->out_bytes) *dsink->out_bytes = bytes;
		if ((rc = check_device_ptr(dsink->d_out, "d_out"))) return rc;
		if (dsink->capacity < bytes) { g_err = "d_out is smaller than the box (" + std::to_string(bytes) + " bytes)"; return LFM_ERR_CREATE; }
		out = (uint16_t*)dsink->d_out;
	}
	// slabs intersecting the ROI along z, c, t
	std::vector<uint64_t> slabs;
	for (uint64_t s = 0; s < L.nSlabs; s++) {
		uint64_t bz = s % L.nb[2], r = s / L.nb[2], bc = r % L.nb[3], bt = r / L.nb[3];
		auto hit = [&](int d, uint64_t b) { uint64_t a0 = b * h.blockSize[d], a1 = std::min<uint64_t>(h.xyzct[d], a0 + h.blockSize[d]) - 1; return a0 <= ub[d] && a1 >= lb[d]; };
		if (hit(2, bz) && hit(3, bc) && hit(4, bt)) slabs.push_back(s);
	}
	// video + predictor: an odd first frame needs the even frame before it -> also the slab that holds it
	if (k != 0 && video && !slabs.empty()) {
		uint64_t f0, f1; slab_frames(h, L, slabs.front(), slabs.front() + 1, f0, f1);
		if ((f0 & 1) && slabs.front() > 0) slabs.insert(slabs.begin(), slabs.front() - 1);
	}
	const bool contiguous = !slabs.empty() && (slabs.back() - slabs.front() + 1 == slabs.size());
	// Full reads are sharded over the GPUs by slab ranges whose frame ranges are disjoint: with c or t blocked (blockSize[3] or
	// blockSize[4] > 1) the frames of neighbouring slabs interleave, and one GPU decodes the stack.  A device buffer is on the
	// first device, which decodes everything.
	const bool disjoint = h.blockSize[3] == 1 && h.blockSize[4] == 1;
	const int D = (!dsink && full && contiguous && disjoint && slabs.size() == L.nSlabs) ? (int)std::min<uint64_t>((uint64_t)ndev, slabs.size()) : 1;
	// The decode and inverse-predictor kernels take 16-byte vector paths from the frame width alone, assuming a frame buffer
	// aligned as the engine's are: a caller's buffer that is not 16-byte aligned only receives k_roi_gather's copy of the box
	// (the whole stack for a full read), which handles any alignment.
	const bool sink_aligned = dsink && ((uintptr_t)dsink->d_out & 15) == 0;
	if (full && D == 1 && desc.codec == 1 && (!dsink || sink_aligned)) {
		const uint64_t per = slabs_per_batch(h, L, k != 0 && video);
		if (per) return decompress_pipelined(h, L, desc, k, video, psrc, out, dsink != nullptr, per);
	}
	const bool direct = dsink && full && sink_aligned;   // decode into the caller's device buffer, no copy at the end
	const std::vector<uint64_t> cut = shard_cuts(h, L, D, k != 0 && video);

	std::vector<int> rcs(D, 0);
	std::vector<DecompressStats> sts(D);
	std::vector<double> h2d(D, 0), d2h(D, 0);
	std::vector<std::string> errs(D);
	auto work = [&](int d) {
		// this shard's slabs
		std::vector<uint64_t> my = D == 1 ? slabs : std::vector<uint64_t>(slabs.begin() + cut[d], slabs.begin() + cut[d + 1]);
		if (my.empty()) return;
		uint64_t f0 = ~0ull, f1 = 0;
		for (uint64_t s : my) { uint64_t a, b; slab_frames(h, L, s, s + 1, a, b); f0 = std::min(f0, a); f1 = std::max(f1, b); }
		if (k != 0 && video && (f0 & 1)) { rcs[d] = LFM_ERR_UNSUPPORTED; return; }   // odd block depth + video across shards
		const uint64_t nf = f1 - f0 + 1;
		// block list.  Full read: every block.  ROI without predictor: the blocks that intersect it.  ROI with a predictor: every
		// operand of the prediction rules lies up and/or left of the pixel (lfm_predict.cuh), so a pixel only depends on the
		// pixels with x' <= x and y' <= y of its frame (and of the previous frame, video) -> the blocks that start at or before
		// the ROI's lower right corner; what lies right of / below it keeps zero symbols and decodes to values nobody reads.
		std::vector<uint64_t> ids, beg, end;
		for (uint64_t s : my) for (uint64_t b = 0; b < L.blocksPerSlab; b++) {
			if (!full) {
				uint64_t bx = b % L.nb[0], by = b / L.nb[0];
				uint64_t x0 = bx * h.blockSize[0], x1 = std::min<uint64_t>(h.xyzct[0], x0 + h.blockSize[0]) - 1;
				uint64_t y0 = by * h.blockSize[1], y1 = std::min<uint64_t>(h.xyzct[1], y0 + h.blockSize[1]) - 1;
				if (x0 > ub[0] || y0 > ub[1]) continue;
				if (k == 0 && (x1 < lb[0] || y1 < lb[1])) continue;
			}
			uint64_t id = s * L.blocksPerSlab + b;
			ids.push_back(id); beg.push_back(id ? h.blockOffset[id - 1] : 0); end.push_back(h.blockOffset[id]);
			if (end.back() < beg.back()) { rcs[d] = LFM_ERR_BZIP; return; }
		}
		// byte ranges of the payload to fetch (runs of consecutive needed blocks), packed back to back on the device
		std::vector<std::pair<uint64_t, uint64_t>> ranges;
		uint64_t need_bytes = 0;
		for (size_t i = 0; i < ids.size(); i++) {
			if (!ranges.empty() && ranges.back().second == beg[i]) ranges.back().second = end[i];
			else ranges.emplace_back(beg[i], end[i]);
			const uint64_t len = end[i] - beg[i];
			beg[i] = need_bytes; end[i] = need_bytes + len;           // position inside the packed device copy
			need_bytes += len;
		}
		Engine& e = Engine::for_device(g_set.first_device + d);
		cudaSetDevice(e.device());
		cudaStream_t st = (cudaStream_t)e.stream();
		if (e.reserve(e.user[UB_PAY], need_bytes + 16) || (!(direct && k == 0) && e.reserve(e.user[UB_SYM], nf * L.fpx * 2)) ||
		    (k != 0 && !direct && e.reserve(e.user[UB_IMG], nf * L.fpx * 2))) { rcs[d] = LFM_ERR_CUDA; return; }
		struct { void* p; } dpay{ e.user[UB_PAY].p }, dsym{ e.user[UB_SYM].p }, dimg{ e.user[UB_IMG].p };
		double t0 = now_ms();
		if ((rcs[d] = psrc.to_device(e, dpay.p, ranges, st))) { if (rcs[d] == LFM_ERR_BZIP) std::cerr << "ERROR: lfm_b200: file is truncated" << std::endl; return; }
		if (!full) cudaMemsetAsync(dsym.p, 0, nf * L.fpx * 2, st);
		h2d[d] = now_ms() - t0;
		// a direct read covers the whole stack (f0 == 0): the caller's buffer is the frame buffer
		uint16_t* sym_base = (direct && k == 0) ? out : (uint16_t*)dsym.p - f0 * L.fpx;
		rcs[d] = e.decompress_blocks((const uint8_t*)dpay.p, beg.data(), end.data(), ids.data(), ids.size(), sym_base, desc, &sts[d]);
		if (rcs[d]) { errs[d] = e.last_error(); return; }
		const uint16_t* res_base = sym_base;
		if (k != 0) {
			uint16_t* res = direct ? out : (uint16_t*)dimg.p - f0 * L.fpx;
			rcs[d] = e.unpredict(sym_base, res, desc, k, video, (uint32_t)f0, (uint32_t)nf);
			sts[d].launches += video ? 2 : 1;
			if (rcs[d]) return;
			res_base = res;
		}
		t0 = now_ms();
		if (dsink) {
			if (!direct) { rcs[d] = e.roi_gather(res_base, desc, lb, ub, out); sts[d].launches++; if (rcs[d]) { errs[d] = e.last_error(); return; } }
		} else if (full) {
			// this shard's frames, contiguous in the output
			uint64_t a, b; slab_frames(h, L, my.front(), my.back() + 1, a, b);
			d2h_staged(e, out + a * L.fpx, res_base + a * L.fpx, (b - a + 1) * L.fpx * 2, st);
		} else {
			// crop: ROI rows are contiguous runs of (ub0-lb0+1) pixels
			const uint64_t rx = ub[0] - lb[0] + 1, ry = ub[1] - lb[1] + 1;
			uint64_t o = 0;
			for (uint64_t t = lb[4]; t <= ub[4]; t++) for (uint64_t c = lb[3]; c <= ub[3]; c++) for (uint64_t z = lb[2]; z <= ub[2]; z++) {
				uint64_t f = z + (uint64_t)h.xyzct[2] * (c + (uint64_t)h.xyzct[3] * t);
				cudaMemcpy2DAsync(out + o, rx * 2, res_base + f * L.fpx + (uint64_t)lb[1] * h.xyzct[0] + lb[0], (size_t)h.xyzct[0] * 2,
				                  rx * 2, ry, cudaMemcpyDeviceToHost, st);
				o += rx * ry;
			}
		}
		cudaStreamSynchronize(st);
		d2h[d] = dsink ? 0 : now_ms() - t0;
		if (k != 0) sts[d].ms_unpredict = e.last_unpredict_ms();
		if (cudaGetLastError() != cudaSuccess) rcs[d] = LFM_ERR_CUDA;
	};
	if (D == 1) work(0);
	else {
		std::vector<std::thread> th;
		for (int d = 0; d < D; d++) th.emplace_back(work, d);
		for (auto& t : th) t.join();
	}
	for (int d = 0; d < D; d++) {
		if (rcs[d]) { g_err = errs[d]; return rcs[d]; }
		g_stats.ms_decode = std::max(g_stats.ms_decode, sts[d].ms_decode); g_stats.ms_imtf = std::max(g_stats.ms_imtf, sts[d].ms_imtf); g_stats.ms_ibwt = std::max(g_stats.ms_ibwt, sts[d].ms_ibwt);
		g_stats.ms_unrle = std::max(g_stats.ms_unrle, sts[d].ms_unrle); g_stats.ms_unpredict = std::max(g_stats.ms_unpredict, sts[d].ms_unpredict);
		g_stats.ms_h2d = std::max(g_stats.ms_h2d, h2d[d]); g_stats.ms_d2h = std::max(g_stats.ms_d2h, d2h[d]);
		g_stats.gpu_launches += sts[d].launches;
	}
	g_stats.ms_total = now_ms() - t_start;
	return LFM_OK;
}

}  // namespace

// ------------------------------------------------------------------------------------------------ klb_imageIO
klb_imageIO::klb_imageIO() { numThreads = (int)std::thread::hardware_concurrency(); }
klb_imageIO::klb_imageIO(const std::string& filename_) : filename(filename_) { numThreads = (int)std::thread::hardware_concurrency(); }

// Payload -> file.  Every shard streams its compacted streams from its GPU through a ring of pinned staging buffers of its
// engine (D2H of chunk i+1 in flight while chunk i is pwrite()n at its final file position), one host thread per shard; no
// payload-sized host allocation (the counterpart of blockWriter's staging queue, src/klb_imageIO.cpp:1152-1217).
static int stream_payload_to_fd(std::vector<ShardOut>& shards, int fd, uint64_t file_off)
{
	const double t0 = now_ms();
	std::vector<uint64_t> off(shards.size(), 0);
	uint64_t acc = 0;
	for (size_t d = 0; d < shards.size(); d++) { off[d] = acc; acc += shards[d].payload_bytes; }
	std::vector<int> rcs(shards.size(), LFM_OK);
	auto work = [&](size_t d) {
		ShardOut& s = shards[d];
		if (!s.payload_bytes) return;
		cudaSetDevice(s.device);
		Engine& e = Engine::for_device(s.device);
		cudaStream_t st = (cudaStream_t)e.stream();
		uint8_t* pin = (uint8_t*)e.pinned(kStageBufs * kStageChunk, 1);
		if (!pin) { rcs[d] = LFM_ERR_CUDA; return; }
		cudaEvent_t ev[kStageBufs];
		for (auto& x : ev) cudaEventCreateWithFlags(&x, cudaEventDisableTiming);
		const uint64_t bytes = s.payload_bytes;
		const size_t CH = kStageChunk;
		// destination: a shared mapping of this shard's byte range when the file allows it.  write() / pwrite() of one file serialise
		// on its inode lock (ranks and threads that write disjoint ranges of ONE .lfm file queue up: measured 0.39 -> 1.0 ms per
		// 4 MB payload with two ranks); stores through a mapping do not, and the copy is split over the pool.
		static const int mmap_on = env_int("LFM_B200_MMAP_WRITE", 1);
		const uint64_t fbeg = file_off + off[d], fend = fbeg + bytes;
		const uint64_t page = (uint64_t)sysconf(_SC_PAGESIZE), mbase = fbeg & ~(page - 1);
		uint8_t* map = nullptr;
		if (mmap_on && bytes >= ((uint64_t)256 << 10)) {
			struct stat sb;
			if (fstat(fd, &sb) == 0 && ((uint64_t)sb.st_size >= fend || posix_fallocate(fd, sb.st_size, (off_t)(fend - (uint64_t)sb.st_size)) == 0)) {
				void* m = mmap(nullptr, (size_t)(fend - mbase), PROT_READ | PROT_WRITE, MAP_SHARED, fd, (off_t)mbase);
				if (m != MAP_FAILED) map = (uint8_t*)m;
			}
		}
		const size_t nch = (size_t)((bytes + CH - 1) / CH);
		auto issue = [&](size_t i) {
			const uint64_t o = (uint64_t)i * CH; const size_t len = (size_t)std::min<uint64_t>(CH, bytes - o);
			cudaMemcpyAsync(pin + (i % kStageBufs) * CH, s.d_payload + o, len, cudaMemcpyDeviceToHost, st);
			cudaEventRecord(ev[i % kStageBufs], st);
		};
		for (size_t i = 0; i < std::min<size_t>(nch, kStageBufs - 1); i++) issue(i);
		for (size_t i = 0; i < nch && rcs[d] == LFM_OK; i++) {
			if (i + kStageBufs - 1 < nch) issue(i + kStageBufs - 1);       // its buffer was written out in the previous iteration
			if (cudaEventSynchronize(ev[i % kStageBufs]) != cudaSuccess) { cudaGetLastError(); rcs[d] = LFM_ERR_CUDA; break; }
			const uint64_t o = (uint64_t)i * CH; const size_t len = (size_t)std::min<uint64_t>(CH, bytes - o);
			if (map) par_memcpy(map + (fbeg - mbase) + o, pin + (i % kStageBufs) * CH, len);
			else rcs[d] = write_all(fd, pin + (i % kStageBufs) * CH, len, fbeg + o);
		}
		if (map) munmap(map, (size_t)(fend - mbase));
		cudaStreamSynchronize(st);
		for (auto& x : ev) cudaEventDestroy(x);
	};
	if (shards.size() == 1) work(0);
	else {
		std::vector<std::thread> th;
		for (size_t d = 0; d < shards.size(); d++) th.emplace_back(work, d);
		for (auto& t : th) t.join();
	}
	g_stats.ms_d2h = now_ms() - t0;
	g_stats.ms_total += g_stats.ms_d2h;
	for (int rc : rcs) if (rc) return rc;
	return LFM_OK;
}

// header + blockOffset table + payload (src/klb_imageIO.cpp:1145-1225: header first, blocks appended in id order)
static int write_file(int fd, klb_image_header& h, std::vector<ShardOut>& shards)
{
	uint8_t fixed[320]; h.packFixed(fixed);
	int rc = write_all(fd, fixed, sizeof(fixed), 0);
	if (rc == 0 && h.Nb) rc = write_all(fd, h.blockOffset, h.Nb * sizeof(uint64_t), sizeof(fixed));
	if (rc) return rc;
	return stream_payload_to_fd(shards, fd, sizeof(fixed) + h.Nb * sizeof(uint64_t));
}

static int write_stack_to_file(const std::string& filename, const FrameSource& src, klb_image_header& header)
{
	LFM_API_LOCK();
	// the file is overwritten in place and cut to its final size at the end (same result as "wb", but an existing file of about
	// the same size keeps its pages: rewriting a stack does not pay for page allocation again)
	const int fd = open(filename.c_str(), O_RDWR | O_CREAT, 0666);
	if (fd < 0) { std::cout << "ERROR: file " << filename << " could not be opened" << std::endl; return LFM_ERR_CREATE; }
	int rc;
	try {
		std::vector<ShardOut> shards; std::vector<uint64_t> first;
		FileSink sink; sink.fd = fd;
		rc = compress_core(src, header, shards, first, &sink);
		if (rc == 0) rc = write_file(fd, header, shards);              // header + table (+ whatever payload is still on the GPUs)
		if (rc == 0 && ftruncate(fd, (off_t)header.getCompressedFileSizeInBytes()) != 0) rc = LFM_ERR_CREATE;
		if (rc != 0 && ftruncate(fd, 0) != 0) { /* nothing more to do */ }
	} catch (const std::bad_alloc&) { g_err = "out of host memory"; rc = LFM_ERR_CREATE; }
	if (close(fd) != 0 && rc == 0) rc = LFM_ERR_CREATE;
	return rc;
}

int klb_imageIO::writeImage(const char* img, int /*numThreads*/)
{
	FrameSource src; src.base = (const uint16_t*)img;
	return write_stack_to_file(filename, src, header);
}

int klb_imageIO::writeImageStackSlices(const char** img, int /*numThreads*/)
{
	if (header.xyzct[3] != 1 || header.xyzct[4] != 1) {
		std::cout << "ERROR: writeImageStackSlices: number of channels or number of time points must be 1 for this API call" << std::endl;
		return LFM_ERR_OPEN;
	}
	FrameSource src; src.slices = (const uint16_t* const*)img;
	return write_stack_to_file(filename, src, header);
}

int klb_imageIO::writeImageToMemory(const char* img, std::string& fileBytes)
try {
	LFM_API_LOCK();
	FrameSource src; src.base = (const uint16_t*)img;
	std::vector<ShardOut> shards; std::vector<uint64_t> first;
	int rc = compress_core(src, header, shards, first);
	if (rc) return rc;
	uint8_t fixed[320]; header.packFixed(fixed);
	uint64_t total = 0;
	for (const auto& s : shards) total += s.payload_bytes;
	fileBytes.resize(320 + header.Nb * 8 + total);
	memcpy(&fileBytes[0], fixed, 320);
	memcpy(&fileBytes[320], header.blockOffset, header.Nb * 8);
	return fetch_payload(shards, (uint8_t*)&fileBytes[320 + header.Nb * 8]);
} LFM_CATCH

int klb_imageIO::readImageFromMemory(const char* fileBytes, size_t fileSize, char* imgOut, const klb_ROI* ROI)
try {
	LFM_API_LOCK();
	if (fileSize < 320) return LFM_ERR_BZIP;
	header.unpackFixed((const uint8_t*)fileBytes);
	size_t nb = 0;
	if (!header.numBlocksBounded((fileSize - 320) / 8, &nb) || nb == 0) return LFM_ERR_BZIP;    // the table must fit the buffer
	header.resizeBlockOffset(nb);
	memcpy(header.blockOffset, fileBytes + 320, header.Nb * 8);
	PayloadSource ps; ps.base = (const uint8_t*)fileBytes + 320 + header.Nb * 8; ps.size = fileSize - 320 - header.Nb * 8;
	return decompress_core(header, ps, (uint16_t*)imgOut, ROI);
} LFM_CATCH

// header (+ blockOffset table) of the file, then decode straight from the open file: only the needed byte ranges are read
static int read_from_file(const std::string& filename, klb_image_header& header, uint16_t* out, const klb_ROI* roi,
                          const DeviceSink* dsink = nullptr)
try {
	LFM_API_LOCK();
	if (filename.empty()) { std::cerr << "ERROR: Filename has not been defined. We cannot read image" << std::endl; return LFM_ERR_OPEN; }
	if (header.Nb == 0) {
		int err = header.readHeader(filename.c_str());
		if (err > 0) return err;
		if (header.Nb == 0) { std::cerr << "ERROR: Image to read has not blocks" << std::endl; return LFM_ERR_BZIP; }
	}
	const int fd = open(filename.c_str(), O_RDONLY);
	if (fd < 0) { std::cout << "ERROR: blockUncompressor: thread opening file " << filename << std::endl; return LFM_ERR_OPEN; }
	struct stat sb;
	PayloadSource ps; ps.fd = fd; ps.file_off = header.getSizeInBytes();
	ps.size = (fstat(fd, &sb) == 0 && (uint64_t)sb.st_size > ps.file_off) ? (uint64_t)sb.st_size - ps.file_off : 0;
	const int rc = decompress_core(header, ps, out, roi, dsink);
	close(fd);
	return rc;
} LFM_CATCH

int klb_imageIO::readImageFull(char* imgOut, int /*numThreads*/) { return read_from_file(filename, header, (uint16_t*)imgOut, NULL); }

int klb_imageIO::readImage(char* img, const klb_ROI* ROI, int /*numThreads*/) { return read_from_file(filename, header, (uint16_t*)img, ROI); }

// ------------------------------------------------------------------------------------------------ extension C ABI
extern "C" {

int lfmSetPredictorWay(int way) { int prev = current_way(); if (way < 0 || way > 2) return -1; g_set.way = way; return prev; }
int lfmGetPredictorWay(void) { return current_way(); }
int lfmSetDevices(int first_device, int count)
{
	int vis = visible_devices();
	if (first_device < 0) first_device = 0;
	g_set.first_device = first_device;
	g_set.ndev = std::max(1, count);
	return std::max(0, std::min(g_set.ndev, vis - first_device));
}

int writeLFMstackEx(const void* im, const char* filename, const uint32_t xyzct[5], enum KLB_DATA_TYPE dataType, int numThreads,
                    const float32_t pixelSize[5], const uint32_t blockSize[5], enum KLB_COMPRESSION_TYPE compressionType,
                    const char metadata[256], uint8_t headerVersion, uint8_t Nnum)
try {
	if (!filename || !*filename) return LFM_ERR_OPEN;
	klb_imageIO io{ std::string(filename) };
	io.header.setHeader(xyzct, dataType, pixelSize, blockSize, compressionType, metadata, headerVersion, Nnum);
	return io.writeImage((const char*)im, numThreads);
} LFM_CATCH

int writeLFMstackDevice(const void* d_im, const char* filename, const uint32_t xyzct[5], enum KLB_DATA_TYPE dataType, int /*numThreads*/,
                        const float32_t pixelSize[5], const uint32_t blockSize[5], enum KLB_COMPRESSION_TYPE compressionType,
                        const char metadata[256], uint8_t headerVersion, uint8_t Nnum)
try {
	g_err.clear();
	if (!filename || !*filename) return LFM_ERR_OPEN;
	klb_image_header h;
	h.setHeader(xyzct, dataType, pixelSize, blockSize, compressionType, metadata, headerVersion, Nnum);
	FrameSource src; src.base = (const uint16_t*)d_im; src.device = true;
	return write_stack_to_file(std::string(filename), src, h);
} LFM_CATCH

int readLFMroiDevice(const char* filename, const uint32_t lb[5], const uint32_t ub[5], void* d_out, uint64_t capacity, uint64_t* out_bytes)
try {
	g_err.clear();
	if (out_bytes) *out_bytes = 0;
	if (!filename || !*filename || (lb == nullptr) != (ub == nullptr)) return LFM_ERR_OPEN;
	if (access(filename, R_OK) != 0) { g_err = std::string("cannot open ") + filename; return LFM_ERR_OPEN; }
	klb_image_header h;
	klb_ROI roi;
	if (lb) for (int d = 0; d < 5; d++) { roi.xyzctLB[d] = lb[d]; roi.xyzctUB[d] = ub[d]; }
	DeviceSink sink; sink.d_out = d_out; sink.capacity = capacity; sink.out_bytes = out_bytes;
	return read_from_file(std::string(filename), h, nullptr, lb ? &roi : nullptr, &sink);
} LFM_CATCH

int readLFMheaderEx(const char* filename, uint8_t* headerVersion, uint8_t* Nnum)
{
	klb_image_header h;
	int err = h.readHeader(filename);
	if (err) return err;
	if (headerVersion) *headerVersion = h.headerVersion;
	if (Nnum) *Nnum = h.Nnum;
	return 0;
}

int lfmCompressToMemory(const void* im, const uint32_t xyzct[5], const uint32_t blockSize[5], uint8_t headerVersion, uint8_t Nnum,
                        void** file_bytes, uint64_t* file_size)
try {
	LFM_API_LOCK();
	klb_imageIO io;
	io.header.setHeader(xyzct, KLB_DATA_TYPE::UINT16_TYPE, NULL, blockSize, KLB_COMPRESSION_TYPE::BZIP2, NULL, headerVersion, Nnum);
	FrameSource src; src.base = (const uint16_t*)im;
	std::vector<ShardOut> shards; std::vector<uint64_t> first;
	int rc = compress_core(src, io.header, shards, first);
	if (rc) return rc;
	uint64_t total = 0;
	for (const auto& s : shards) total += s.payload_bytes;
	const size_t hdr = 320 + io.header.Nb * 8;
	uint8_t* p = (uint8_t*)malloc(hdr + total);
	if (!p) return LFM_ERR_CREATE;
	io.header.packFixed(p);
	memcpy(p + 320, io.header.blockOffset, io.header.Nb * 8);
	rc = fetch_payload(shards, p + hdr);
	if (rc) { free(p); return rc; }
	*file_bytes = p; *file_size = hdr + total;
	return 0;
} LFM_CATCH

int lfmCompressToBuffer(const void* im, const uint32_t xyzct[5], const uint32_t blockSize[5], uint8_t headerVersion, uint8_t Nnum,
                        void* file_bytes, uint64_t capacity, uint64_t* file_size)
try {
	LFM_API_LOCK();
	klb_imageIO io;
	io.header.setHeader(xyzct, KLB_DATA_TYPE::UINT16_TYPE, NULL, blockSize, KLB_COMPRESSION_TYPE::BZIP2, NULL, headerVersion, Nnum);
	FrameSource src; src.base = (const uint16_t*)im;
	std::vector<ShardOut> shards; std::vector<uint64_t> first;
	int rc = compress_core(src, io.header, shards, first);
	if (rc) return rc;
	uint64_t total = 0;
	for (const auto& s : shards) total += s.payload_bytes;
	const size_t hdr = 320 + io.header.Nb * 8;
	if (file_size) *file_size = hdr + total;
	if (!file_bytes || capacity < hdr + total) return LFM_ERR_CREATE;
	uint8_t* p = (uint8_t*)file_bytes;
	io.header.packFixed(p);
	memcpy(p + 320, io.header.blockOffset, io.header.Nb * 8);
	return fetch_payload(shards, p + hdr);
} LFM_CATCH

int lfmDecompressFromMemory(const void* file_bytes, uint64_t file_size, void* im)
try {
	klb_imageIO io;
	return io.readImageFromMemory((const char*)file_bytes, (size_t)file_size, (char*)im, NULL);
} LFM_CATCH

uint64_t lfmNumBlocks(const uint32_t xyzct[5], const uint32_t blockSize[5])
{
	klb_image_header h;
	h.setHeader(xyzct, KLB_DATA_TYPE::UINT16_TYPE, NULL, blockSize);
	for (int d = 0; d < 5; d++) { if (h.xyzct[d] == 0) return 0; h.blockSize[d] = std::min(h.blockSize[d], h.xyzct[d]); }
	return h.calculateNumBlocks();
}

int lfmCompressDevice(const void* d_im, const uint32_t xyzct[5], const uint32_t blockSize[5], uint8_t headerVersion, uint8_t Nnum,
                      uint8_t* storedHeaderVersion, uint64_t* blockOffset, uint64_t numBlocks, const void** d_payload, uint64_t* payload_bytes)
try {
	LFM_API_LOCK();
	klb_image_header h;
	h.setHeader(xyzct, KLB_DATA_TYPE::UINT16_TYPE, NULL, blockSize, KLB_COMPRESSION_TYPE::BZIP2, NULL, headerVersion, Nnum);
	int rc = validate(h, true);
	if (rc) return rc;
	if (current_ndev() <= 0) return LFM_ERR_CUDA;
	for (int d = 0; d < 5; d++) h.blockSize[d] = std::min(h.blockSize[d], h.xyzct[d]);
	const Layout L = make_layout(h);
	if (numBlocks != L.Nb) return LFM_ERR_OPEN;
	const int way = current_way();
	const StackDesc desc = make_desc(h, way);
	Engine& e = Engine::for_device(g_set.first_device);
	cudaSetDevice(e.device());
	memset(&g_stats, 0, sizeof(g_stats));
	const int video = (headerVersion & 0x80) ? 1 : 0;
	int k;
	if ((headerVersion & 0x7F) < NUM_PREDICTORS) {
		const double t0 = now_ms();
		rc = e.select_mode((const uint16_t*)d_im, desc, g_stats.entropy, &k);
		if (rc) return rc;
		g_stats.ms_select = now_ms() - t0;
		g_stats.selected = 1; g_stats.gpu_launches += 12;
	} else { k = headerVersion & 0x77 & 0x7F; if (k > 7) return LFM_ERR_UNSUPPORTED; }
	if (k != 0 && video && way != 0) return LFM_ERR_UNSUPPORTED;
	if (storedHeaderVersion) *storedHeaderVersion = (uint8_t)((headerVersion & 0x80) | k);
	g_stats.predictor = k;
	static thread_local DevMem* symbuf = nullptr; static thread_local size_t symcap = 0;
	const uint16_t* sym = (const uint16_t*)d_im;
	CompressStats st;
	if (k != 0) {
		size_t need = L.F * L.fpx * 2;
		if (!symbuf || symcap < need) { delete symbuf; symbuf = new DevMem(); if (symbuf->alloc(need)) { delete symbuf; symbuf = nullptr; symcap = 0; return LFM_ERR_CUDA; } symcap = need; }
		rc = e.predict((const uint16_t*)d_im, (uint16_t*)symbuf->p, desc, k, video, 0, (uint32_t)L.F);
		if (rc) return rc;
		st.launches++;
		sym = (const uint16_t*)symbuf->p;
	}
	std::vector<uint32_t> sizes(L.Nb);
	const uint8_t* dpay = nullptr; uint64_t pb = 0;
	rc = e.compress_blocks(sym, desc, 0, L.Nb, sizes.data(), &dpay, &pb, &st);
	if (rc) { g_err = e.last_error(); return rc; }
	uint64_t acc = 0;
	for (uint64_t i = 0; i < L.Nb; i++) { acc += sizes[i]; blockOffset[i] = acc; }
	*d_payload = dpay; *payload_bytes = pb;
	g_stats.ms_rle = st.ms_rle; g_stats.ms_bwt = st.ms_bwt; g_stats.ms_mtf = st.ms_mtf; g_stats.ms_huff = st.ms_huff;
	if (k != 0) g_stats.ms_predict = e.last_predict_ms();
	g_stats.gpu_launches += st.launches; g_stats.periodic_blocks = st.periodic_blocks; g_stats.payload_bytes = pb;
	return 0;
} LFM_CATCH

int lfmSelectDevice(const void* d_frame0, const uint32_t xy[2], uint8_t Nnum, int* predictor, float entropy[8])
try {
	LFM_API_LOCK();
	if (!d_frame0 || !xy || !predictor || xy[0] == 0 || xy[1] == 0) return LFM_ERR_OPEN;
	if (current_ndev() <= 0) return LFM_ERR_CUDA;
	StackDesc s;
	const uint32_t xyzct[5] = { xy[0], xy[1], 1, 1, 1 };
	for (int d = 0; d < 5; d++) { s.xyzct[d] = xyzct[d]; s.blockSize[d] = xyzct[d]; }
	s.Nnum = Nnum ? Nnum : 1; s.way = current_way();
	Engine& e = Engine::for_device(g_set.first_device);
	cudaSetDevice(e.device());
	memset(&g_stats, 0, sizeof(g_stats));
	float ent[8];
	int k = 0;
	const double t0 = now_ms();
	int rc = e.select_mode((const uint16_t*)d_frame0, s, ent, &k);
	if (rc) { g_err = e.last_error(); return rc; }
	g_stats.ms_select = now_ms() - t0; g_stats.selected = 1; g_stats.predictor = k; g_stats.gpu_launches = 12;
	memcpy(g_stats.entropy, ent, sizeof(ent));
	if (entropy) memcpy(entropy, ent, sizeof(ent));
	*predictor = k;
	return LFM_OK;
} LFM_CATCH

int lfmDecompressDevice(const void* d_payload, const uint64_t* blockOffset, uint64_t numBlocks, const uint32_t xyzct[5],
                        const uint32_t blockSize[5], uint8_t storedHeaderVersion, uint8_t Nnum, void* d_out)
try {
	LFM_API_LOCK();
	klb_image_header h;
	h.setHeader(xyzct, KLB_DATA_TYPE::UINT16_TYPE, NULL, blockSize, KLB_COMPRESSION_TYPE::BZIP2, NULL, storedHeaderVersion, Nnum);
	int rc = validate(h, false);
	if (rc) return rc;
	if (current_ndev() <= 0) return LFM_ERR_CUDA;
	for (int d = 0; d < 5; d++) h.blockSize[d] = std::min(h.blockSize[d], h.xyzct[d]);
	const Layout L = make_layout(h);
	if (numBlocks != L.Nb) return LFM_ERR_OPEN;
	const int way = current_way();
	const StackDesc desc = make_desc(h, way);
	const int k = storedHeaderVersion & 0x7F, video = (storedHeaderVersion & 0x80) ? 1 : 0;
	if (k > 7 || (k != 0 && video && way != 0)) return LFM_ERR_UNSUPPORTED;
	Engine& e = Engine::for_device(g_set.first_device);
	cudaSetDevice(e.device());
	memset(&g_stats, 0, sizeof(g_stats));
	std::vector<uint64_t> ids(L.Nb), beg(L.Nb), end(L.Nb);
	for (uint64_t i = 0; i < L.Nb; i++) { ids[i] = i; beg[i] = i ? blockOffset[i - 1] : 0; end[i] = blockOffset[i]; }
	static thread_local DevMem* symbuf = nullptr; static thread_local size_t symcap = 0;
	uint16_t* sym = (uint16_t*)d_out;
	if (k != 0) {
		size_t need = L.F * L.fpx * 2;
		if (!symbuf || symcap < need) { delete symbuf; symbuf = new DevMem(); if (symbuf->alloc(need)) { delete symbuf; symbuf = nullptr; symcap = 0; return LFM_ERR_CUDA; } symcap = need; }
		sym = (uint16_t*)symbuf->p;
	}
	DecompressStats st;
	rc = e.decompress_blocks((const uint8_t*)d_payload, beg.data(), end.data(), ids.data(), L.Nb, sym, desc, &st);
	if (rc) { g_err = e.last_error(); return rc; }
	if (k != 0) {
		rc = e.unpredict(sym, (uint16_t*)d_out, desc, k, video, 0, (uint32_t)L.F);
		if (rc) return rc;
		st.launches += video ? 2 : 1;
		cudaStreamSynchronize((cudaStream_t)e.stream());
		if (cudaGetLastError() != cudaSuccess) return LFM_ERR_CUDA;
		g_stats.ms_unpredict = e.last_unpredict_ms();
	}
	g_stats.predictor = k;
	g_stats.ms_decode = st.ms_decode; g_stats.ms_imtf = st.ms_imtf; g_stats.ms_ibwt = st.ms_ibwt; g_stats.ms_unrle = st.ms_unrle;
	g_stats.gpu_launches = st.launches;
	return 0;
} LFM_CATCH

// ---- multi-process sharding (one process per GPU, SURVEY.md 8e): compress now, write once the offsets are known
namespace { thread_local std::vector<ShardOut> g_pending; }

int lfmShardCompress(const void* im_local, const uint32_t xyzct_local[5], const uint32_t blockSize[5], uint8_t headerVersion, uint8_t Nnum,
                     uint8_t* storedHeaderVersion, uint32_t* blockSizes, uint64_t numBlocks, uint64_t* payload_bytes)
try {
	LFM_API_LOCK();
	g_pending.clear();
	klb_imageIO io;
	io.header.setHeader(xyzct_local, KLB_DATA_TYPE::UINT16_TYPE, NULL, blockSize, KLB_COMPRESSION_TYPE::BZIP2, NULL, headerVersion, Nnum);
	FrameSource src; src.base = (const uint16_t*)im_local;
	std::vector<ShardOut> shards; std::vector<uint64_t> first;
	int rc = compress_core(src, io.header, shards, first);
	if (rc) return rc;
	if (numBlocks != io.header.Nb) return LFM_ERR_OPEN;
	uint64_t total = 0, prev = 0;
	for (uint64_t i = 0; i < io.header.Nb; i++) { blockSizes[i] = (uint32_t)(io.header.blockOffset[i] - prev); prev = io.header.blockOffset[i]; }
	for (const auto& s : shards) total += s.payload_bytes;
	if (storedHeaderVersion) *storedHeaderVersion = io.header.headerVersion;
	if (payload_bytes) *payload_bytes = total;
	g_pending.swap(shards);
	return LFM_OK;
} LFM_CATCH

int lfmShardWritePayload(const char* filename, uint64_t file_offset)
try {
	LFM_API_LOCK();
	if (!filename || !*filename) return LFM_ERR_OPEN;
	const int fd = open(filename, O_RDWR | O_CREAT, 0666);        // no truncation: ranks write their ranges in any order (O_RDWR: the range is mapped)
	if (fd < 0) return LFM_ERR_CREATE;
	int rc = stream_payload_to_fd(g_pending, fd, file_offset);
	if (close(fd) != 0 && rc == 0) rc = LFM_ERR_CREATE;
	return rc;
} LFM_CATCH

int lfmShardFetchPayload(void* dst, uint64_t capacity)
try {
	LFM_API_LOCK();
	uint64_t total = 0;
	for (const auto& s : g_pending) total += s.payload_bytes;
	if (!dst || capacity < total) return LFM_ERR_CREATE;
	return fetch_payload(g_pending, (uint8_t*)dst);
} LFM_CATCH

int lfmWriteHeader(const char* filename, const uint32_t xyzct[5], const uint32_t blockSize[5], uint8_t storedHeaderVersion, uint8_t Nnum,
                   const uint64_t* blockOffset, uint64_t numBlocks)
try {
	if (!filename || !*filename) return LFM_ERR_OPEN;
	klb_image_header h;
	h.setHeader(xyzct, KLB_DATA_TYPE::UINT16_TYPE, NULL, blockSize, KLB_COMPRESSION_TYPE::BZIP2, NULL, storedHeaderVersion, Nnum);
	for (int d = 0; d < 5; d++) { if (h.xyzct[d] == 0 || h.blockSize[d] == 0) return LFM_ERR_BZIP; h.blockSize[d] = std::min(h.blockSize[d], h.xyzct[d]); }
	if (numBlocks == 0 || numBlocks != h.calculateNumBlocks()) return LFM_ERR_OPEN;
	const int fd = open(filename, O_WRONLY | O_CREAT, 0666);      // no truncation to 0: other ranks may already be writing their payload
	if (fd < 0) return LFM_ERR_CREATE;
	uint8_t fixed[320]; h.packFixed(fixed);
	int rc = write_all(fd, fixed, sizeof(fixed), 0);
	if (rc == 0) rc = write_all(fd, blockOffset, (size_t)numBlocks * 8, sizeof(fixed));
	if (rc == 0 && ftruncate(fd, (off_t)(sizeof(fixed) + numBlocks * 8 + blockOffset[numBlocks - 1])) != 0) rc = LFM_ERR_CREATE;
	if (close(fd) != 0 && rc == 0) rc = LFM_ERR_CREATE;
	return rc;
} LFM_CATCH

/* test hook (no GPU needed): the threaded host copy the staging paths use (pageable <-> pinned memory, mapped file ranges) */
int lfmDebugParMemcpy(void* dst, const void* src, uint64_t n) { if (!dst || !src) return 1; par_memcpy(dst, src, (size_t)n); return 0; }

// ---- standalone bzip2 streams (bz_stream.cu): one stream per call, on the first device of lfmSetDevices
namespace {
int bz2_compress_core(Engine& e, const uint8_t* d_src, uint64_t n, int level, const void** d_out, uint64_t* out_size)
{
	CompressStats st;
	const uint8_t* p = nullptr; uint64_t bytes = 0;
	const int rc = e.bz2_compress(d_src, n, level, &p, &bytes, &st);
	if (rc) { g_err = e.last_error(); return rc; }
	g_stats.ms_rle = st.ms_rle; g_stats.ms_bwt = st.ms_bwt; g_stats.ms_mtf = st.ms_mtf; g_stats.ms_huff = st.ms_huff;
	g_stats.gpu_launches += st.launches; g_stats.payload_bytes = bytes;
	*d_out = p; *out_size = bytes;
	return LFM_OK;
}
}

int lfmBz2CompressDevice(const void* d_src, uint64_t n, int level, const void** d_out, uint64_t* out_size)
try {
	LFM_API_LOCK();
	memset(&g_stats, 0, sizeof(g_stats));
	if ((!d_src && n > 0) || !d_out || !out_size || level < 1 || level > 9) return LFM_ERR_OPEN;
	if (n >= (1ull << 32)) { g_err = "input of 2^32 bytes or more"; return LFM_ERR_UNSUPPORTED; }
	if (current_ndev() <= 0) return LFM_ERR_CUDA;
	Engine& e = Engine::for_device(g_set.first_device);
	cudaSetDevice(e.device());
	if (n > 0) {
		cudaPointerAttributes a;
		if (cudaPointerGetAttributes(&a, d_src) != cudaSuccess) { cudaGetLastError(); return LFM_ERR_OPEN; }
		if (a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) { g_err = "d_src is not device memory"; return LFM_ERR_OPEN; }
		if (a.device != e.device()) { g_err = "d_src is not on the first device of lfmSetDevices"; return LFM_ERR_OPEN; }
	}
	const double t0 = now_ms();
	const int rc = bz2_compress_core(e, (const uint8_t*)d_src, n, level, d_out, out_size);
	g_stats.ms_total = now_ms() - t0;
	return rc;
} LFM_CATCH

int lfmBz2Compress(const void* src, uint64_t n, int level, void* dst, uint64_t capacity, uint64_t* dst_size)
try {
	LFM_API_LOCK();
	memset(&g_stats, 0, sizeof(g_stats));
	if ((!src && n > 0) || !dst_size || level < 1 || level > 9) return LFM_ERR_OPEN;
	if (n >= (1ull << 32)) { g_err = "input of 2^32 bytes or more"; return LFM_ERR_UNSUPPORTED; }
	if (current_ndev() <= 0) return LFM_ERR_CUDA;
	Engine& e = Engine::for_device(g_set.first_device);
	cudaSetDevice(e.device());
	cudaStream_t st = (cudaStream_t)e.stream();
	const double t0 = now_ms();
	uint8_t* d_in = e.bz2_staging(n);
	if (!d_in) { g_err = e.last_error(); return LFM_ERR_CUDA; }
	if (n) cudaMemcpyAsync(d_in, src, n, cudaMemcpyHostToDevice, st);
	cudaStreamSynchronize(st);
	const double t1 = now_ms();
	const void* d_out = nullptr; uint64_t bytes = 0;
	int rc = bz2_compress_core(e, d_in, n, level, &d_out, &bytes);
	g_stats.ms_h2d = t1 - t0;
	if (rc) return rc;
	*dst_size = bytes;
	if (!dst || capacity < bytes) { g_err = "destination buffer too small"; g_stats.ms_total = now_ms() - t0; return LFM_ERR_CREATE; }
	const double t2 = now_ms();
	cudaMemcpyAsync(dst, d_out, bytes, cudaMemcpyDeviceToHost, st);
	cudaStreamSynchronize(st);
	if (cudaGetLastError() != cudaSuccess) { g_err = "copy of the stream to the host failed"; return LFM_ERR_CUDA; }
	g_stats.ms_d2h = now_ms() - t2;
	g_stats.ms_total = now_ms() - t0;
	return LFM_OK;
} LFM_CATCH

namespace {
int bz2_decompress_core(const void* src, uint64_t n, bool on_host, uint8_t* d_dst, uint64_t capacity, const void** d_out, uint64_t* out_size)
{
	if (current_ndev() <= 0) return LFM_ERR_CUDA;
	Engine& e = Engine::for_device(g_set.first_device);
	cudaSetDevice(e.device());
	DecompressStats st;
	const uint8_t* p = nullptr; uint64_t bytes = 0;
	const int rc = e.bz2_decompress(src, n, on_host, d_dst, capacity, &p, &bytes, &st);
	*out_size = bytes;
	if (rc) { g_err = e.last_error(); return rc; }
	g_stats.ms_decode = st.ms_decode; g_stats.ms_unrle = st.ms_unrle;
	g_stats.gpu_launches += st.launches; g_stats.payload_bytes = n;
	*d_out = p;
	return LFM_OK;
}
}

int lfmBz2Decompress(const void* src, uint64_t n, void* dst, uint64_t capacity, uint64_t* dst_size)
try {
	LFM_API_LOCK();
	memset(&g_stats, 0, sizeof(g_stats));
	if ((!src && n > 0) || !dst_size || (!dst && capacity > 0)) return LFM_ERR_OPEN;
	if (n == 0) { g_err = "empty input"; return LFM_ERR_BZIP; }
	if (n >= (1ull << 32)) { g_err = "input of 2^32 bytes or more"; return LFM_ERR_UNSUPPORTED; }
	const double t0 = now_ms();
	const void* d_out = nullptr; uint64_t bytes = 0;
	int rc = bz2_decompress_core(src, n, true, nullptr, capacity, &d_out, &bytes);
	*dst_size = bytes;
	if (rc) return rc;
	Engine& e = Engine::for_device(g_set.first_device);
	cudaStream_t st = (cudaStream_t)e.stream();
	const double t2 = now_ms();
	if (bytes) cudaMemcpyAsync(dst, d_out, bytes, cudaMemcpyDeviceToHost, st);
	cudaStreamSynchronize(st);
	if (cudaGetLastError() != cudaSuccess) { g_err = "copy of the data to the host failed"; return LFM_ERR_CUDA; }
	g_stats.ms_d2h = now_ms() - t2;
	g_stats.ms_total = now_ms() - t0;
	return LFM_OK;
} LFM_CATCH

int lfmBz2DecompressDevice(const void* d_src, uint64_t n, void* d_dst, uint64_t capacity, uint64_t* dst_size)
try {
	LFM_API_LOCK();
	memset(&g_stats, 0, sizeof(g_stats));
	if ((!d_src && n > 0) || !dst_size || (!d_dst && capacity > 0)) return LFM_ERR_OPEN;
	if (n == 0) { g_err = "empty input"; return LFM_ERR_BZIP; }
	if (n >= (1ull << 32)) { g_err = "input of 2^32 bytes or more"; return LFM_ERR_UNSUPPORTED; }
	const double t0 = now_ms();
	const void* d_out = nullptr;
	const int rc = bz2_decompress_core(d_src, n, false, (uint8_t*)d_dst, capacity, &d_out, dst_size);
	g_stats.ms_total = now_ms() - t0;
	return rc;
} LFM_CATCH

int lfmGetLastStats(lfm_stats* out) { if (!out) return 1; *out = g_stats; return 0; }
const char* lfmLastError(void) { return g_err.c_str(); }

int lfmDebugPredictDevice(const void* d_in, void* d_out, const uint32_t xyzct[5], uint8_t Nnum, int k, int video, int inverse,
                          int reps, float* ms_per_rep)
try {
	LFM_API_LOCK();
	if (current_ndev() <= 0) return LFM_ERR_CUDA;
	if (reps < 1 || !ms_per_rep) return LFM_ERR_OPEN;
	Engine& e = Engine::for_device(g_set.first_device);
	cudaSetDevice(e.device());
	StackDesc s;
	for (int d = 0; d < 5; d++) { s.xyzct[d] = xyzct[d]; s.blockSize[d] = xyzct[d]; }
	s.Nnum = Nnum ? Nnum : 1; s.way = current_way();
	const uint32_t F = xyzct[2] * xyzct[3] * xyzct[4];
	cudaStream_t st = (cudaStream_t)e.stream();
	cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
	int rc = 0;
	cudaEventRecord(a, st);
	for (int r = 0; r < reps && rc == 0; r++)
		rc = inverse ? e.unpredict((const uint16_t*)d_in, (uint16_t*)d_out, s, k, video, 0, F)
		             : e.predict((const uint16_t*)d_in, (uint16_t*)d_out, s, k, video, 0, F);
	cudaEventRecord(b, st);
	cudaStreamSynchronize(st);
	float ms = 0.f;
	if (rc == 0 && cudaEventElapsedTime(&ms, a, b) != cudaSuccess) { cudaGetLastError(); rc = LFM_ERR_CUDA; }
	cudaEventDestroy(a); cudaEventDestroy(b);
	*ms_per_rep = ms / (float)reps;
	return rc;
} LFM_CATCH

int lfmDebugEncodeBlock(const void* bytes, uint32_t n, uint8_t* rle1, uint8_t* bwt, uint16_t* mtfv, uint8_t* stream, uint32_t info[8])
try {
	LFM_API_LOCK();
	if (n == 0 || (n & 1)) return LFM_ERR_OPEN;
	if (current_ndev() <= 0) return LFM_ERR_CUDA;
	Engine& e = Engine::for_device(g_set.first_device);
	cudaSetDevice(e.device());
	StackDesc s;
	const uint32_t xyzct[5] = { n / 2, 1, 1, 1, 1 };
	for (int d = 0; d < 5; d++) { s.xyzct[d] = xyzct[d]; s.blockSize[d] = xyzct[d]; }
	s.Nnum = 13; s.way = 0;
	DevMem dimg;
	if (dimg.alloc(n)) return LFM_ERR_CUDA;
	cudaMemcpyAsync(dimg.p, bytes, n, cudaMemcpyHostToDevice, (cudaStream_t)e.stream());
	uint32_t size = 0; const uint8_t* dpay = nullptr; uint64_t pb = 0;
	int rc = e.compress_blocks((const uint16_t*)dimg.p, s, 0, 1, &size, &dpay, &pb, nullptr);
	if (rc) { g_err = e.last_error(); return rc; }
	Engine::EncodeTrace t;
	rc = e.fetch_encode_trace(t);
	if (rc) return rc;
	const uint32_t* J = (const uint32_t*)t.jobs.data();   // EncJob fields in declaration order
	const uint32_t nblock = J[1];
	memcpy(rle1, t.txt.data(), nblock); memcpy(bwt, t.bwt.data(), nblock);
	memcpy(mtfv, t.mtfv.data(), (size_t)J[4] * 2);
	cudaMemcpyAsync(stream, dpay, pb, cudaMemcpyDeviceToHost, (cudaStream_t)e.stream());
	cudaStreamSynchronize((cudaStream_t)e.stream());
	info[0] = nblock; info[1] = J[2]; info[2] = J[3]; info[3] = J[5]; info[4] = J[4]; info[5] = J[6]; info[6] = J[7]; info[7] = (uint32_t)pb;
	return 0;
} LFM_CATCH

}  // extern "C"
