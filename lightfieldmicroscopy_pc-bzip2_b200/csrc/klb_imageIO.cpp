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
#include <system_error>
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
inline size_t stage_chunk(size_t bytes) { return bytes >= ((size_t)64 << 20) ? kStageChunk : kStageMin; }

// pageable source: through `ring` (kStageBufs * kStageChunk pinned bytes); pinned / registered / device memory, or no ring: one copy
static void h2d_ring(uint8_t* ring, void* dst, const void* src, size_t bytes, cudaStream_t st)
{
	uint8_t* pin = (ring && bytes >= kStageMin && is_pageable(src)) ? ring : nullptr;
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
	cudaStreamSynchronize(st);                                   // the ring is free again when this returns
	for (auto& x : ev) cudaEventDestroy(x);
}
void h2d_staged(Engine& e, void* dst, const void* src, size_t bytes, cudaStream_t st)
{
	const bool staged = bytes >= kStageMin && is_pageable(src);        // the engine's ring is only allocated when it is needed
	h2d_ring(staged ? (uint8_t*)e.pinned(kStageBufs * kStageChunk, 0) : nullptr, dst, src, bytes, st);
}

// pageable destination: through `ring` (kStageBufs * kStageChunk pinned bytes); pinned / registered memory, or no ring: one copy
static void d2h_ring(uint8_t* ring, void* dst, const void* src, size_t bytes, cudaStream_t st)
{
	uint8_t* pin = (ring && bytes >= kStageMin && is_pageable(dst)) ? ring : nullptr;
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
void d2h_staged(Engine& e, void* dst, const void* src, size_t bytes, cudaStream_t st)
{
	const bool staged = bytes >= kStageMin && is_pageable(dst);
	d2h_ring(staged ? (uint8_t*)e.pinned(kStageBufs * kStageChunk, 1) : nullptr, dst, src, bytes, st);
}

// ------------------------------------------------------------------------------------------------ compress core
struct ShardOut {
	std::vector<uint32_t> sizes; int rc = 0; CompressStats st; double ms_h2d = 0, ms_d2h = 0; std::string err;
	const uint8_t* d_payload = nullptr; uint64_t payload_bytes = 0; int device = 0;      // streams stay on the GPU until fetched
};
enum { UB_IMG = 0, UB_SYM = 1, UB_PAY = 2, UB_F0 = 3 };

// ------------------------------------------------------------------------------------------------ stack writer (one GPU)
// A recording is compressed in batches of whole z-slabs as its frames arrive (DESIGN.md §4c): lfmStackWriterAppend copies frames
// into one of two batch image buffers (pinned staging ring + upload stream), a worker thread predicts and compresses every
// complete batch on the engine under the API lock, and a file thread streams its payload to its final offset behind the
// blockOffset table of the declared stack (pinned ring + download stream + pwrite) while the next batch fills.  Large stacks of
// writeLFMstackEx / writeLFMstackDevice go through the same writer (write_stack_with_writer).  Everything a writer needs
// between two calls is its own (PipeRes): other calls may use the engine's buffers, pinned slots and streams in between.
constexpr uint64_t kBatchBytes = (uint64_t)96 << 20;               // raw bytes per batch (at least one slab)
constexpr uint64_t kBatchBlocks = 2048;                            // ... and at least this many KLB blocks

static int payload_to_fd(uint8_t* pin, const uint8_t* d_payload, uint64_t bytes, int fd, uint64_t file_off, cudaStream_t st)
{
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
		rc = write_all(fd, pin + (i % kStageBufs) * kStageChunk, len, file_off + o);
	}
	cudaStreamSynchronize(st);
	for (auto& x : ev) cudaEventDestroy(x);
	return rc;
}

// slabs per batch of a stack written or read in batches (at least; batch_cuts may make a batch longer)
static uint64_t batch_slabs(const klb_image_header& h, const Layout& L)
{
	const uint64_t batch_bytes = env_int("LFM_B200_BATCH_KB", 0) > 0 ? (uint64_t)env_int("LFM_B200_BATCH_KB", 0) << 10 : kBatchBytes;   // test knob
	const uint64_t slab_bytes = (uint64_t)h.blockSize[2] * L.fpx * 2;
	uint64_t n = std::max<uint64_t>(1, batch_bytes / std::max<uint64_t>(1, slab_bytes));
	// the block codec kernels are latency bound: a batch needs a few thousand KLB blocks to fill the GPU (k_huff_decode alone keeps
	// ~1500 streams in flight), or the overlap won is lost again in half-empty kernels
	if (env_int("LFM_B200_BATCH_KB", 0) <= 0) n = std::max<uint64_t>(n, (kBatchBlocks + L.blocksPerSlab - 1) / L.blocksPerSlab);
	return n;
}
// slabs per batch of the pipelined paths; 0 when the stack is not worth / not fit for batching (few slabs, c or t blocked)
static uint64_t slabs_per_batch(const klb_image_header& h, const Layout& L)
{
	if (env_int("LFM_B200_NO_PIPELINE", 0) || h.blockSize[3] != 1 || h.blockSize[4] != 1) return 0;
	const uint64_t n = batch_slabs(h, L);
	return L.nSlabs >= 2 * n ? n : 0;
}
// first flattened frame of slab s (c and t not blocked: the slabs tile the frames in order); L.F past the last slab
static uint64_t slab_first_frame(const klb_image_header& h, const Layout& L, uint64_t s)
{
	return s >= L.nSlabs ? L.F : (s / L.nb[2]) * h.xyzct[2] + (s % L.nb[2]) * h.blockSize[2];
}
// Batch boundaries of slabs [s_begin, s_end): cut[0] = s_begin, cut.back() = s_end, at least `per` slabs apart.  With pair_frames (video stack +
// predictor: an odd frame is predicted from the even frame before it) a batch only starts on a slab whose first frame is even, so
// that it holds the frame each of its odd frames needs; a cut moves forward to the next such slab.  Slab s starts at frame
// (s / nb[2]) * Z + (s % nb[2]) * blockSize[2]: with Z not a multiple of the block depth and c or t above 1, slabs in the middle of
// the stack start on odd frames whatever the batch length (with Z odd and an even depth, every slab of an odd volume does).
static std::vector<uint64_t> batch_cuts(const klb_image_header& h, const Layout& L, uint64_t per, bool pair_frames,
                                        uint64_t s_begin, uint64_t s_end)
{
	std::vector<uint64_t> cut(1, s_begin);
	for (;;) {
		uint64_t c = cut.back() + per;
		while (pair_frames && c < s_end && (slab_first_frame(h, L, c) & 1)) c++;
		if (c >= s_end) break;
		cut.push_back(c);
	}
	cut.push_back(s_end);
	return cut;
}

struct PipeRes {                  // device memory, pinned staging rings and copy streams of one open writer or reader
	int dev = -1;
	Engine::Buf img[2], sym, pay[2], stage;     // stage: a reader's cropped frames on their way to host memory
	uint8_t* up_pin = nullptr;    // kStageBufs * kStageChunk bytes each
	uint8_t* down_pin = nullptr;
	cudaStream_t up_st = nullptr, down_st = nullptr;
	int init(int device)
	{
		dev = device;
		cudaSetDevice(dev);
		if (cudaStreamCreateWithFlags(&up_st, cudaStreamNonBlocking) != cudaSuccess || cudaStreamCreateWithFlags(&down_st, cudaStreamNonBlocking) != cudaSuccess ||
		    cudaHostAlloc((void**)&up_pin, kStageBufs * kStageChunk, cudaHostAllocDefault) != cudaSuccess ||
		    cudaHostAlloc((void**)&down_pin, kStageBufs * kStageChunk, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return LFM_ERR_CUDA; }
		return LFM_OK;
	}
	~PipeRes()
	{
		if (dev < 0) return;
		DeviceGuard g;
		cudaSetDevice(dev);
		for (Engine::Buf* b : { &img[0], &img[1], &sym, &pay[0], &pay[1], &stage }) if (b->p) cudaFree(b->p);
		if (up_pin) cudaFreeHost(up_pin);
		if (down_pin) cudaFreeHost(down_pin);
		if (up_st) cudaStreamDestroy(up_st);
		if (down_st) cudaStreamDestroy(down_st);
	}
};
// The resources of the last closed writer or reader wait for the next one on the same device: writeLFMstackEx and full reads open
// one per large stack, and pinning 64 MB of staging memory costs more than a batch.  Never destroyed (CUDA may be gone at exit).
std::mutex g_spare_mu;
PipeRes* g_spare = nullptr;
PipeRes* take_res(int dev)
{
	std::lock_guard<std::mutex> lk(g_spare_mu);
	PipeRes* r = g_spare;
	if (r && r->dev == dev) { g_spare = nullptr; return r; }
	return nullptr;
}
void give_res(PipeRes* r)
{
	std::lock_guard<std::mutex> lk(g_spare_mu);
	std::swap(r, g_spare);
	delete r;
}
}  // namespace

struct lfm_stack_writer {
	klb_image_header h;               // the declared recording (blockSize clamped); headerVersion stored once the predictor is known
	int fd = -1;
	uint8_t hv_in = 0;
	int video = 0, k = -1;            // k: predictor, -1 until frame 0 has been through mode selection
	Layout L;
	StackDesc desc;
	std::vector<uint64_t> cut;        // batch b = slabs [cut[b], cut[b + 1]) (batch_cuts)
	uint64_t nbatch = 0, base = 0;    // batches, file offset of payload byte 0 (declared table)
	Engine* e = nullptr;
	PipeRes* res = nullptr;
	uint64_t received = 0;            // frames taken by Append (calling thread only)
	std::mutex mu;                    // guards the fields below
	std::condition_variable cv;
	uint64_t ready = 0, computed = 0; // batches whose frames are all on the GPU / that are predicted and compressed
	bool closing = false;
	int rc = LFM_OK;                  // first failure: the writer is failed from then on
	std::string err;
	std::thread worker, wr_th[2];     // wr_th[i]: the payload of the last batch compressed into res->pay[i] on its way to the file
	int wr_rc[2] = { 0, 0 };
	uint64_t pay_off = 0;             // payload bytes of the batches compressed so far (worker thread)
	lfm_stats st;
	double t_open = 0;

	int fail(int code, const std::string& what)
	{
		std::lock_guard<std::mutex> lk(mu);
		if (!rc) { rc = code; err = what; }
		cv.notify_all();
		return rc;
	}
	int failed() { std::lock_guard<std::mutex> lk(mu); return rc; }
	uint64_t batch_of_frame(uint64_t f) const
	{
		const uint64_t s = (f / h.xyzct[2]) * L.nb[2] + (f % h.xyzct[2]) / h.blockSize[2];
		return (uint64_t)(std::upper_bound(cut.begin(), cut.end(), s) - cut.begin()) - 1;
	}
	uint64_t batch_first_frame(uint64_t b) const { return slab_first_frame(h, L, cut[b]); }
	// predict + compress slabs [s0, s1) of image buffer `slot`, whose first frame is slab s0's, as the stack `d` (the declared one,
	// or at an early close the kept prefix); block sizes -> h.blockOffset (kept blocks are a prefix of the declared ones)
	int compress(const StackDesc& d, const klb_image_header& hd, const Layout& Ld, uint64_t s0, uint64_t s1, int slot,
	             const uint8_t** dpay, uint64_t* pbytes)
	{
		LFM_API_LOCK();
		cudaSetDevice(e->device());
		const uint64_t f0 = slab_first_frame(hd, Ld, s0), nf = slab_first_frame(hd, Ld, s1) - f0;
		const uint16_t* img_base = (const uint16_t*)res->img[slot].p - f0 * L.fpx;     // virtual base: absolute frame indexing
		const uint16_t* sym_base = img_base;
		CompressStats cs;
		int r;
		if (k != 0) {
			uint16_t* sb = (uint16_t*)res->sym.p - f0 * L.fpx;
			if ((r = e->predict(img_base, sb, d, k, video, (uint32_t)f0, (uint32_t)nf))) return fail(r, "predictor launch failed");
			cs.launches++;
			sym_base = sb;
		}
		const uint64_t first = s0 * L.blocksPerSlab, count = (s1 - s0) * L.blocksPerSlab;
		std::vector<uint32_t> sizes(count);
		if ((r = e->compress_blocks(sym_base, d, first, count, sizes.data(), dpay, pbytes, &cs, &res->pay[slot]))) return fail(r, e->last_error());
		if (k != 0) st.ms_predict += e->last_predict_ms();
		uint64_t acc = first ? h.blockOffset[first - 1] : 0;
		for (uint64_t i = 0; i < count; i++) { acc += sizes[i]; h.blockOffset[first + i] = acc; }
		st.ms_rle += cs.ms_rle; st.ms_bwt += cs.ms_bwt; st.ms_mtf += cs.ms_mtf; st.ms_huff += cs.ms_huff;
		st.gpu_launches += cs.launches; st.periodic_blocks += cs.periodic_blocks;
		return LFM_OK;
	}
	// the worker: every batch once all its frames are on the GPU; its payload leaves on a file thread while the next one computes
	void run()
	{
		try { run_batches(); }
		catch (const std::bad_alloc&) { fail(LFM_ERR_CREATE, "out of host memory"); }
		catch (const std::exception& ex) { fail(LFM_ERR_BZIP, ex.what()); }
		for (int i = 0; i < 2; i++) if (wr_th[i].joinable()) { wr_th[i].join(); if (wr_rc[i]) fail(wr_rc[i], "payload write failed"); }
	}
	void run_batches()
	{
		cudaSetDevice(res->dev);
		for (uint64_t b = 0; b < nbatch; b++) {
			{
				std::unique_lock<std::mutex> lk(mu);
				cv.wait(lk, [&] { return ready > b || closing || rc; });
				if (rc || ready <= b) break;
			}
			const int slot = (int)(b & 1);
			if (wr_th[slot].joinable()) { wr_th[slot].join(); if (wr_rc[slot]) { fail(wr_rc[slot], "payload write failed"); break; } }
			const uint8_t* dpay = nullptr; uint64_t pbytes = 0;
			if (compress(desc, h, L, cut[b], cut[b + 1], slot, &dpay, &pbytes)) break;
			{ std::lock_guard<std::mutex> lk(mu); computed = b + 1; }
			cv.notify_all();                                            // image buffer `slot` is free for batch b + 2
			// one file thread at a time (they share the download ring and stream)
			if (wr_th[slot ^ 1].joinable()) { wr_th[slot ^ 1].join(); if (wr_rc[slot ^ 1]) { fail(wr_rc[slot ^ 1], "payload write failed"); break; } }
			const uint64_t at = base + pay_off;
			wr_th[slot] = std::thread([this, slot, dpay, pbytes, at]() {
				cudaSetDevice(res->dev);
				try { wr_rc[slot] = pbytes ? payload_to_fd(res->down_pin, dpay, pbytes, fd, at, res->down_st) : LFM_OK; }
				catch (const std::exception&) { wr_rc[slot] = LFM_ERR_CREATE; }
			});
			pay_off += pbytes;
		}
	}
};

namespace {
// xyzct / blockSize of `h` checked as writeLFMstackEx checks them, plus what a writer cannot do; `h` comes back clamped
int writer_open(lfm_stack_writer** out, const std::string& filename, const klb_image_header& h_in)
{
	*out = nullptr;
	klb_image_header h(h_in);
	int rc = validate(h, true);
	if (rc) return rc;
	if (current_ndev() <= 0) { std::cout << "ERROR: lfm_b200: no CUDA device available (this engine has no CPU fallback)" << std::endl; return LFM_ERR_CUDA; }
	for (int d = 0; d < 5; d++) h.blockSize[d] = std::min(h.blockSize[d], h.xyzct[d]);     // src/klb_imageIO.cpp:2407-2408
	if (h.blockSize[3] != 1 || h.blockSize[4] != 1) {
		g_err = "blocks over several channels or time points span frames that do not arrive one after the other"; return LFM_ERR_UNSUPPORTED;
	}
	const uint8_t hv = h.headerVersion;
	const int video = (hv & 0x80) ? 1 : 0, way = current_way();
	int k = -1;
	if ((hv & 0x7F) >= NUM_PREDICTORS) {
		k = hv & 0x77 & 0x7F;                          // `hv & 0x7F - 8` parses as hv & 0x77 (src/klb_imageIO.cpp:2380)
		if (k > 7) { std::cout << "ERROR: The predictors hava not selected!" << std::endl; return LFM_ERR_UNSUPPORTED; }
		if (k != 0 && video && way != 0) {
			std::cout << "ERROR: lfm_b200: video stacks are only invertible with predictor way 0 (tiles); refusing to write" << std::endl;
			return LFM_ERR_UNSUPPORTED;
		}
	}
	std::unique_ptr<lfm_stack_writer> w(new lfm_stack_writer);
	w->t_open = now_ms();
	memset(&w->st, 0, sizeof(w->st));
	w->L = make_layout(h);
	h.resizeBlockOffset(w->L.Nb);
	w->h = h;
	w->hv_in = hv; w->video = video; w->k = k;
	w->desc = make_desc(h, way);
	// the predictor is not known before frame 0 with auto-selection: video batches start on even frames in any case
	w->cut = batch_cuts(h, w->L, batch_slabs(h, w->L), video != 0, 0, w->L.nSlabs);
	w->nbatch = w->cut.size() - 1;
	uint64_t max_nf = 0;
	for (uint64_t b = 0; b < w->nbatch; b++) max_nf = std::max(max_nf, w->batch_first_frame(b + 1) - w->batch_first_frame(b));
	w->base = 320 + w->L.Nb * sizeof(uint64_t);
	w->e = &Engine::for_device(g_set.first_device);
	const int dev = w->e->device();
	cudaSetDevice(dev);
	std::unique_ptr<PipeRes> res(take_res(dev));
	if (!res) { res.reset(new PipeRes); if (res->init(dev)) { g_err = "pinned staging memory or copy streams could not be allocated"; return LFM_ERR_CUDA; } }
	const size_t img_bytes = (size_t)max_nf * w->L.fpx * 2;
	if (w->e->reserve(res->img[0], img_bytes) || w->e->reserve(res->img[1], img_bytes) || (k > 0 && w->e->reserve(res->sym, img_bytes))) {
		give_res(res.release()); g_err = "batch buffers could not be allocated"; return LFM_ERR_CUDA;
	}
	const bool existed = access(filename.c_str(), F_OK) == 0;
	const int fd = open(filename.c_str(), O_RDWR | O_CREAT, 0666);
	if (fd < 0) { give_res(res.release()); std::cout << "ERROR: file " << filename << " could not be opened" << std::endl; return LFM_ERR_CREATE; }
	// an existing file is overwritten in place (its pages are kept) and cut to size at Close; until then its old header must not
	// make it look like a valid .lfm file
	uint8_t zero[320] = { 0 };
	struct stat sb;
	if (fstat(fd, &sb) == 0 && sb.st_size > 0 && write_all(fd, zero, std::min<size_t>(sizeof(zero), (size_t)sb.st_size), 0)) {
		close(fd); give_res(res.release()); return LFM_ERR_CREATE;
	}
	w->fd = fd;
	w->res = res.release();
	lfm_stack_writer* p = w.get();
	try { w->worker = std::thread([p]() { p->run(); }); }
	catch (const std::system_error&) {
		close(fd); if (!existed) unlink(filename.c_str());
		give_res(w->res); g_err = "the writer thread could not be started"; return LFM_ERR_CREATE;
	}
	*out = w.release();
	return LFM_OK;
}

int writer_append(lfm_stack_writer* w, const void* frames, uint64_t n, bool device)
{
	if (int r = w->failed()) { g_err = w->err; return r; }
	if (n == 0) return LFM_OK;
	if (w->received + n > w->L.F || w->received + n < n) {
		g_err = "append past the declared frame count (" + std::to_string(w->L.F) + " frames)"; return LFM_ERR_OPEN;
	}
	int rc = LFM_OK;
	if (!frames) w->fail(LFM_ERR_OPEN, "frames is NULL");
	else if (device && (rc = check_device_ptr(frames, "d_frames"))) w->fail(rc, g_err);
	if (int r = w->failed()) { g_err = w->err; return r; }
	PipeRes& R = *w->res;
	cudaSetDevice(R.dev);
	const size_t frame_bytes = (size_t)w->L.fpx * 2;
	const uint8_t* src = (const uint8_t*)frames;
	uint64_t f = w->received;
	const uint64_t end = w->received + n;
	while (f < end) {
		const uint64_t b = w->batch_of_frame(f), f0 = w->batch_first_frame(b), f1 = w->batch_first_frame(b + 1);
		const int slot = (int)(b & 1);
		{
			// back-pressure: image buffer `slot` is free once batch b - 2 has been compressed
			std::unique_lock<std::mutex> lk(w->mu);
			w->cv.wait(lk, [&] { return b < 2 || w->computed >= b - 1 || w->rc; });
			if (w->rc) break;
		}
		const uint64_t m = std::min(f1, end) - f;
		uint8_t* dst = (uint8_t*)R.img[slot].p + (f - f0) * frame_bytes;
		if (device) cudaMemcpyAsync(dst, src, m * frame_bytes, cudaMemcpyDeviceToDevice, R.up_st);
		else h2d_ring(R.up_pin, dst, src, m * frame_bytes, R.up_st);
		const bool batch_done = f + m == f1;
		if ((f == 0 || batch_done) && cudaStreamSynchronize(R.up_st) != cudaSuccess) { cudaGetLastError(); w->fail(LFM_ERR_CUDA, "frame upload failed"); break; }
		if (f == 0 && w->k < 0) {
			// mode selection on frame 0 (branches A and B of writeImage, src/klb_imageIO.cpp:2273-2377)
			LFM_API_LOCK();
			const double t0 = now_ms();
			int k = 0;
			if ((rc = w->e->select_mode((const uint16_t*)R.img[0].p, w->desc, w->st.entropy, &k))) { w->fail(rc, w->e->last_error()); break; }
			w->st.ms_select = now_ms() - t0;
			w->st.selected = 1; w->st.gpu_launches += 7 + 5;       // 7 candidate predictions + the selection (memset, walk, link, entropy: counted as 5, as bench.py does)
			if (k != 0 && w->video && w->desc.way != 0) {
				std::cout << "ERROR: lfm_b200: video stacks are only invertible with predictor way 0 (tiles); refusing to write" << std::endl;
				w->fail(LFM_ERR_UNSUPPORTED, "video stacks are only invertible with predictor way 0"); break;
			}
			if (k != 0 && w->e->reserve(R.sym, R.img[0].cap)) { w->fail(LFM_ERR_CUDA, "symbol buffer could not be allocated"); break; }
			w->k = k;
		}
		if (f == 0) {
			w->h.headerVersion = (uint8_t)((w->hv_in & 0x80) | w->k);
			w->st.predictor = w->k;
		}
		f += m; src += m * frame_bytes;
		if (batch_done) {
			{ std::lock_guard<std::mutex> lk(w->mu); w->ready = b + 1; }
			w->cv.notify_all();
		}
	}
	// the caller may reuse its buffer when this returns: a pinned or device source is read by copies still in flight
	if (cudaStreamSynchronize(R.up_st) != cudaSuccess) { cudaGetLastError(); w->fail(LFM_ERR_CUDA, "frame upload failed"); }
	w->received = f;
	if (int r = w->failed()) { g_err = w->err; return r; }
	return LFM_OK;
}

// the kept prefix of an early close: whole steps of the slowest of z, c, t with more than one entry; its last partial batch is
// compressed here, the payload already in the file moves left by the table entries it no longer needs
int writer_finish(lfm_stack_writer* w, uint64_t* kept_out)
{
	const klb_image_header& H = w->h;
	const Layout& L = w->L;
	int d = 2; uint64_t u = 1;
	if (H.xyzct[4] > 1) { d = 4; u = (uint64_t)H.xyzct[2] * H.xyzct[3]; }
	else if (H.xyzct[3] > 1) { d = 3; u = H.xyzct[2]; }
	const uint64_t kept = w->received / u * u;
	*kept_out = kept;
	if (kept == 0) { g_err = "no frame was recorded"; return LFM_ERR_BZIP; }
	klb_image_header h2(H);
	const uint64_t done_slabs = w->cut[w->computed];
	Layout L2 = L;
	if (kept < L.F) {
		h2.xyzct[d] = (uint32_t)(kept / u);
		for (int i = 0; i < 5; i++) h2.blockSize[i] = std::min(h2.blockSize[i], h2.xyzct[i]);
		L2 = make_layout(h2);
	}
	const uint64_t done = std::min(done_slabs, L2.nSlabs);
	uint64_t bytes = done ? H.blockOffset[done * L.blocksPerSlab - 1] : 0;     // payload of the kept blocks already in the file
	int rc = LFM_OK;
	if (done < L2.nSlabs) {
		// the tail: slabs [done, kept) sit in the image buffer of batch `computed`, which starts at slab `done`
		const StackDesc d2 = make_desc(h2, w->desc.way);
		const int slot = (int)(w->computed & 1);
		const uint8_t* dpay = nullptr; uint64_t pbytes = 0;
		if ((rc = w->compress(d2, h2, L2, done, L2.nSlabs, slot, &dpay, &pbytes))) return rc;
		cudaSetDevice(w->res->dev);
		if (pbytes && (rc = payload_to_fd(w->res->down_pin, dpay, pbytes, w->fd, w->base + bytes, w->res->down_st))) return rc;
		bytes += pbytes;
	}
	h2.resizeBlockOffset(L2.Nb);
	memcpy(h2.blockOffset, H.blockOffset, L2.Nb * sizeof(uint64_t));
	const uint64_t base2 = 320 + L2.Nb * sizeof(uint64_t);
	// front to back: the destination lies before the source
	for (uint64_t o = 0; base2 != w->base && o < bytes; o += kStageBufs * kStageChunk) {
		const size_t len = (size_t)std::min<uint64_t>(kStageBufs * kStageChunk, bytes - o);
		if ((rc = read_all(w->fd, w->res->down_pin, len, w->base + o))) return LFM_ERR_CREATE;
		if ((rc = write_all(w->fd, w->res->down_pin, len, base2 + o))) return rc;
	}
	uint8_t fixed[320]; h2.packFixed(fixed);
	if ((rc = write_all(w->fd, fixed, sizeof(fixed), 0)) || (rc = write_all(w->fd, h2.blockOffset, L2.Nb * sizeof(uint64_t), sizeof(fixed)))) return rc;
	if (ftruncate(w->fd, (off_t)(base2 + bytes)) != 0) return LFM_ERR_CREATE;
	w->st.payload_bytes = bytes;
	w->h = h2;
	return LFM_OK;
}

// finishes the file (or cuts it to 0 bytes after a failure), frees w; the recording's statistics become the calling thread's
int writer_close(lfm_stack_writer* w, uint64_t* frames_kept, klb_image_header* h_out = nullptr)
{
	{ std::lock_guard<std::mutex> lk(w->mu); w->closing = true; }
	w->cv.notify_all();
	w->worker.join();
	uint64_t kept = 0;
	int rc = w->rc;
	std::string err = w->err;
	if (!rc) rc = writer_finish(w, &kept);
	if (rc && ftruncate(w->fd, 0) != 0) { /* nothing more to do */ }
	if (close(w->fd) != 0 && !rc) rc = LFM_ERR_CREATE;
	if (frames_kept) *frames_kept = rc ? 0 : kept;
	w->st.ms_total = now_ms() - w->t_open;
	g_stats = w->st;
	if (w->rc) g_err = err;
	if (!rc && h_out) *h_out = w->h;
	give_res(w->res);
	delete w;
	return rc;
}

// writeLFMstackEx / writeLFMstackDevice of a stack that fills at least two batches on one GPU: open a writer, append the stack, close
bool takes_writer(const FrameSource& src, const klb_image_header& header)
{
	klb_image_header h(header);
	if ((h.compressionType != KLB_COMPRESSION_TYPE::BZIP2 && h.compressionType != KLB_COMPRESSION_TYPE::NONE) || h.getBytesPerPixel() != 2) return false;
	for (int d = 0; d < 5; d++) { if (h.xyzct[d] == 0 || h.blockSize[d] == 0) return false; h.blockSize[d] = std::min(h.blockSize[d], h.xyzct[d]); }
	const int ndev = current_ndev();
	if (ndev <= 0) return false;
	const Layout L = make_layout(h);
	if (!src.device && std::min<uint64_t>((uint64_t)ndev, L.nSlabs) != 1) return false;   // sharded over several GPUs
	return slabs_per_batch(h, L) != 0;
}

int write_stack_with_writer(const std::string& filename, const FrameSource& src, klb_image_header& header)
{
	memset(&g_stats, 0, sizeof(g_stats));
	lfm_stack_writer* w = nullptr;
	int rc = writer_open(&w, filename, header);
	if (rc) {
		// as the one-shot path, which has created the file before it meets the error: an empty file is left
		const int fd = rc == LFM_ERR_CREATE ? -1 : open(filename.c_str(), O_RDWR | O_CREAT | O_TRUNC, 0666);
		if (fd >= 0) close(fd);
		return rc;
	}
	const uint64_t F = w->L.F;
	try {
		if (src.slices) { for (uint64_t f = 0; f < F && rc == LFM_OK; f++) rc = writer_append(w, src.slices[f], 1, false); }
		else rc = writer_append(w, src.base, F, src.device);
	} catch (const std::exception&) { rc = w->fail(LFM_ERR_CREATE, "out of host memory"); }   // the writer is closed all the same
	uint64_t kept = 0;
	const int rc2 = writer_close(w, &kept, &header);
	return rc ? rc : rc2;
}
// Phase 1: everything up to the compacted streams in device memory + header.blockOffset[].
int compress_core(const FrameSource& src, klb_image_header& h, std::vector<ShardOut>& shards, std::vector<uint64_t>& shardFirstBlock)
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
		g_stats.selected = 1; g_stats.gpu_launches += 7 + 5;       // 7 candidate predictions + the selection (memset, walk, link, entropy: counted as 5, as bench.py does)
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
	// go through two halves of the pinned staging ring `pin` (kStageBufs * kStageChunk bytes): chunk i+1 is read from the file while
	// chunk i crosses PCIe.  Returns 0, or LFM_ERR_BZIP on a short read.
	int to_device(uint8_t* pin, void* dst, const std::vector<std::pair<uint64_t, uint64_t>>& ranges, cudaStream_t st) const
	{
		uint64_t dpos = 0;
		if (base) {
			for (const auto& r : ranges) { cudaMemcpyAsync((uint8_t*)dst + dpos, base + r.first, r.second - r.first, cudaMemcpyHostToDevice, st); dpos += r.second - r.first; }
			return LFM_OK;
		}
		uint64_t total = 0;
		for (const auto& r : ranges) total += r.second - r.first;
		const uint64_t CH = total >= ((uint64_t)64 << 20) ? (uint64_t)16 << 20 : (uint64_t)2 << 20;      // two buffers: 16 MB chunks fit the 32 MB ring
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
		cudaStreamSynchronize(st);                                // the staging buffers are free again
		cudaEventDestroy(ev[0]); cudaEventDestroy(ev[1]);
		return rc;
	}
};

// What every read checks of a file's header and table before it decodes anything, in this order; *k, *video: the stored predictor
// and video bit
int check_stack(const klb_image_header& h, uint64_t payload_size, int* k, int* video)
{
	int rc = validate(h, false);
	if (rc) return rc;
	if (current_ndev() <= 0) { std::cout << "ERROR: lfm_b200: no CUDA device available (this engine has no CPU fallback)" << std::endl; return LFM_ERR_CUDA; }
	if (h.Nb == 0) { std::cerr << "ERROR: Image to read has not blocks" << std::endl; return LFM_ERR_BZIP; }
	const Layout L = make_layout(h);
	if (L.Nb != h.Nb) return LFM_ERR_BZIP;
	if (h.blockOffset[L.Nb - 1] > payload_size) { std::cerr << "ERROR: lfm_b200: file is truncated" << std::endl; return LFM_ERR_BZIP; }
	// the table comes from an untrusted file: END offsets must not decrease and none may point past the payload (an ROI read
	// skips blocks, so checking only the last one is not enough)
	for (uint64_t i = 1; i < L.Nb; i++)
		if (h.blockOffset[i] < h.blockOffset[i - 1]) { std::cerr << "ERROR: lfm_b200: corrupt blockOffset table" << std::endl; return LFM_ERR_BZIP; }
	*k = h.headerVersion & 0x7F; *video = (h.headerVersion & 0x80) ? 1 : 0;
	if (*k > 7) return LFM_ERR_UNSUPPORTED;
	if (*k != 0 && *video && current_way() != 0) {
		std::cout << "ERROR: lfm_b200: video stack written with predictor way != 0 cannot be inverted (reference defect, see DESIGN.md)" << std::endl;
		return LFM_ERR_UNSUPPORTED;
	}
	return LFM_OK;
}
// the inclusive box in_lb..in_ub (NULL: the whole stack) -> lb, ub; LFM_ERR_OPEN when it does not lie inside the stack
int check_box(const klb_image_header& h, const uint32_t* in_lb, const uint32_t* in_ub, uint32_t lb[5], uint32_t ub[5], bool* full)
{
	*full = true;
	for (int d = 0; d < 5; d++) {
		lb[d] = in_lb ? in_lb[d] : 0; ub[d] = in_ub ? in_ub[d] : h.xyzct[d] - 1;
		if (ub[d] >= h.xyzct[d] || lb[d] > ub[d]) return LFM_ERR_OPEN;
		if (lb[d] != 0 || ub[d] != h.xyzct[d] - 1) *full = false;
	}
	return LFM_OK;
}
// Block b of a slab (x fastest) is decoded for a read of the box lb..ub.  Without a predictor: the blocks that intersect it.  With
// a predictor: every operand of the prediction rules lies up and/or left of the pixel (lfm_predict.cuh), so a pixel only depends on
// the pixels with x' <= x and y' <= y of its frame (and of the previous frame, video) -> the blocks that start at or before the
// box's lower right corner; what lies right of / below it keeps zero symbols and decodes to values nobody reads.
bool block_needed(const klb_image_header& h, const Layout& L, uint64_t b, const uint32_t lb[5], const uint32_t ub[5], int k)
{
	const uint64_t bx = b % L.nb[0], by = b / L.nb[0];
	const uint64_t x0 = bx * h.blockSize[0], x1 = std::min<uint64_t>(h.xyzct[0], x0 + h.blockSize[0]) - 1;
	const uint64_t y0 = by * h.blockSize[1], y1 = std::min<uint64_t>(h.xyzct[1], y0 + h.blockSize[1]) - 1;
	if (x0 > ub[0] || y0 > ub[1]) return false;
	return k != 0 || (x1 >= lb[0] && y1 >= lb[1]);
}
}  // namespace

// ------------------------------------------------------------------------------------------------ stack reader (one GPU)
// The read side of the slab pipeline (DESIGN.md §4d): the slabs a box touches are decoded in batches of whole z-slabs (batch_cuts)
// and handed out frame by frame.  A fetch thread reads the needed byte ranges of batch b + 2 into payload buffer (b + 2) & 1
// (pinned ring + upload stream), a worker thread decodes and un-predicts batch b + 1 into frame buffer (b + 1) & 1 on the engine
// under the API lock, and lfmStackReaderRead crops the box out of batch b (k_roi_gather on the download stream) into the caller's
// device buffer, or into a staging buffer drained to host memory through the download ring.  Everything a reader needs between
// two calls is its own (PipeRes).  Full reads of large single-GPU stacks go through a reader too (read_with_reader).
struct lfm_stack_reader {
	klb_image_header h;
	Layout L;
	StackDesc desc;
	int k = 0, video = 0;
	bool pair = false;                // video + predictor: an odd frame is predicted from the even frame before it
	uint32_t lb[5], ub[5];
	bool full = false;
	PayloadSource src;
	int own_fd = -1;                  // the file Open opened, closed by Close
	uint64_t frames = 0, box_fpx = 0; // frames of the box, pixels of one cropped frame
	struct Batch { uint64_t s0, s1, f0, f1, u0, u1, i0, i1; };   // slabs [s0, s1) hold frames [f0, f1); [u0, u1) are un-predicted;
	std::vector<Batch> B;                                        // box frames [i0, i1) come from this batch
	uint64_t max_box_frames = 0;      // box frames of the largest batch
	uint16_t* direct = nullptr;       // full read into a 16-byte aligned device buffer: the batches decode straight into it
	Engine* e = nullptr;
	PipeRes* res = nullptr;
	uint64_t pos = 0, cur = 0;        // box frames delivered, batch they come from (calling thread)
	std::mutex mu;                    // guards the fields below
	std::condition_variable cv;
	uint64_t fetched = 0, decoded = 0, delivered = 0;   // batches whose payload is on the GPU / that are decoded / handed out
	bool closing = false;
	int rc = LFM_OK;                  // first failure: the reader is failed from then on
	std::string err;
	std::vector<uint64_t> ids[2], beg[2], end[2];       // blocks of the batch in payload buffer i (fetch thread -> worker)
	std::thread fetch_th, worker;
	lfm_stats st;
	double t_open = 0;

	int fail(int code, const std::string& what)
	{
		std::lock_guard<std::mutex> lk(mu);
		if (!rc) { rc = code; err = what; }
		cv.notify_all();
		return rc;
	}
	int failed() { std::lock_guard<std::mutex> lk(mu); return rc; }
	// box frame i (t slowest, z fastest) -> frame of the stack
	uint64_t flat(uint64_t i) const
	{
		const uint64_t nz = ub[2] - lb[2] + 1, nc = ub[3] - lb[3] + 1;
		return (lb[2] + i % nz) + (uint64_t)h.xyzct[2] * ((lb[3] + (i / nz) % nc) + (uint64_t)h.xyzct[3] * (lb[4] + i / (nz * nc)));
	}
	// box frames whose frame of the stack lies below f
	uint64_t box_before(uint64_t f) const
	{
		const uint64_t Z = h.xyzct[2], C = h.xyzct[3];
		const uint64_t t = f / (Z * C), c = (f / Z) % C, z = f % Z;
		const uint64_t nz = ub[2] - lb[2] + 1, nc = ub[3] - lb[3] + 1;
		auto below = [](uint64_t v, uint32_t a, uint32_t b) { return std::min<uint64_t>(std::max<uint64_t>(v, a), (uint64_t)b + 1) - a; };
		uint64_t n = below(t, lb[4], ub[4]) * nc * nz;
		if (t >= lb[4] && t <= ub[4]) {
			n += below(c, lb[3], ub[3]) * nz;
			if (c >= lb[3] && c <= ub[3]) n += below(z, lb[2], ub[2]);
		}
		return n;
	}
	bool touched(uint64_t s) const
	{
		const uint64_t bz = s % L.nb[2], c = (s / L.nb[2]) % h.xyzct[3], t = s / ((uint64_t)L.nb[2] * h.xyzct[3]);
		const uint64_t z0 = bz * h.blockSize[2], z1 = std::min<uint64_t>(h.xyzct[2], z0 + h.blockSize[2]) - 1;
		return z0 <= ub[2] && z1 >= lb[2] && c >= lb[3] && c <= ub[3] && t >= lb[4] && t <= ub[4];
	}
	// slabs decoded: those the box touches, and with pair frames the slab before one whose odd first frame is in the box
	bool slab_needed(uint64_t s) const
	{
		if (touched(s)) return true;
		if (!pair || s + 1 >= L.nSlabs || !touched(s + 1) || !(slab_first_frame(h, L, s + 1) & 1)) return false;
		return ((s + 1) % L.nb[2]) * h.blockSize[2] >= lb[2];
	}
	void fetch_loop()
	{
		cudaSetDevice(res->dev);
		std::vector<std::pair<uint64_t, uint64_t>> ranges;
		for (uint64_t b = 0; b < B.size(); b++) {
			{
				// payload buffer b & 1 is free once batch b - 2 is decoded
				std::unique_lock<std::mutex> lk(mu);
				cv.wait(lk, [&] { return b < 2 || decoded + 1 >= b || closing || rc; });
				if (closing || rc) return;
			}
			const int slot = (int)(b & 1);
			const double t0 = now_ms();
			std::vector<uint64_t>& I = ids[slot]; std::vector<uint64_t>& Bg = beg[slot]; std::vector<uint64_t>& E = end[slot];
			I.clear(); Bg.clear(); E.clear(); ranges.clear();
			uint64_t packed = 0;                                     // the needed runs of consecutive blocks, packed back to back
			for (uint64_t s = B[b].s0; s < B[b].s1; s++) {
				if (!slab_needed(s)) continue;
				for (uint64_t i = 0; i < L.blocksPerSlab; i++) {
					if (!block_needed(h, L, i, lb, ub, k)) continue;
					const uint64_t id = s * L.blocksPerSlab + i, a = id ? h.blockOffset[id - 1] : 0, z = h.blockOffset[id];
					if (!ranges.empty() && ranges.back().second == a) ranges.back().second = z;
					else ranges.emplace_back(a, z);
					I.push_back(id); Bg.push_back(packed); packed += z - a; E.push_back(packed);
				}
			}
			int r = src.to_device(res->up_pin, res->pay[slot].p, ranges, res->up_st);
			if (!r && cudaStreamSynchronize(res->up_st) != cudaSuccess) { cudaGetLastError(); r = LFM_ERR_CUDA; }
			if (r) { fail(r, r == LFM_ERR_BZIP ? "file is truncated" : "payload upload failed"); return; }
			{ std::lock_guard<std::mutex> lk(mu); fetched = b + 1; st.ms_h2d += now_ms() - t0; }
			cv.notify_all();
		}
	}
	void decode_loop()
	{
		cudaSetDevice(res->dev);
		for (uint64_t b = 0; b < B.size(); b++) {
			{
				// frame buffer b & 1 is free once batch b - 2 has been handed out
				std::unique_lock<std::mutex> lk(mu);
				cv.wait(lk, [&] { return (fetched > b && (direct || b < 2 || delivered + 1 >= b)) || closing || rc; });
				if (closing || rc) return;
			}
			const int slot = (int)(b & 1);
			const Batch& bt = B[b];
			uint16_t* fb = direct ? direct : (uint16_t*)res->img[slot].p - bt.f0 * L.fpx;      // virtual bases: absolute frame indexing
			uint16_t* sym = k != 0 ? (uint16_t*)res->sym.p - bt.f0 * L.fpx : fb;
			DecompressStats ds;
			double ms_unpredict = 0;
			if (!ids[slot].empty()) {
				LFM_API_LOCK();
				cudaSetDevice(e->device());
				cudaStream_t es = (cudaStream_t)e->stream();
				if (!full) cudaMemsetAsync(sym + bt.f0 * L.fpx, 0, (bt.f1 - bt.f0) * L.fpx * 2, es);
				int r = e->decompress_blocks((const uint8_t*)res->pay[slot].p, beg[slot].data(), end[slot].data(), ids[slot].data(),
				                             ids[slot].size(), sym, desc, &ds);
				if (r) { fail(r, e->last_error()); return; }
				if (k != 0 && bt.u1 > bt.u0) {
					if ((r = e->unpredict(sym, fb, desc, k, video, (uint32_t)bt.u0, (uint32_t)(bt.u1 - bt.u0)))) { fail(r, e->last_error()); return; }
					ds.launches += video ? 2 : 1;
				}
				if (cudaStreamSynchronize(es) != cudaSuccess) { cudaGetLastError(); fail(LFM_ERR_CUDA, "decode failed"); return; }
				if (k != 0 && bt.u1 > bt.u0) ms_unpredict = e->last_unpredict_ms();
			}
			{
				std::lock_guard<std::mutex> lk(mu);
				st.ms_decode += ds.ms_decode; st.ms_imtf += ds.ms_imtf; st.ms_ibwt += ds.ms_ibwt; st.ms_unrle += ds.ms_unrle;
				st.ms_unpredict += ms_unpredict; st.gpu_launches += ds.launches;
				decoded = b + 1;
			}
			cv.notify_all();                                            // payload buffer `slot` is free for batch b + 2
		}
	}
};

namespace {
// header, table and box checked as readLFMroiDevice checks them, plus what a reader cannot do (c or t blocked); the batches are cut
int reader_init(std::unique_ptr<lfm_stack_reader>& r, const klb_image_header& h, const PayloadSource& src, const uint32_t* lb, const uint32_t* ub)
{
	r.reset(new lfm_stack_reader);
	r->t_open = now_ms();
	memset(&r->st, 0, sizeof(r->st));
	int rc = check_stack(h, src.size, &r->k, &r->video);
	if (rc) return rc;
	if ((rc = check_box(h, lb, ub, r->lb, r->ub, &r->full))) return rc;
	if (h.blockSize[3] != 1 || h.blockSize[4] != 1) {
		g_err = "blocks over several channels or time points interleave their frames: there is no in-order stream to read"; return LFM_ERR_UNSUPPORTED;
	}
	r->h = h;
	r->src = src;
	r->L = make_layout(h);
	r->desc = make_desc(h, current_way());
	r->pair = r->k != 0 && r->video;
	r->st.predictor = r->k;
	const Layout& L = r->L;
	uint64_t nf = 1;
	for (int d = 2; d < 5; d++) nf *= (uint64_t)(r->ub[d] - r->lb[d] + 1);
	r->frames = nf;
	r->box_fpx = (uint64_t)(r->ub[0] - r->lb[0] + 1) * (r->ub[1] - r->lb[1] + 1);
	// slabs from the box's first to its last; with pair frames the first batch starts early enough to hold the even frame its
	// first frame needs
	const uint64_t C = h.xyzct[3];
	uint64_t s_begin = ((uint64_t)r->lb[4] * C + r->lb[3]) * L.nb[2] + r->lb[2] / h.blockSize[2];
	const uint64_t s_end = ((uint64_t)r->ub[4] * C + r->ub[3]) * L.nb[2] + r->ub[2] / h.blockSize[2] + 1;
	const uint64_t first = r->flat(0), last = r->flat(nf - 1);
	if (r->pair && (first & 1) && slab_first_frame(h, L, s_begin) == first) s_begin--;
	const std::vector<uint64_t> cut = batch_cuts(h, L, batch_slabs(h, L), r->pair, s_begin, s_end);
	const uint64_t u_first = r->pair ? first & ~1ull : first;
	for (size_t b = 0; b + 1 < cut.size(); b++) {
		lfm_stack_reader::Batch bt;
		bt.s0 = cut[b]; bt.s1 = cut[b + 1];
		bt.f0 = slab_first_frame(h, L, bt.s0); bt.f1 = slab_first_frame(h, L, bt.s1);
		bt.u0 = std::max(bt.f0, u_first); bt.u1 = std::min(bt.f1, last + 1);
		bt.i0 = r->box_before(bt.f0); bt.i1 = r->box_before(bt.f1);
		r->max_box_frames = std::max(r->max_box_frames, bt.i1 - bt.i0);
		r->B.push_back(bt);
	}
	return LFM_OK;
}

// buffers, resources and the two threads; with `direct` (a full read into an aligned device buffer) no frame buffer is needed
int reader_start(lfm_stack_reader* r, uint16_t* direct)
{
	r->direct = direct;
	r->e = &Engine::for_device(g_set.first_device);
	const int dev = r->e->device();
	cudaSetDevice(dev);
	std::unique_ptr<PipeRes> res(take_res(dev));
	if (!res) { res.reset(new PipeRes); if (res->init(dev)) { g_err = "pinned staging memory or copy streams could not be allocated"; return LFM_ERR_CUDA; } }
	const Layout& L = r->L;
	const klb_image_header& h = r->h;
	uint64_t max_nf = 0, max_pay = 0;
	for (const auto& bt : r->B) {
		max_nf = std::max(max_nf, bt.f1 - bt.f0);
		const uint64_t id0 = bt.s0 * L.blocksPerSlab, id1 = bt.s1 * L.blocksPerSlab;
		max_pay = std::max(max_pay, h.blockOffset[id1 - 1] - (id0 ? h.blockOffset[id0 - 1] : 0));
	}
	const size_t img_bytes = (size_t)max_nf * L.fpx * 2;
	Engine& e = *r->e;
	if (e.reserve(res->pay[0], max_pay + 16) || e.reserve(res->pay[1], max_pay + 16) ||
	    (!direct && (e.reserve(res->img[0], img_bytes) || e.reserve(res->img[1], img_bytes))) || (r->k != 0 && e.reserve(res->sym, img_bytes))) {
		give_res(res.release()); g_err = "batch buffers could not be allocated"; return LFM_ERR_CUDA;
	}
	r->res = res.release();
	try {
		r->fetch_th = std::thread([r]() { r->fetch_loop(); });
		r->worker = std::thread([r]() { r->decode_loop(); });
	} catch (const std::system_error&) {
		r->fail(LFM_ERR_CREATE, "the reader threads could not be started");
		if (r->fetch_th.joinable()) r->fetch_th.join();
		g_err = r->err; return LFM_ERR_CREATE;
	}
	return LFM_OK;
}

// box frames [i, j) of batch b (decoded) -> dst: device memory, or host memory through the staging buffer and the download ring
int reader_deliver(lfm_stack_reader* r, uint64_t b, uint64_t i, uint64_t j, uint8_t* dst, bool device)
{
	PipeRes& R = *r->res;
	const auto& bt = r->B[b];
	const Layout& L = r->L;
	const uint16_t* fb = (const uint16_t*)R.img[b & 1].p - bt.f0 * L.fpx;
	const size_t bytes = (size_t)(j - i) * r->box_fpx * 2;
	const bool whole_frames = r->box_fpx == L.fpx;
	if (!device && whole_frames && r->flat(j - 1) - r->flat(i) == j - 1 - i) {
		// uncropped frames that follow each other in the frame buffer: straight to the caller
		d2h_ring(R.down_pin, dst, fb + r->flat(i) * L.fpx, bytes, R.down_st);
	} else {
		if (!device && r->e->reserve(R.stage, (size_t)r->max_box_frames * r->box_fpx * 2)) return r->fail(LFM_ERR_CUDA, "staging buffer could not be allocated");
		uint16_t* to = device ? (uint16_t*)dst : (uint16_t*)R.stage.p;
		const uint64_t nz = r->ub[2] - r->lb[2] + 1;
		for (uint64_t u = i; u < j;) {
			// frames of one channel and time point: one sub-box
			const uint64_t f = r->flat(u), zoff = u % nz, n = std::min(j - u, nz - zoff);
			const uint32_t z = (uint32_t)(f % r->h.xyzct[2]), c = (uint32_t)((f / r->h.xyzct[2]) % r->h.xyzct[3]);
			const uint32_t t = (uint32_t)(f / ((uint64_t)r->h.xyzct[2] * r->h.xyzct[3]));
			const uint32_t lb[5] = { r->lb[0], r->lb[1], z, c, t }, ub[5] = { r->ub[0], r->ub[1], (uint32_t)(z + n - 1), c, t };
			if (int rc = r->e->roi_gather(fb, r->desc, lb, ub, to + (u - i) * r->box_fpx, R.down_st)) return r->fail(rc, "k_roi_gather launch failed");
			{ std::lock_guard<std::mutex> lk(r->mu); r->st.gpu_launches++; }
			u += n;
		}
		if (!device) d2h_ring(R.down_pin, dst, R.stage.p, bytes, R.down_st);
	}
	if (cudaStreamSynchronize(R.down_st) != cudaSuccess) { cudaGetLastError(); return r->fail(LFM_ERR_CUDA, "frame delivery failed"); }
	return LFM_OK;
}

int reader_read(lfm_stack_reader* r, void* dst, uint64_t n, uint64_t* got, bool device)
{
	if (got) *got = 0;
	if (int c = r->failed()) { g_err = r->err; return c; }
	if (n == 0) return LFM_OK;
	int rc = LFM_OK;
	if (!dst) r->fail(LFM_ERR_OPEN, "dst is NULL");
	else if (device && (rc = check_device_ptr(dst, "d_dst"))) r->fail(rc, g_err);
	if (int c = r->failed()) { g_err = r->err; return c; }
	if (r->pos >= r->frames) return LFM_OK;
	cudaSetDevice(r->res->dev);
	const double t0 = now_ms();
	const uint64_t end = r->pos + std::min(n, r->frames - r->pos);
	const size_t frame_bytes = (size_t)r->box_fpx * 2;
	uint64_t i = r->pos;
	while (i < end) {
		const auto& bt = r->B[r->cur];
		{
			std::unique_lock<std::mutex> lk(r->mu);
			r->cv.wait(lk, [&] { return r->decoded > r->cur || r->rc; });
			if (r->rc) break;
		}
		const uint64_t j = std::min(end, bt.i1);
		if (j > i && reader_deliver(r, r->cur, i, j, (uint8_t*)dst + (i - r->pos) * frame_bytes, device)) break;
		i = j;
		if (i == bt.i1) {
			// batch cur is handed out: its frame buffer takes batch cur + 2 (batches without box frames go by as well)
			do r->cur++; while (r->cur < r->B.size() && r->B[r->cur].i1 == r->B[r->cur].i0);
			{ std::lock_guard<std::mutex> lk(r->mu); r->delivered = r->cur; }
			r->cv.notify_all();
		}
	}
	if (!device) { std::lock_guard<std::mutex> lk(r->mu); r->st.ms_d2h += now_ms() - t0; }
	if (int c = r->failed()) { g_err = r->err; return c; }
	if (got) *got = i - r->pos;
	r->pos = i;
	return LFM_OK;
}

// stops the threads, frees r; the reader's statistics become the calling thread's
int reader_close(lfm_stack_reader* r)
{
	{ std::lock_guard<std::mutex> lk(r->mu); r->closing = true; }
	r->cv.notify_all();
	if (r->fetch_th.joinable()) r->fetch_th.join();
	if (r->worker.joinable()) r->worker.join();
	const int rc = r->rc;
	if (rc) g_err = r->err;
	if (r->own_fd >= 0) close(r->own_fd);
	r->st.ms_total = now_ms() - r->t_open;
	g_stats = r->st;
	if (r->res) give_res(r->res);
	delete r;
	return rc;
}

// Full reads of large single-GPU stacks take the reader (the pixels of both paths are identical): host memory, or a device buffer
bool takes_reader(const klb_image_header& h, const klb_ROI* roi, const DeviceSink* dsink)
{
	if (validate(h, false) || h.Nb == 0 || h.blockSize[3] != 1 || h.blockSize[4] != 1) return false;   // the other path reports these
	if (roi) for (int d = 0; d < 5; d++) if (roi->xyzctLB[d] != 0 || roi->xyzctUB[d] != h.xyzct[d] - 1) return false;
	const int ndev = current_ndev();
	if (ndev <= 0) return false;
	const Layout L = make_layout(h);
	if (!dsink && std::min<uint64_t>((uint64_t)ndev, L.nSlabs) != 1) return false;                       // sharded over several GPUs
	return slabs_per_batch(h, L) != 0;
}

// open a reader over the whole stack, read it into `out` (host) or the sink, close.  The batches decode straight into a 16-byte
// aligned device buffer; anything else receives the frames as a reader's Read hands them out.
int read_with_reader(const klb_image_header& h, const PayloadSource& src, uint16_t* out, const DeviceSink* dsink)
{
	memset(&g_stats, 0, sizeof(g_stats));
	std::unique_ptr<lfm_stack_reader> up;
	int rc = reader_init(up, h, src, nullptr, nullptr);
	if (rc) return rc;
	if (dsink) {
		// the caller's buffer is checked before any kernel runs: nothing is written to it unless the whole stack fits
		const uint64_t bytes = up->frames * up->box_fpx * 2;
		if (dsink->out_bytes) *dsink->out_bytes = bytes;
		if ((rc = check_device_ptr(dsink->d_out, "d_out"))) return rc;
		if (dsink->capacity < bytes) { g_err = "d_out is smaller than the box (" + std::to_string(bytes) + " bytes)"; return LFM_ERR_CREATE; }
		out = (uint16_t*)dsink->d_out;
	}
	const bool direct = dsink && ((uintptr_t)out & 15) == 0;
	if ((rc = reader_start(up.get(), direct ? out : nullptr))) return rc;
	lfm_stack_reader* r = up.release();
	if (direct) {
		std::unique_lock<std::mutex> lk(r->mu);
		r->cv.wait(lk, [&] { return r->decoded == r->B.size() || r->rc; });
	} else {
		uint64_t got = 0;
		try { rc = reader_read(r, out, r->frames, &got, dsink != nullptr); }
		catch (const std::exception&) { rc = r->fail(LFM_ERR_CREATE, "out of host memory"); }   // the reader is closed all the same
	}
	const int rc2 = reader_close(r);
	return rc ? rc : rc2;
}

// Pixels go to the host buffer `out`, or with a DeviceSink to its device buffer (then `out` is ignored): full reads into a
// 16-byte aligned buffer decode straight into it; ROI reads, and full reads into any other buffer, decode into the engine's
// frame buffers and k_roi_gather copies the box out.
int decompress_core(const klb_image_header& h, const PayloadSource& psrc, uint16_t* out, const klb_ROI* roi, const DeviceSink* dsink = nullptr)
{
	memset(&g_stats, 0, sizeof(g_stats));
	int k = 0, video = 0;
	int rc = check_stack(h, psrc.size, &k, &video);
	if (rc) return rc;
	const int ndev = current_ndev();
	const Layout L = make_layout(h);
	const StackDesc desc = make_desc(h, current_way());
	const double t_start = now_ms();
	g_stats.predictor = k;

	// which slabs / blocks are needed
	uint32_t lb[5], ub[5];
	bool full = true;
	if ((rc = check_box(h, roi ? roi->xyzctLB : nullptr, roi ? roi->xyzctUB : nullptr, lb, ub, &full))) return rc;
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
		// block list.  Full read: every block.  ROI: block_needed.
		std::vector<uint64_t> ids, beg, end;
		for (uint64_t s : my) for (uint64_t b = 0; b < L.blocksPerSlab; b++) {
			if (!full && !block_needed(h, L, b, lb, ub, k)) continue;
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
		if ((rcs[d] = psrc.to_device((uint8_t*)e.pinned(kStageBufs * kStageChunk, 0), dpay.p, ranges, st))) { if (rcs[d] == LFM_ERR_BZIP) std::cerr << "ERROR: lfm_b200: file is truncated" << std::endl; return; }
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
		const uint64_t fbeg = file_off + off[d], fend = fbeg + bytes;
		const uint64_t page = (uint64_t)sysconf(_SC_PAGESIZE), mbase = fbeg & ~(page - 1);
		uint8_t* map = nullptr;
		if (bytes >= ((uint64_t)256 << 10)) {
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
	{
		DeviceGuard g;
		if (takes_writer(src, header)) return write_stack_with_writer(filename, src, header);
	}
	LFM_API_LOCK();
	// the file is overwritten in place and cut to its final size at the end (same result as "wb", but an existing file of about
	// the same size keeps its pages: rewriting a stack does not pay for page allocation again)
	const int fd = open(filename.c_str(), O_RDWR | O_CREAT, 0666);
	if (fd < 0) { std::cout << "ERROR: file " << filename << " could not be opened" << std::endl; return LFM_ERR_CREATE; }
	int rc;
	try {
		std::vector<ShardOut> shards; std::vector<uint64_t> first;
		rc = compress_core(src, header, shards, first);
		if (rc == 0) rc = write_file(fd, header, shards);
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
	DeviceGuard g;
	if (fileSize < 320) return LFM_ERR_BZIP;
	header.unpackFixed((const uint8_t*)fileBytes);
	size_t nb = 0;
	if (!header.numBlocksBounded((fileSize - 320) / 8, &nb) || nb == 0) return LFM_ERR_BZIP;    // the table must fit the buffer
	header.resizeBlockOffset(nb);
	memcpy(header.blockOffset, fileBytes + 320, header.Nb * 8);
	PayloadSource ps; ps.base = (const uint8_t*)fileBytes + 320 + header.Nb * 8; ps.size = fileSize - 320 - header.Nb * 8;
	if (takes_reader(header, ROI, nullptr)) return read_with_reader(header, ps, (uint16_t*)imgOut, nullptr);
	LFM_API_LOCK();
	return decompress_core(header, ps, (uint16_t*)imgOut, ROI);
} LFM_CATCH

// header (+ blockOffset table) of the file, then decode straight from the open file: only the needed byte ranges are read
static int read_from_file(const std::string& filename, klb_image_header& header, uint16_t* out, const klb_ROI* roi,
                          const DeviceSink* dsink = nullptr)
try {
	DeviceGuard g;
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
	int rc;
	try {
		// a reader's worker thread takes the API lock itself: the full reads it serves run without holding it
		if (takes_reader(header, roi, dsink)) rc = read_with_reader(header, ps, out, dsink);
		else { LFM_API_LOCK(); rc = decompress_core(header, ps, out, roi, dsink); }
	} catch (...) { close(fd); throw; }
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

int lfmStackWriterOpen(lfm_stack_writer** w, const char* filename, const uint32_t xyzct[5], enum KLB_DATA_TYPE dataType,
                       const float32_t pixelSize[5], const uint32_t blockSize[5], enum KLB_COMPRESSION_TYPE compressionType,
                       const char metadata[256], uint8_t headerVersion, uint8_t Nnum)
try {
	g_err.clear();
	if (!w) return LFM_ERR_OPEN;
	*w = nullptr;
	if (!filename || !*filename || !xyzct) return LFM_ERR_OPEN;
	DeviceGuard g;
	klb_image_header h;
	h.setHeader(xyzct, dataType, pixelSize, blockSize, compressionType, metadata, headerVersion, Nnum);
	return writer_open(w, std::string(filename), h);
} LFM_CATCH

int lfmStackWriterAppend(lfm_stack_writer* w, const void* frames, uint64_t nframes)
try {
	g_err.clear();
	if (!w) return LFM_ERR_OPEN;
	DeviceGuard g;
	try { return writer_append(w, frames, nframes, false); }
	catch (const std::exception&) { g_err = "out of host memory"; return w->fail(LFM_ERR_CREATE, g_err); }   // fails the writer, as every other error
} LFM_CATCH

int lfmStackWriterAppendDevice(lfm_stack_writer* w, const void* d_frames, uint64_t nframes)
try {
	g_err.clear();
	if (!w) return LFM_ERR_OPEN;
	DeviceGuard g;
	try { return writer_append(w, d_frames, nframes, true); }
	catch (const std::exception&) { g_err = "out of host memory"; return w->fail(LFM_ERR_CREATE, g_err); }   // fails the writer, as every other error
} LFM_CATCH

int lfmStackWriterClose(lfm_stack_writer* w, uint64_t* frames_kept)
try {
	g_err.clear();
	if (frames_kept) *frames_kept = 0;
	if (!w) return LFM_ERR_OPEN;
	DeviceGuard g;
	return writer_close(w, frames_kept);
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

int lfmStackReaderOpen(lfm_stack_reader** r, const char* filename, const uint32_t lb[5], const uint32_t ub[5], uint64_t* frames, uint64_t* frame_bytes)
try {
	g_err.clear();
	if (frames) *frames = 0;
	if (frame_bytes) *frame_bytes = 0;
	if (!r) return LFM_ERR_OPEN;
	*r = nullptr;
	// the checks of readLFMroiDevice, in its order
	if (!filename || !*filename || (lb == nullptr) != (ub == nullptr)) return LFM_ERR_OPEN;
	if (access(filename, R_OK) != 0) { g_err = std::string("cannot open ") + filename; return LFM_ERR_OPEN; }
	DeviceGuard g;
	klb_image_header h;
	int rc = h.readHeader(filename);
	if (rc > 0) return rc;
	if (h.Nb == 0) { std::cerr << "ERROR: Image to read has not blocks" << std::endl; return LFM_ERR_BZIP; }
	const int fd = open(filename, O_RDONLY);
	if (fd < 0) { g_err = std::string("cannot open ") + filename; return LFM_ERR_OPEN; }
	struct stat sb;
	PayloadSource ps; ps.fd = fd; ps.file_off = h.getSizeInBytes();
	ps.size = (fstat(fd, &sb) == 0 && (uint64_t)sb.st_size > ps.file_off) ? (uint64_t)sb.st_size - ps.file_off : 0;
	std::unique_ptr<lfm_stack_reader> up;
	try { rc = reader_init(up, h, ps, lb, ub); } catch (...) { close(fd); throw; }
	if (!rc) rc = reader_start(up.get(), nullptr);
	if (rc) { close(fd); return rc; }
	up->own_fd = fd;
	if (frames) *frames = up->frames;
	if (frame_bytes) *frame_bytes = up->box_fpx * 2;
	*r = up.release();
	return LFM_OK;
} LFM_CATCH

int lfmStackReaderRead(lfm_stack_reader* r, void* dst, uint64_t n, uint64_t* got)
try {
	g_err.clear();
	if (got) *got = 0;
	if (!r) return LFM_ERR_OPEN;
	DeviceGuard g;
	try { return reader_read(r, dst, n, got, false); }
	catch (const std::exception&) { g_err = "out of host memory"; return r->fail(LFM_ERR_CREATE, g_err); }   // fails the reader, as every other error
} LFM_CATCH

int lfmStackReaderReadDevice(lfm_stack_reader* r, void* d_dst, uint64_t n, uint64_t* got)
try {
	g_err.clear();
	if (got) *got = 0;
	if (!r) return LFM_ERR_OPEN;
	DeviceGuard g;
	try { return reader_read(r, d_dst, n, got, true); }
	catch (const std::exception&) { g_err = "out of host memory"; return r->fail(LFM_ERR_CREATE, g_err); }   // fails the reader, as every other error
} LFM_CATCH

int lfmStackReaderClose(lfm_stack_reader* r)
try {
	g_err.clear();
	if (!r) return LFM_ERR_OPEN;
	DeviceGuard g;
	return reader_close(r);
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
