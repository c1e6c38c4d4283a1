// engine.h -- device pipeline of the B200 LFM engine (one instance per GPU).
//
// The engine owns the CUDA stream, the growable device workspace and the kernel sequence for
//   compress   : [mode selection] -> predict+symbolize -> per KLB block: RLE1/CRC -> BWT -> MTF/RLE2 -> Huffman+pack
//   decompress : per KLB block: Huffman/MTF decode -> inverse BWT -> un-RLE1/CRC + scatter -> inverse predictor
// and nothing else: file format, block partition across GPUs and the reference-compatible API live in klb_imageIO.cpp.
#pragma once
#include <cstdint>
#include <cstddef>
#include <vector>
#include <string>

namespace lfm {

// error codes shared with the C ABI (0..5 are the reference's, src/klb_Cwrapper.cpp:33-46; >= 6 are new)
enum : int {
	LFM_OK = 0,
	LFM_ERR_BZIP = 2,          // codec failure / corrupt stream / CRC mismatch / no blocks
	LFM_ERR_OPEN = 3,          // cannot open for read, unsupported API combination
	LFM_ERR_CREATE = 5,        // cannot create output / unknown codec
	LFM_ERR_CUDA = 6,          // CUDA runtime failure (the reference ignores these)
	LFM_ERR_UNSUPPORTED = 7,   // data type / codec / block size outside what this engine implements
};

struct StackDesc {
	uint32_t xyzct[5];
	uint32_t blockSize[5];     // already clamped to xyzct
	int      Nnum;
	int      way;              // 0 tiles(both), 1 angle, 2 space  (compile-time LFM_PREDICTOR_WAY in the reference)
	int      codec = 1;        // KLB_COMPRESSION_TYPE of the block payloads: 1 bzip2, 0 none (rows copied verbatim)
};

struct CompressStats {
	int      predictor = 0;
	float    entropy[8] = { 0, 0, 0, 0, 0, 0, 0, 0 };
	bool     selected = false;
	double   ms_select = 0, ms_predict = 0, ms_rle = 0, ms_bwt = 0, ms_mtf = 0, ms_huff = 0, ms_total = 0;
	uint64_t launches = 0;
	uint32_t periodic_blocks = 0;
};
struct DecompressStats {
	double   ms_decode = 0, ms_imtf = 0, ms_ibwt = 0, ms_unrle = 0, ms_unpredict = 0, ms_total = 0;
	uint64_t launches = 0;
};

class Engine {
public:
	static Engine& for_device(int device);     // one engine per GPU, created on first use

	// Mode selection on frame 0 of a device-resident stack (SURVEY Appendix C). Returns the winner 0..7.
	int select_mode(const uint16_t* d_frame0, const StackDesc& s, float entropy[8], int* winner);

	// Forward predictor + symbolize over frames [z0, z0+nz) of a device-resident stack (predictor 1..7).
	int predict(const uint16_t* d_img, uint16_t* d_sym, const StackDesc& s, int predictor, int video, uint32_t z0, uint32_t nz);

	// Compress KLB blocks [first, first+count) of the device-resident SYMBOL image.
	// sizes_out[count] (host) receives each block's stream size; the streams are left compacted, in block order,
	// in an engine-owned device buffer (*d_payload, *payload_bytes) that stays valid until the next call, or in `payload` (grown as
	// needed) when the caller owns the buffer: a stack writer keeps its payload there while other calls use the engine.
	struct Buf { void* p = nullptr; size_t cap = 0; };
	int compress_blocks(const uint16_t* d_sym, const StackDesc& s, uint64_t first, uint64_t count,
	                    uint32_t* sizes_out, const uint8_t** d_payload, uint64_t* payload_bytes, CompressStats* st, Buf* payload = nullptr);

	// Decode the listed KLB blocks from a device-resident payload into the device-resident symbol image.
	// begin/end: byte range of each listed block inside d_payload (host arrays).
	int decompress_blocks(const uint8_t* d_payload, const uint64_t* begin, const uint64_t* end, const uint64_t* block_ids,
	                      uint64_t count, uint16_t* d_sym, const StackDesc& s, DecompressStats* st);

	// One bzip2 stream of the device-resident bytes d_src[0, n), byte-identical to BZ2_bzBuffToBuffCompress(.., level, 0, 30);
	// n < 2^32, level 1..9.  The stream is left in an engine-owned device buffer (*d_out, *out_size) valid until the next call.
	int bz2_compress(const uint8_t* d_src, uint64_t n, int level, const uint8_t** d_out, uint64_t* out_size, CompressStats* st);
	// Any .bz2 data (src: n bytes, host or device memory) -> its decompressed bytes: one or more concatenated streams, block
	// and stream CRCs checked.  Output into d_dst (device, `capacity` bytes) or, when d_dst is NULL, an engine-owned device
	// buffer (*d_out) valid until the next call.  *out_size = decompressed size; LFM_ERR_CREATE (5) when it exceeds capacity
	// (nothing written).
	int bz2_decompress(const void* src, uint64_t n, bool src_on_host, uint8_t* d_dst, uint64_t capacity, const uint8_t** d_out,
	                   uint64_t* out_size, DecompressStats* st);
	// device buffer of at least `bytes` for a caller's input that has to be staged on this GPU first
	uint8_t* bz2_staging(size_t bytes);

	// Inverse predictor (unsymbolize fused) over frames [z0, z0+nz); in place is NOT allowed (d_sym != d_out).
	int unpredict(const uint16_t* d_sym, uint16_t* d_out, const StackDesc& s, int predictor, int video, uint32_t z0, uint32_t nz);

	// The box lb..ub (inclusive x,y,z,c,t bounds) of the decoded frames d_frames (absolute frame indexing) -> dense
	// [t][c][z][y][x] at d_out, one k_roi_gather launch on `stream` (NULL: the engine stream), not synchronised.
	int roi_gather(const uint16_t* d_frames, const StackDesc& s, const uint32_t lb[5], const uint32_t ub[5], uint16_t* d_out, void* stream = nullptr);

	// device time of the last predict() / unpredict() call (valid once the stream has been synchronised)
	double last_predict_ms();
	double last_unpredict_ms();

	void* stream() const { return stream_; }
	int   device() const { return device_; }
	int   sm_count() const { return sm_count_; }
	const std::string& last_error() const { return err_; }

	// growable device scratch, kept across calls
	int reserve(Buf& b, size_t bytes);
	// buffers the orchestrator (klb_imageIO.cpp) keeps on this GPU between calls: image, symbol image, payload, frame 0
	Buf user[4];
	// growable pinned host staging buffers: slot 0 = towards the GPU, slot 1 = from the GPU
	void* pinned(size_t bytes, int slot = 0);

	// debugging / stage-parity hook: copies of the intermediate arrays of the LAST compress_blocks batch
	struct EncodeTrace {
		std::vector<uint8_t> jobs;      // raw EncJob records
		std::vector<uint8_t> txt, bwt;  // [njobs * cap]
		std::vector<uint16_t> mtfv;     // [njobs * mcap]
		uint32_t cap = 0, mcap = 0, njobs = 0;
	};
	int fetch_encode_trace(EncodeTrace& t);

private:
	explicit Engine(int device);
	int check(const char* what);
	// KLB_COMPRESSION_TYPE::NONE (src/klb_imageIO.cpp:207-210, :620-623): gather / scatter only
	int compress_blocks_none(const uint16_t* d_sym, const StackDesc& s, uint64_t first, uint64_t count,
	                         uint32_t* sizes_out, const uint8_t** d_payload, uint64_t* payload_bytes, CompressStats* st, Buf& pay);
	int decompress_blocks_none(const uint8_t* d_payload, const uint64_t* begin, const uint64_t* end, const uint64_t* block_ids,
	                           uint64_t count, uint16_t* d_sym, const StackDesc& s, DecompressStats* st);

	int device_ = 0, sm_count_ = 148;
	void* stream_ = nullptr;
	std::string err_;
	// workspace
	Buf jobs_, txt_, bwt_, rank_, mtfv_, sel_, out_, scratch_, payload_, sizes_, offs_;
	Buf djobs_, dbegin_, dend_, dids_, tt_;
	Buf sel_tabs_, sel_hist_, sel_e_, sel_cand_;
	Buf sz_tiles_, sz_bits_, sz_blocks_, sz_out_, sz_in_;      // bz2_compress: tile records, record-end bitmap, block records, stream, staging
	Buf dz_in_, dz_cand_, dz_out_;                              // bz2_decompress: padded input, candidate / block records, output
	uint32_t last_cap_ = 0, last_mcap_ = 0, last_njobs_ = 0;
	void* pin_[2] = { nullptr, nullptr }; size_t pin_cap_[2] = { 0, 0 };
	void* ev_[4] = { nullptr };          // predictor / inverse predictor timing
	std::vector<void*> ev_pool_;     // stage-timing events, created once and reused (event creation costs host time per call)
	void* pooled_event(size_t i);
};

}  // namespace lfm
