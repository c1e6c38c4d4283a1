/*
 * lfm_b200.h -- extension C ABI of the B200 LFM engine (plain pointers and sizes; no CUDA or torch types).
 * Everything the reference can only do through its C++ object (header knobs, src/klb_imageHeader.h:32-94; the
 * compile-time predictor "way", src/common.h:19) plus memory-to-memory and device-resident entry points used for
 * measurement. The file-based functions produce/consume exactly the .lfm layout of the reference
 * (src/klb_imageHeader.cpp:164-196, src/klb_imageIO.cpp:1145-1225).
 */
#ifndef __LFM_B200_H__
#define __LFM_B200_H__

#ifdef __cplusplus
extern "C" {
#endif

#include <stdint.h>
#include "common.h"

/* run-time replacement of the compile-time LFM_PREDICTOR_WAY (src/common.h:19): 0 tiles/both, 1 angle, 2 space.
   The way is NOT stored in the file (reference defect, SURVEY.md F.2): reader and writer must agree.
   Initial value: environment LFM_PREDICTOR_WAY, else 0. Returns the previous value, -1 on a bad argument. */
int lfmSetPredictorWay(int way);
int lfmGetPredictorWay(void);

/* number of GPUs the blocks are sharded over (default: environment LFM_B200_GPUS, else 1; clamped to the visible
   devices). first_device: index of the first device used. Returns the count in effect. */
int lfmSetDevices(int first_device, int count);

/* writeKLBstack with the header knobs exposed (mirrors matlabWrapper/writeLFMstack.cpp:424-443 and
   test/mainTest_lfmIO.cxx:60-97): headerVersion 0..7 = auto-select, 8+k = force predictor k, |0x80 = video stack. */
int writeLFMstackEx(const void* im, const char* filename, const uint32_t xyzct[KLB_DATA_DIMS], enum KLB_DATA_TYPE dataType,
                    int numThreads, const float32_t pixelSize[KLB_DATA_DIMS], const uint32_t blockSize[KLB_DATA_DIMS],
                    enum KLB_COMPRESSION_TYPE compressionType, const char metadata[KLB_METADATA_SIZE],
                    uint8_t headerVersion, uint8_t Nnum);

/* ---- device-resident files: the pixels stay in GPU memory, only the compressed payload crosses PCIe.
   Both calls run on the first device of lfmSetDevices only, also with lfmSetDevices(first, n > 1), and return with the engine
   stream synchronised.  The caller's buffer must be device or managed memory on that device (code 3 otherwise); a caller
   that writes it on another stream synchronises that stream first.

   writeLFMstackEx with the stack in DEVICE memory (d_im: x fastest, frames = z*c*t).  Same arguments, same return codes, and a
   file byte-identical to what writeLFMstackEx writes for the same pixels.  lfmGetLastStats: ms_h2d stays 0. */
int writeLFMstackDevice(const void* d_im, const char* filename, const uint32_t xyzct[KLB_DATA_DIMS], enum KLB_DATA_TYPE dataType,
                        int numThreads, const float32_t pixelSize[KLB_DATA_DIMS], const uint32_t blockSize[KLB_DATA_DIMS],
                        enum KLB_COMPRESSION_TYPE compressionType, const char metadata[KLB_METADATA_SIZE],
                        uint8_t headerVersion, uint8_t Nnum);
/* decode a file, or the box lb..ub of it (inclusive x,y,z,c,t bounds; both NULL = whole stack), into DEVICE memory d_out:
   dense [t][c][z][y][x] of the box, the same pixels readKLBstackInPlace / readKLBroiInPlace return.  *out_bytes (may be NULL)
   receives the size of the box in bytes; when capacity is smaller the call returns 5 and writes nothing to d_out.  Any 2-byte
   aligned d_out works; a whole-stack read decodes in place only into a 16-byte aligned d_out (cudaMalloc's are), into any
   other one through the engine's frame buffers and one more device copy.
   Return codes: 2 truncated or corrupt file, 3 a file that cannot be opened (readKLBstackInPlace gives 2 there), a box outside
   the stack or a bad d_out, 6 no CUDA device, 7 ZLIB payloads or pixels that are not 16-bit.  lfmGetLastStats: ms_d2h stays 0. */
int readLFMroiDevice(const char* filename, const uint32_t lb[KLB_DATA_DIMS], const uint32_t ub[KLB_DATA_DIMS],
                     void* d_out, uint64_t capacity, uint64_t* out_bytes);

/* ---- recording: a stack written frame by frame as its frames arrive, in device and host memory that do not grow with its length.
   lfmStackWriterOpen takes the arguments of writeLFMstackEx; xyzct is the shape of the whole recording.  Frames arrive in the order
   writeLFMstackEx reads im: frame f = z + Z*(c + C*t), x fastest within a frame.  Append copies its frames before it returns (the
   caller may reuse its buffer at once): host frames are staged into the writer's batch buffer on the GPU, device frames (device or
   managed memory on the first device of lfmSetDevices, code 3 otherwise; the caller synchronises its stream first) are copied
   device to device.  Mode selection (headerVersion 0..7, with or without the video bit) runs on frame 0 when it arrives.  Every
   batch of whole z-slabs (>= 96 MB and >= 2048 KLB blocks) is predicted and compressed once all its frames are in, and its payload
   goes to its final file offset while the next batch fills; when the GPU is two batches behind, Append blocks.  A recording runs on
   the first device of lfmSetDevices only.  Until Close, the file is not a valid .lfm file (the header and table are written last).
   Close with every declared frame: the file is byte-identical to writeLFMstackEx of the whole stack with the same arguments, for any
   append chunking and any mix of host and device frames; lfmGetLastStats reports the recording's totals.
   Close earlier: with d the slowest of z, c, t whose extent is above 1 and u the frames per step of d, the largest multiple of u
   received is kept (*frames_kept), xyzct[d] becomes kept / u and the file is byte-identical to writeLFMstackEx of that prefix
   (blockSize clamped to the new extent); later frames are dropped.  Nothing kept: code 2 and an empty file.
   Return codes.  Open: those of writeLFMstackEx for the same arguments (7 pixels that are not 16-bit, ZLIB, a forced predictor on a
   video stack with way != 0; 3 a bad filename; 5 a file that cannot be created; 6 no device), and 7 for blockSize[3] or [4] above 1
   after clamping (such blocks span frames that do not arrive one after the other); no file is created on an error.  Append: 3 past
   the declared frame count (nothing is taken, the writer stays usable).  Any other failure (7 when auto-selection picks a predictor
   a video stack with way != 0 cannot use, 6 CUDA, 5 file I/O, 3 a bad frames pointer) fails the writer: later appends return the
   same code, and Close cuts the file to 0 bytes and returns it.  Close always frees w.  Calls on one writer come from one thread at a
   time; writers and every other call of this library may be used side by side. */
typedef struct lfm_stack_writer lfm_stack_writer;
int lfmStackWriterOpen(lfm_stack_writer** w, const char* filename, const uint32_t xyzct[KLB_DATA_DIMS], enum KLB_DATA_TYPE dataType,
                       const float32_t pixelSize[KLB_DATA_DIMS], const uint32_t blockSize[KLB_DATA_DIMS],
                       enum KLB_COMPRESSION_TYPE compressionType, const char metadata[KLB_METADATA_SIZE], uint8_t headerVersion,
                       uint8_t Nnum);
int lfmStackWriterAppend(lfm_stack_writer* w, const void* frames, uint64_t nframes);             /* host memory */
int lfmStackWriterAppendDevice(lfm_stack_writer* w, const void* d_frames, uint64_t nframes);     /* device memory */
int lfmStackWriterClose(lfm_stack_writer* w, uint64_t* frames_kept);                               /* finishes the file, frees w */

/* ---- playing a stack back frame by frame, in bounded memory (single GPU: the first device of lfmSetDevices).
   lfmStackReaderOpen opens `filename` for reading the inclusive x,y,z,c,t box lb..ub (NULL, NULL: the whole stack) as
   readLFMroiDevice takes it; *frames = frames the box holds (its z*c*t extent), *frame_bytes = 2 * (x extent) * (y extent).  The
   header and blockOffset table are read and checked once, and the same codes as readLFMroiDevice's come back in the same order:
   2 corrupt or truncated table or payload, 3 file that cannot be opened or box outside the stack, 6 no device, 7 ZLIB payloads,
   pixels that are not 16-bit, video written with way != 0, and blockSize[3] or [4] above 1 (blocks over several channels or time
   points interleave their frames).
   lfmStackReaderRead / ReadDevice deliver the next n frames of the box, dense [t][c][z][y][x] order, into host memory (pageable
   or pinned) / device memory of the first device of lfmSetDevices (any even byte offset; code 3 for anything else), and return
   once the frames are in dst.  *got = frames delivered: fewer than n only at the end, 0 past it (the reader stays usable).  The
   concatenation of all reads is readLFMroiDevice's output for the box, bit for bit, whatever the chunking; host and device reads
   may be mixed.  While the caller holds frames of batch b, batch b + 1 is decoded and batch b + 2 read from the file.  Any other
   failure (a payload found truncated or corrupt on the way: 2) fails the reader: later reads and Close return its code, and
   nothing is written past n frames of dst.  One reader is used from one thread at a time; other readers, writers and calls may
   run between its reads.  Memory: two batches of frames and payload on the GPU, the staging rings, and the table.
   lfmStackReaderClose frees the reader; lfmGetLastStats then holds the reader's totals. */
typedef struct lfm_stack_reader lfm_stack_reader;
int lfmStackReaderOpen(lfm_stack_reader** r, const char* filename, const uint32_t lb[KLB_DATA_DIMS], const uint32_t ub[KLB_DATA_DIMS],
                       uint64_t* frames, uint64_t* frame_bytes);
int lfmStackReaderRead(lfm_stack_reader* r, void* dst, uint64_t n, uint64_t* got);              /* host memory */
int lfmStackReaderReadDevice(lfm_stack_reader* r, void* d_dst, uint64_t n, uint64_t* got);      /* device memory */
int lfmStackReaderClose(lfm_stack_reader* r);                                                     /* frees r, returns its failure code */

/* header byte 0 / byte 1 of a file (stored predictor | video bit, Nnum); 0 ok */
int readLFMheaderEx(const char* filename, uint8_t* headerVersion, uint8_t* Nnum);

/* memory -> memory: the complete .lfm file image (header + blockOffset + payload) of a HOST stack into a malloc()ed
   buffer the caller free()s. Same arguments as writeLFMstackEx. */
int lfmCompressToMemory(const void* im, const uint32_t xyzct[KLB_DATA_DIMS], const uint32_t blockSize[KLB_DATA_DIMS],
                        uint8_t headerVersion, uint8_t Nnum, void** file_bytes, uint64_t* file_size);
/* same, into a caller-owned HOST buffer of `capacity` bytes (pinned memory makes the D2H copy a straight DMA);
   *file_size receives the size needed; returns 5 when the buffer is too small (nothing is written then) */
int lfmCompressToBuffer(const void* im, const uint32_t xyzct[KLB_DATA_DIMS], const uint32_t blockSize[KLB_DATA_DIMS],
                        uint8_t headerVersion, uint8_t Nnum, void* file_bytes, uint64_t capacity, uint64_t* file_size);
/* inverse: decode a complete .lfm file image held in HOST memory into im (host, full stack) */
int lfmDecompressFromMemory(const void* file_bytes, uint64_t file_size, void* im);

/* device-resident entry points (one GPU, the current lfmSetDevices first device). d_im / d_out are CUDA device pointers.
   lfmCompressDevice leaves the compacted block streams on the device; *d_payload stays valid until the next call other than
   lfmDecompressDevice, which only reads the payload it is given.
   blockOffset[Nb] (host) receives the inclusive prefix sum of the stream sizes = header.blockOffset[]. */
int lfmCompressDevice(const void* d_im, const uint32_t xyzct[KLB_DATA_DIMS], const uint32_t blockSize[KLB_DATA_DIMS],
                      uint8_t headerVersion, uint8_t Nnum, uint8_t* storedHeaderVersion, uint64_t* blockOffset,
                      uint64_t numBlocks, const void** d_payload, uint64_t* payload_bytes);
/* mode selection alone (predict_and_2DEntropy x 8 + the min-entropy pick, src/klb_imageIO.cpp:2197-2225, :2300-2305) on a
   device-resident frame of xy[0] x xy[1] pixels: *predictor = winner 0..7, entropy[8] (may be NULL) the candidates' estimates.
   With one process per GPU the owner of frame 0 calls this and broadcasts the 3 bits. */
int lfmSelectDevice(const void* d_frame0, const uint32_t xy[2], uint8_t Nnum, int* predictor, float entropy[8]);
int lfmDecompressDevice(const void* d_payload, const uint64_t* blockOffset, uint64_t numBlocks,
                        const uint32_t xyzct[KLB_DATA_DIMS], const uint32_t blockSize[KLB_DATA_DIMS],
                        uint8_t storedHeaderVersion, uint8_t Nnum, void* d_out);

/* ---- one process per GPU (SURVEY.md 8e): KLB blocks are independent streams and a range of z-slabs is a contiguous block-id and
   payload range (block ids are x fastest, src/klb_imageIO.cpp:133-140), so every rank compresses the slabs it owns as a stack of
   its own and the only exchange is the host-side prefix sum of the block sizes (blockWriter, src/klb_imageIO.cpp:1145-1225):
     1. lfmShardCompress   this rank's frames (host) -> streams left on its GPU; blockSizes[numBlocks] = size of each local block.
                           Ranks other than the owner of frame 0 pass a forced headerVersion (8 + k | video bit); a video shard
                           must start on an even frame of the whole stack.
     2. the caller all-gathers the sizes, prefix-sums them into blockOffset[] and calls lfmWriteHeader once (creates the file,
        writes the 320 bytes + table, sizes the file);
     3. lfmShardWritePayload  streams the rank's payload from its GPU to its byte offset of the file (pinned ring + pwrite),
        or lfmShardFetchPayload copies it into a host buffer.
   The read side needs nothing new: readKLBroiInPlace with the rank's z range only fetches and decodes its slabs. */
int lfmShardCompress(const void* im_local, const uint32_t xyzct_local[KLB_DATA_DIMS], const uint32_t blockSize[KLB_DATA_DIMS],
                     uint8_t headerVersion, uint8_t Nnum, uint8_t* storedHeaderVersion, uint32_t* blockSizes, uint64_t numBlocks,
                     uint64_t* payload_bytes);
int lfmShardWritePayload(const char* filename, uint64_t file_offset);
int lfmShardFetchPayload(void* dst, uint64_t capacity);
int lfmWriteHeader(const char* filename, const uint32_t xyzct[KLB_DATA_DIMS], const uint32_t blockSize[KLB_DATA_DIMS],
                   uint8_t storedHeaderVersion, uint8_t Nnum, const uint64_t* blockOffset, uint64_t numBlocks);

/* number of KLB blocks for a stack (klb_imageHeader.cpp:77-85, after clamping blockSize to xyzct; NULL = default) */
uint64_t lfmNumBlocks(const uint32_t xyzct[KLB_DATA_DIMS], const uint32_t blockSize[KLB_DATA_DIMS]);

/* ---- standalone bzip2 streams of arbitrary bytes (no KLB framing), on the first device of lfmSetDevices.
   lfmBz2Compress writes one bzip2 stream byte-identical to BZ2_bzBuffToBuffCompress(dst, &len, src, n, level, 0, 30), level 1..9,
   any number of bzip2 blocks; n == 0 gives the 14-byte empty stream.  *dst_size receives the stream size; when `capacity` is
   smaller, nothing is written and the call returns 5.  lfmBz2CompressDevice takes a device pointer and leaves the stream in an
   engine-owned device buffer (*d_out, *out_size) that stays valid until the next call, as with lfmCompressDevice.
   Return codes: 0 ok, 2 codec failure, 3 bad arguments (level outside 1..9, NULL with n > 0), 5 dst too small, 6 CUDA error,
   7 input or stream of 2^32 bytes or more (the unsigned int limit of libbz2's buffer API).  lfmGetLastStats: ms_rle (run-length
   structure, block boundaries and per-block run-length coding), ms_bwt, ms_mtf, ms_huff (Huffman coding and stream assembly),
   payload_bytes = stream size, gpu_launches. */
int lfmBz2Compress(const void* src, uint64_t n, int level, void* dst, uint64_t capacity, uint64_t* dst_size);
int lfmBz2CompressDevice(const void* d_src, uint64_t n, int level, const void** d_out, uint64_t* out_size);
/* any .bz2 data: one or more concatenated streams (bzip2, pbzip2, lbzip2 output), each with its own level, randomised blocks
   included; block and stream CRCs checked.  *dst_size receives the decompressed size, known before any byte is written: when
   `capacity` is smaller the call returns 5 and writes nothing.  Code 2: corrupt data (bad magic, CRC mismatch, truncated stream, a
   block over 100000 * level bytes, bytes after the last stream that do not start another one, n == 0 as in
   BZ2_bzBuffToBuffDecompress).  lfmGetLastStats: ms_decode (magic scan, speculative Huffman decode of every candidate block, chain
   walk), ms_unrle (the real blocks: decode, inverse BWT, un-RLE1, CRCs), gpu_launches. */
int lfmBz2Decompress(const void* src, uint64_t n, void* dst, uint64_t capacity, uint64_t* dst_size);
int lfmBz2DecompressDevice(const void* d_src, uint64_t n, void* d_dst, uint64_t capacity, uint64_t* dst_size);

/* statistics of the last compress / decompress call made by the calling thread */
typedef struct {
	int    predictor;         /* stored predictor 0..7 */
	int    selected;          /* 1 if chosen by the 2-D entropy rule */
	float  entropy[8];        /* candidate entropies when selected */
	double ms_select, ms_predict, ms_rle, ms_bwt, ms_mtf, ms_huff;       /* kernel time per stage, CUDA events */
	double ms_decode, ms_ibwt, ms_unrle, ms_unpredict;
	double ms_h2d, ms_d2h, ms_total;
	uint64_t gpu_launches;    /* kernels launched */
	uint64_t periodic_blocks; /* exactly periodic bzip2 blocks met (origPtr tie rule applied, DESIGN.md) */
	uint64_t payload_bytes;
	double ms_imtf;           /* inverse MTF + run expansion (ms_decode is the Huffman decode alone) */
} lfm_stats;
int lfmGetLastStats(lfm_stats* out);

/* error text of the last failed call made by the calling thread (valid until its next call) */
const char* lfmLastError(void);

/* test hook: per-stage intermediates of the block encoder for ONE host buffer treated as one KLB block of
   n bytes (n even). Arrays must hold: rle1/bwt >= n*5/4+32 bytes, mtfv >= n*5/4+40 uint16, stream >= 2n+8300 bytes.
   info[8] = { nblock, crc, origPtr, nInUse, nMTF, nGroups, nSelectors, streamBytes } */
int lfmDebugEncodeBlock(const void* bytes, uint32_t n, uint8_t* rle1, uint8_t* bwt, uint16_t* mtfv, uint8_t* stream, uint32_t info[8]);

/* test hook (no GPU needed): the threaded host copy behind the staging paths (pageable <-> pinned memory, mapped file ranges) */
int lfmDebugParMemcpy(void* dst, const void* src, uint64_t n);

/* measurement hook: run ONLY the predictor kernels on a device-resident stack, `reps` times back to back, and return
   the mean device time per repetition (CUDA events on the engine stream).  inverse = 0: forward predictor + symbolize
   d_in (pixels) -> d_out (symbols); inverse = 1: unsymbolize + inverse predictor d_in (symbols) -> d_out (pixels).
   k = 1..7, way = current lfmSetPredictorWay. Algorithmic traffic: 4 bytes per pixel (SURVEY.md 8d). */
int lfmDebugPredictDevice(const void* d_in, void* d_out, const uint32_t xyzct[KLB_DATA_DIMS], uint8_t Nnum, int k, int video,
                          int inverse, int reps, float* ms_per_rep);

#ifdef __cplusplus
}
#endif
#endif
