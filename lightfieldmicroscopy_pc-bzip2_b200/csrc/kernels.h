// kernels.h -- host-callable launchers of the sm_100a kernels (definitions in the .cu files named beside each).
#pragma once
#include "lfm_device.cuh"

namespace lfm {

// lfm_predict.cu
void launch_predict_fwd(const uint16_t* img, uint16_t* sym, int W, int H, int T, int way, int k, int video,
                        uint32_t z0, uint32_t nz, cudaStream_t st);
int launch_unpredict(const uint16_t* sym, uint16_t* out, int W, int H, int T, int way, int k, int video,
                     uint32_t z_start, uint32_t z_step, uint32_t count, int sm_count, cudaStream_t st, const char** failed);
// lfm_roi.cu: the box lb..ub (inclusive x,y,z,c,t) of frames (absolute frame indexing) -> dense [t][c][z][y][x] at out, one launch
void launch_roi_gather(const uint16_t* frames, const uint32_t xyzct[5], const uint32_t lb[5], const uint32_t ub[5], uint16_t* out,
                       int sm_count, cudaStream_t st);
// lfm_select.cu
void launch_select(const uint16_t* const cand_ptrs[8], int ncand, uint64_t fpx, uint32_t chunk_px, uint32_t nchunks,
                   uint8_t* sorted, uint32_t sstride, uint32_t* hist, float* e_out, uint32_t* scratch, cudaStream_t st);
size_t select_scratch_words(int ncand, uint32_t nchunks);
// bz_encode.cu
void launch_rle1(const uint16_t* sym, const Geom& g, uint64_t first_block, uint32_t njobs, uint8_t* txt, uint8_t* raw_scratch,
                 uint32_t cap, uint32_t nsub, uint32_t max_raw_bytes, uint32_t nblock_max, EncJob* jobs, cudaStream_t st);
void launch_mtf(const uint8_t* bwt, uint8_t* rank_scratch, uint32_t cap, EncJob* jobs, uint32_t njobs, uint16_t* mtfv, uint32_t mcap, cudaStream_t st);
void launch_huff_pack(const uint16_t* mtfv, uint32_t mcap, EncJob* jobs, uint32_t njobs, uint8_t* sel, uint32_t selcap,
                      uint8_t* out, uint32_t ocap, int level, cudaStream_t st);
// bz_bwt.cu
size_t bwt_smem_bytes(uint32_t cap, int text_in_smem);
size_t bwt_scratch_elems_per_cta(uint32_t cap);
int bwt_ctas_per_sm(uint32_t cap, int text_in_smem);
void launch_bwt(const uint8_t* txt, uint32_t cap, EncJob* jobs, uint32_t njobs, uint8_t* bwt, uint32_t* scratch,
                int grid, int text_in_smem, cudaStream_t st);
// bz_decode.cu
int launch_decode(const uint8_t* payload, const uint64_t* begin, const uint64_t* end, uint32_t njobs, uint32_t nsub, DecJob* jobs,
                  uint16_t* mtfv, uint32_t mcap, uint8_t* q_scratch, uint8_t* bwt, uint32_t cap, uint32_t selcap, cudaStream_t st,
                  cudaEvent_t between = nullptr, uint64_t* endbit = nullptr, uint32_t* crc_out = nullptr,
                  const uint32_t* job_level = nullptr, bool imtf = true);
size_t inv_bwt_scratch_elems(int grid, uint32_t cap);
int inv_bwt_ctas_per_sm(uint32_t cap);
void launch_inv_bwt(const uint8_t* bwt, uint32_t cap, DecJob* jobs, uint32_t njobs, uint32_t* tt_scratch, uint8_t* txt,
                    int grid, cudaStream_t st);
void launch_unrle(const uint8_t* txt, uint8_t* stage_scratch, uint32_t cap, uint32_t nsub, uint32_t max_raw_bytes, DecJob* jobs, uint32_t njobs,
                  uint16_t* sym, const Geom& g, const uint64_t* block_ids, cudaStream_t st);
// bz_stream.cu -- standalone bzip2 streams (input < 2^32 bytes, cut into tiles of kSzTile bytes)
constexpr uint32_t kSzTile = 8192;
struct SzRun { unsigned long long bits; uint32_t err; uint32_t pad; };     // stream bits so far, OR of the blocks' status
uint32_t sz_tiles(uint64_t n);
void launch_sz_runs(const uint8_t* src, uint32_t n, uint32_t* tfirst, uint32_t* tlast, uint32_t* topen, uint32_t* tnext, cudaStream_t st);
void launch_sz_count(const uint8_t* src, uint32_t n, const uint32_t* topen, const uint32_t* tnext, uint32_t* tcount, uint64_t* tobase,
                     cudaStream_t st);
void launch_sz_chain(const uint8_t* src, uint32_t n, const uint32_t* topen, const uint32_t* tnext, const uint64_t* tobase,
                     uint32_t* bitmap, uint64_t bitmap_words, uint32_t nblock_max, uint32_t max_blocks, uint64_t* bout,
                     uint32_t* nb_out, cudaStream_t st);
void launch_sz_locate(const uint8_t* src, uint32_t n, const uint32_t* topen, const uint32_t* tnext, const uint64_t* tobase,
                      const uint64_t* bout, uint32_t* bin, uint32_t nb, cudaStream_t st);
void launch_sz_emit(const uint8_t* src, const uint32_t* bin, const uint64_t* bout, uint32_t k0, uint32_t nj, uint32_t nb,
                    uint8_t* txt, uint32_t cap, EncJob* jobs, uint32_t* combined, cudaStream_t st);
// reading .bz2 data: candidate magics (count pass: tcount + tbase[ntiles + 1]; write pass), prefix sum, chain walk
void launch_bz_magic(const uint8_t* src, uint64_t n, int write, uint32_t* tcount, uint64_t* tbase, uint64_t* cbit, uint8_t* ceos, cudaStream_t st);
void launch_scan_u32(uint32_t count, const uint32_t* in, uint64_t* out, cudaStream_t st);
void launch_bz_chain(const uint8_t* src, uint64_t n, const uint64_t* cbit, const uint8_t* ceos, uint32_t nc, const uint64_t* cend,
                     const uint32_t* ccrc, uint32_t* succ, uint64_t* bbit, uint32_t* blev, uint32_t* res, cudaStream_t st);
// bz_decode.cu: un-RLE1 of standalone blocks into a flat buffer: lengths, then replay at boff[j] with the CRC check
void launch_unrle_len(const uint8_t* txt, uint32_t cap, const DecJob* jobs, uint32_t njobs, uint32_t* lens, cudaStream_t st);
void launch_unrle_flat(const uint8_t* txt, uint32_t cap, DecJob* jobs, uint32_t njobs, const uint64_t* boff, uint8_t* out, cudaStream_t st);
void launch_sz_assemble(const EncJob* jobs, uint32_t nj, const uint8_t* slots, uint32_t ocap, uint64_t* bitoff, SzRun* run,
                        uint8_t* out, uint64_t out_cap, int sm_count, cudaStream_t st);

}  // namespace lfm
