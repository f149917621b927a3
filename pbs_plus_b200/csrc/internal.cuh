// pbs_plus_b200/csrc/internal.cuh -- declarations shared by the kernels and the C ABI.
// Product code: never includes anything under oracle/.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/pbsgpu.h"

namespace pbsgpu {

// Candidate keys: (stream << 40) | position.  Limits: position < 2^40 (1 TiB per
// stream), stream index < 2^24.
constexpr int KEY_POS_BITS = 40;
constexpr uint64_t KEY_POS_MASK = (1ull << KEY_POS_BITS) - 1;
constexpr uint64_t KEY_SENTINEL = ~0ull;

// upstream scan() tests only after the 64-byte window is full AND has rolled once
__host__ __device__ inline uint32_t min_effective(uint32_t cmin) { return cmin > 64u ? cmin : 65u; }

struct ChunkRef {      // device-side chunk descriptor produced by resolve
    uint32_t stream;
    uint32_t len;      // <= max chunk size <= 2^31
    uint64_t start;    // offset within stream
};

// ---- scan (K1) ---------------------------------------------------------------
// Tuned kernel geometry: one warp owns a tile of 32 lanes x LANE_SPAN bytes.
constexpr int LANE_SPAN = 272;               // 17 x 16 B: conflict-free LDS.128 (lane stride = 17 quads)
constexpr int WARP_TILE = 32 * LANE_SPAN;    // 8704 B
constexpr int SIMPLE_SPAN = 1024;            // cross-check kernel: bytes per thread

struct ScanArgs {
    const uint8_t *base;
    const uint64_t *off;         // [n]
    const uint64_t *len;         // [n]
    const uint64_t *tile_first;  // [n+1] exclusive prefix of per-stream tile counts
    uint32_t n_streams;
    uint64_t total_tiles;
    uint32_t mask, break_min;
    const uint32_t *table;       // [256] device
    uint64_t *cand;              // candidate keys
    uint64_t cand_cap;
    unsigned long long *cand_count;
};
cudaError_t launch_scan_simple(const ScanArgs &a, cudaStream_t st);
cudaError_t launch_scan_tuned(const ScanArgs &a, const uint32_t *rot_table /*[256][64]*/, int sm_count, cudaStream_t st);
cudaError_t launch_scan_lanes(const ScanArgs &a, const uint32_t *rot_table, int sm_count, uint64_t extent, cudaStream_t st);
uint64_t scan_lanes_super_bytes();
uint32_t scan_lanes_align();
uint32_t scan_lanes_steps();
cudaError_t launch_build_rot_table(const uint32_t *table, uint32_t *rot_table, cudaStream_t st);
size_t scan_tuned_smem_bytes();

// ---- resolve (K2) --------------------------------------------------------------
struct ResolveArgs {
    const uint64_t *keys_sorted;           // sorted candidate keys (KEY_SENTINEL padded)
    const unsigned long long *cand_count;  // device
    uint64_t cand_cap;
    const uint64_t *len;                   // [n]
    uint32_t n_streams;
    uint32_t cmin, cmax;
    int eof;                               // 1: emit final short chunk
    uint32_t *counts;                      // [n] chunks per stream
    uint64_t *chunk_first;                 // [n+1]
    ChunkRef *chunks;                      // [chunk_cap]
    uint64_t chunk_cap;
    uint64_t *consumed;                    // [n] bytes covered by emitted chunks (eof==0)
    unsigned long long *n_chunks;          // device total
};
cudaError_t launch_resolve(const ResolveArgs &a, cudaStream_t st);   // count + scan + write (3 launches)
cudaError_t launch_append_keys(const uint64_t *keys, uint64_t n, uint64_t *cand, uint64_t cand_cap, unsigned long long *cand_count,
                               cudaStream_t st);

// ---- SHA-256 (K3) ----------------------------------------------------------------
struct ShaArgs {
    const uint8_t *base;
    const uint64_t *off;                 // [n_streams] stream offsets (NULL: chunks[].start is absolute)
    const ChunkRef *chunks;
    const uint32_t *order;               // processing order (longest first) or NULL
    const unsigned long long *n_chunks;  // device count
    uint64_t chunk_cap;                  // launch bound
    uint8_t *digests;                    // [chunk_cap][32], indexed by chunk id
    // hybrid launch: the first *n_head entries of `order` (the longest chunks) go to the
    // latency-optimised split kernel (part 1), the rest to the throughput kernel (part 2).
    const unsigned long long *n_head;    // device; NULL with part 0
    const unsigned long long *n_mid;     // device; end of the "mid" class (>= *n_head); NULL unless part is 3 or 4
    int part;                            // 0 = everything, 1 = head only, 2 = everything but the head,
                                         // 3 = mid class [head, mid), 4 = short class [mid, n)
    // long-chunk arena (part 1 only; NULL = read the chunks where they lie): head chunk t was copied to
    // arena + arena_off[t] + (its source address mod 16) by k_arena_gather
    const uint8_t *arena = nullptr;
    const uint64_t *arena_off = nullptr;
};
// per-context tuning knobs of K3 (read from the environment once per pbsgpu_open)
struct ShaTune {
    int mode = 2;        // PBSGPU_SHA_MODE: instruction mix of the throughput kernel (0,1,2,3,7) or split-only (10..13)
    int hybrid = 1;      // PBSGPU_SHA_HYBRID: 0 throughput kernel only, 1 hybrid when partitioned, 2 hybrid always
    int thr_x10 = 25;    // PBSGPU_HYBRID_THR_X10: chunks longer than thr_x10/10 x avg take the latency kernel
    int serial = 0;      // PBSGPU_HYBRID_SERIAL: latency kernel on the job's own stream (diagnostic)
    int spread_kb = 30;  // PBSGPU_SPLIT_SPREAD_KB: dummy dynamic shared memory per latency CTA (caps CTAs per SM)
    int head_per_sm = 32; // PBSGPU_HYBRID_HEAD_PER_SM: chunks per SM of the long partition (and job) that may take the latency kernel
    int mid_x10 = 0;      // PBSGPU_BULK_MID_X10: > 0: bulk chunks longer than mid_x10/10 x avg are launched on a HIGH-PRIORITY bulk
                          // stream of their own, so the longer chains of every job in flight start before the short ones
};
cudaError_t launch_sha_simple(const ShaArgs &a, cudaStream_t st);
cudaError_t launch_sha_tuned(const ShaArgs &a, const ShaTune &tune, cudaStream_t st);   // throughput kernel
cudaError_t launch_sha_split(const ShaArgs &a, const ShaTune &tune, cudaStream_t st);   // latency kernel
cudaError_t launch_split_point(const uint32_t *len_sorted_desc, const unsigned long long *n_chunks, uint64_t cap,
                               uint32_t threshold, unsigned long long max_head, unsigned long long *n_head,
                               uint32_t threshold_mid, unsigned long long *n_mid, cudaStream_t st);
// long-chunk arena: plan the placement of the head chunks inside a reservation of `arena_cap` bytes (trims *n_head, whole
// groups of 32, to what fits), then copy them there
cudaError_t launch_arena_plan(const ShaArgs &a, unsigned long long *n_head, uint64_t arena_cap, uint64_t *arena_off,
                              cudaStream_t st);
cudaError_t launch_arena_gather(const ShaArgs &a, uint8_t *arena, const uint64_t *arena_off, int sms, cudaStream_t st);
cudaError_t launch_len_keys(const ChunkRef *chunks, const unsigned long long *n_chunks, uint64_t cap,
                            uint32_t *keys, uint32_t *vals, cudaStream_t st);
cudaError_t launch_pack_chunks(const ChunkRef *chunks, const uint8_t *digests, const uint8_t *hit,
                               const unsigned long long *n_chunks, uint64_t cap, pbsgpu_chunk *out, cudaStream_t st);

// ---- f3: zstd framing of constant runs (zframe.cu) ---------------------------------------
constexpr uint32_t ZFRAME_BLOCK = 128u * 1024u;   // Block_Maximum_Size
constexpr uint32_t ZFRAME_HEADER = 13;            // magic 4 + descriptor 1 + content size 8
cudaError_t launch_zblock_scan(const uint8_t *base, const uint64_t *off, const uint64_t *len, const uint64_t *blk_first,
                               uint32_t n, uint64_t n_blocks, uint32_t *flags, cudaStream_t st);
// Block_Type 2 (Compressed_Block) entries copy from `lz` (K9's slots) instead of `base`; NULL when there are none
cudaError_t launch_zframe_emit(const uint8_t *base, const uint8_t *lz, uint8_t *stage, const uint64_t *src_off,
                               const uint64_t *dst_off, const uint32_t *hdr, uint64_t n_entries, cudaStream_t st);
cudaError_t launch_zframe_hdr(uint8_t *stage, const uint64_t *frame_off, const uint64_t *content_len, uint32_t n, cudaStream_t st);

// ---- f3: zstd match stage (K9, zlz.cu) ------------------------------------------------------
// The greedy parse's constants; oracle/zstd_lz.py (LZ_HLOG, LZ_SEG, LZ_MINMATCH) states the same parse.
constexpr int ZLZ_HLOG = 14;          // hash table of 2^14 positions
constexpr uint32_t ZLZ_SEG = 1024;    // positions look up only earlier segments of this length
constexpr uint32_t ZLZ_MINMATCH = 4;
constexpr uint32_t ZLZ_SLOT = ZFRAME_BLOCK + 64;   // bytes per block in K9's output (a kept block is < its input)
// Block b of the list (blk_src[b] bytes into base, blk_size[b] <= ZFRAME_BLOCK bytes) -> Block_Content at
// slots + b * ZLZ_SLOT + (info[b] >> 24) of (info[b] & 0xFFFFFF) bytes, or info[b] = 0: keep the block raw.  The blocks
// go in passes of pass_blocks; `scratch` holds zlz_scratch_bytes_per_block() per block of a pass.
uint64_t zlz_scratch_bytes_per_block();
cudaError_t launch_zlz(const uint8_t *base, const uint64_t *blk_src, const uint32_t *blk_size, uint32_t n_blk, uint8_t *slots,
                       uint32_t *info, void *scratch, uint32_t pass_blocks, cudaStream_t st);

// ---- digest set (K4) ----------------------------------------------------------------
struct SetTable {
    uint64_t *tags;     // [cap] 0 = empty
    uint64_t *keys;     // [cap][4]
    uint64_t cap;       // power of two
};
cudaError_t launch_set_make_keys(const uint8_t *d32, uint64_t n, uint64_t *tag, uint32_t *idx, cudaStream_t st);
cudaError_t launch_set_mark_probe_insert(SetTable t, const uint8_t *d32, const uint64_t *tag_sorted,
                                         const uint32_t *idx_sorted, uint64_t n, int do_insert, uint8_t *hit,
                                         uint8_t *is_rep_miss, unsigned long long *n_new, cudaStream_t st);
cudaError_t launch_set_rehash(SetTable from, SetTable to, cudaStream_t st);
// fused form (K4 on a job's stream): the element count lives on the device, `cap` bounds the launch; nothing happens when
// *guard > guard_max.  Padding entries (index >= *n_dev) get the all-ones tag and sort last.
cudaError_t launch_set_make_keys_dev(const uint8_t *d32, const unsigned long long *n_dev, uint64_t cap, uint64_t *tag, uint32_t *idx,
                                     cudaStream_t st);
cudaError_t launch_set_mark_probe_insert_dev(SetTable t, const uint8_t *d32, const uint64_t *tag_sorted, const uint32_t *idx_sorted,
                                             const unsigned long long *n_dev, uint64_t cap, const unsigned long long *guard,
                                             uint64_t guard_max, uint8_t *hit, uint8_t *is_rep_miss, unsigned long long *n_new,
                                             cudaStream_t st);
// multi-GPU merge: compact the padded all-gather payload [rank][max_n][32] into global order [sum(counts)][32]
cudaError_t launch_set_compact_gather(const uint8_t *padded, const uint64_t *counts_dev, uint32_t nranks, uint64_t max_n,
                                      uint8_t *dense, cudaStream_t st);

// ---- CRC-32 (K6, DataBlob checksums) -----------------------------------------------------
cudaError_t launch_crc32(const uint8_t *base, const uint64_t *off, const uint64_t *len, const uint64_t *wb_first,
                         uint32_t n, uint64_t total_wb, const void *tables, uint32_t *part_crc, uint32_t *out,
                         int sm_count, cudaStream_t st);
cudaError_t launch_crc32_tiled(const uint8_t *base, const uint64_t *off, const uint64_t *len,
                               const uint64_t *region_first, uint32_t n, uint64_t total_regions, const void *tables,
                               uint32_t *part_crc, uint32_t *out, int sm_count, cudaStream_t st);
uint64_t crc_region_bytes();
size_t crc_tables_bytes();
// K7 (xxh3.cu)
size_t xxh3_tables_bytes();
void xxh3_fill_tables_host(void *dst);
cudaError_t launch_xxh3_pass(const uint8_t *base, const uint64_t *off, const uint64_t *len, const uint64_t *first, uint32_t n,
                             uint64_t total, uint64_t win_lo, uint64_t win, const void *tab, uint64_t *S, uint64_t *state,
                             uint64_t *out, cudaStream_t st);
cudaError_t launch_xxh3_small(const uint8_t *base, const uint64_t *off, const uint64_t *len, uint32_t n, const void *tab,
                              uint64_t *out, cudaStream_t st);
void crc_fill_tables_host(void *dst);
uint64_t crc_wb_bytes();

// ---- corpus (K5) ------------------------------------------------------------------
cudaError_t launch_corpus_fill(const pbsgpu_corpus &c, uint64_t first_file, uint32_t n_files, uint8_t *dst,
                               uint64_t stride, cudaStream_t st);

}  // namespace pbsgpu
