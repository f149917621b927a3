// f3: zstd framing of constant runs for DataBlobs (sm_100a).
//
// PBS stores a chunk as a zstd-compressed DataBlob when that is smaller than the raw one (upstream pbs-datastore
// data_blob.rs `DataBlob::encode`; magic = sha256("Proxmox Backup zstd compressed blob v1.0")[0..8]).  The entropy
// and match stages of zstd are out of scope here; what this file builds is the part of the format that needs neither:
// a standard frame (RFC 8878 section 3.1.1) whose 128 KiB blocks are RLE_Blocks where the input block is one repeated
// byte and Raw_Blocks elsewhere.  Any zstd decoder reads it; on backup data it removes the zero runs of disk images
// and sparse files, which is where most of the compressible bytes are.
//
//   K8a k_zblock_scan : one CTA per 128 KiB block, "are all bytes equal to the first one?" with an exit after the
//                       first 16 KiB that disagrees -- HBM traffic ~ the constant bytes + 16 KiB per other block
//   K8b k_zframe_emit : one CTA per block of the chunks that come out smaller: 3-byte Block_Header + 1 byte (RLE) or
//                       + the raw bytes (funnel-shifted 4-byte copy: the 3-byte headers misalign source and target)
//                       or + a Compressed_Block's content from K9's slots (zlz.cu)
//   K8c k_zframe_hdr  : the 13-byte Frame_Header of each such chunk
#include "internal.cuh"

namespace pbsgpu {

__global__ void __launch_bounds__(256) k_zblock_scan(const uint8_t *base, const uint64_t *off, const uint64_t *len,
                                                     const uint64_t *blk_first, uint32_t n, uint32_t *flags) {
    const uint64_t b = blockIdx.x;
    uint32_t lo = 0, hi = n;   // blk_first[lo] <= b < blk_first[hi]: the LAST such lo (chunks without blocks are skipped)
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (blk_first[mid] <= b) lo = mid; else hi = mid;
    }
    const uint64_t within = (b - blk_first[lo]) * (uint64_t)ZFRAME_BLOCK;
    const uint64_t rem = len[lo] - within;
    const uint32_t size = rem < ZFRAME_BLOCK ? (uint32_t)rem : ZFRAME_BLOCK;
    const uint8_t *p = base + off[lo] + within;
    const uint8_t c = p[0];
    const uint32_t cw = (uint32_t)c * 0x01010101u;
    uint32_t head = (uint32_t)((16 - ((uintptr_t)p & 15)) & 15);
    if (head > size) head = size;
    const uint32_t nvec = (size - head) >> 4, tail0 = head + (nvec << 4);
    bool bad = false;
    if (threadIdx.x < head) bad = p[threadIdx.x] != c;
    if (threadIdx.x < size - tail0) bad |= p[tail0 + threadIdx.x] != c;
    const uint4 *q = (const uint4 *)(p + head);
    for (uint32_t v0 = 0; v0 < nvec; v0 += 1024) {   // 16 KiB per round, then a vote
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const uint32_t v = v0 + k * 256 + threadIdx.x;
            if (v < nvec) {
                const uint4 x = __ldg(q + v);
                bad |= ((x.x ^ cw) | (x.y ^ cw) | (x.z ^ cw) | (x.w ^ cw)) != 0;
            }
        }
        if (__syncthreads_or(bad)) { bad = true; break; }
    }
    bad = __syncthreads_or(bad) != 0;
    if (threadIdx.x == 0) flags[b] = bad ? 0u : (0x100u | c);
}
cudaError_t launch_zblock_scan(const uint8_t *base, const uint64_t *off, const uint64_t *len, const uint64_t *blk_first,
                               uint32_t n, uint64_t n_blocks, uint32_t *flags, cudaStream_t st) {
    if (n_blocks == 0) return cudaSuccess;
    if (n_blocks >= (1ull << 31)) return cudaErrorInvalidValue;
    k_zblock_scan<<<(unsigned)n_blocks, 256, 0, st>>>(base, off, len, blk_first, n, flags);
    return cudaGetLastError();
}

// hdr[e]: bits 0..23 = the Block_Header (Last_Block | Block_Type << 1 | Block_Size << 3), bits 24..31 = the RLE byte
__global__ void __launch_bounds__(256) k_zframe_emit(const uint8_t *base, const uint8_t *lz, uint8_t *stage,
                                                     const uint64_t *src_off, const uint64_t *dst_off, const uint32_t *hdr) {
    const uint64_t e = blockIdx.x;
    const uint32_t h = hdr[e];
    uint8_t *d = stage + dst_off[e];
    if (threadIdx.x < 3) d[threadIdx.x] = (uint8_t)(h >> (8 * threadIdx.x));
    const uint32_t type = (h >> 1) & 3, size = (h & 0xFFFFFFu) >> 3;
    if (type == 1) {
        if (threadIdx.x == 0) d[3] = (uint8_t)(h >> 24);
        return;
    }
    uint8_t *dst = d + 3;
    const uint8_t *src = (type == 2 ? lz : base) + src_off[e];
    uint32_t head = (uint32_t)((4 - ((uintptr_t)dst & 3)) & 3);
    if (head > size) head = size;
    if (threadIdx.x < head) dst[threadIdx.x] = src[threadIdx.x];
    const uint32_t nw = (size - head) >> 2, tail0 = head + (nw << 2);
    if (threadIdx.x < size - tail0) dst[tail0 + threadIdx.x] = src[tail0 + threadIdx.x];
    uint32_t *dst32 = (uint32_t *)(dst + head);
    const uint8_t *sp = src + head;
    const uint32_t mis = (uint32_t)((uintptr_t)sp & 3), sh = mis * 8;
    const uint32_t *src32 = (const uint32_t *)(sp - mis);
    for (uint32_t w = threadIdx.x; w < nw; w += 256) {
        const uint32_t a0 = __ldg(src32 + w), a1 = mis ? __ldg(src32 + w + 1) : 0u;   // a1 holds bytes this word needs when mis != 0
        dst32[w] = __funnelshift_r(a0, a1, sh);
    }
}
cudaError_t launch_zframe_emit(const uint8_t *base, const uint8_t *lz, uint8_t *stage, const uint64_t *src_off,
                               const uint64_t *dst_off, const uint32_t *hdr, uint64_t n_entries, cudaStream_t st) {
    if (n_entries == 0) return cudaSuccess;
    if (n_entries >= (1ull << 31)) return cudaErrorInvalidValue;
    k_zframe_emit<<<(unsigned)n_entries, 256, 0, st>>>(base, lz, stage, src_off, dst_off, hdr);
    return cudaGetLastError();
}

// Frame_Header: Magic_Number 0xFD2FB528 LE | Frame_Header_Descriptor 0xE0 (Frame_Content_Size_flag 3 = 8 bytes,
// Single_Segment_flag: no Window_Descriptor, the window is the content) | Frame_Content_Size u64 LE
__global__ void k_zframe_hdr(uint8_t *stage, const uint64_t *frame_off, const uint64_t *content_len, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint8_t *d = stage + frame_off[i];
    d[0] = 0x28; d[1] = 0xB5; d[2] = 0x2F; d[3] = 0xFD; d[4] = 0xE0;
    const uint64_t L = content_len[i];
    for (int k = 0; k < 8; k++) d[5 + k] = (uint8_t)(L >> (8 * k));
}
cudaError_t launch_zframe_hdr(uint8_t *stage, const uint64_t *frame_off, const uint64_t *content_len, uint32_t n, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    k_zframe_hdr<<<(n + 255) / 256, 256, 0, st>>>(stage, frame_off, content_len, n);
    return cudaGetLastError();
}

}  // namespace pbsgpu
