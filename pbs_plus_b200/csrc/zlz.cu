// f3: the match stage of zstd for DataBlobs (sm_100a), K9.
//
// Turns the non-constant 128 KiB blocks of a batch into zstd Compressed_Blocks (RFC 8878 3.1.1.3) built from a greedy,
// block-local parse: Raw_Literals_Block, then the sequences with LL, ML and OF all in Predefined_Mode (no table
// descriptions, no repeat offsets).  The parse is fixed so that oracle/zstd_lz.py `lz_parse` and this file agree bit for
// bit; zframe.cu's frame and block grid stay as they are, and capi_aux.cu keeps a compressed block only where it is
// smaller than the block.
//
// Parse (constants in internal.cuh):  h(p) = (u32le(block[p..p+4]) * 0x9E3779B1) >> (32 - ZLZ_HLOG) for p <= S - 4;
// cand(p) = the largest q < ZLZ_SEG * floor(p / ZLZ_SEG) with h(q) = h(p) -- earlier SEGMENTS only, so one segment's
// lookups all read the table as it stood after the segments before it; m(p) = cand(p) exists and the 4 bytes there and
// at p agree.  Walk from p = 0: the next q >= p with m(q) starts a match of the longest common prefix of block[cand(q)..]
// and block[q..] (capped at the block end), p = q + length; no match left = trailing literals.
//
// The blocks go in passes of a bounded number (scratch: cand + m bitmap per block of the pass, ~528 KiB), two kernels each:
//   K9a k_zlz_scan   : one CTA per block, data-parallel.  Per segment: hash, lookup in a 2^14-entry table in shared
//                      memory, 4-byte check, m bitmap word by ballot, cand to scratch; then the segment's inserts
//                      (atomicMax).
//   K9b k_zlz_encode : one WARP per block -- the walk is serial, so an SM runs many walkers side by side.  The next
//                      match start by ballot over 32 bitmap words, the match length by 128-byte warp compares, the
//                      sequence list written over cand; then the literal runs into the block's slot, then lane 0
//                      FSE-encodes the sequences behind them (64-bit bit accumulator).
#include <algorithm>
#include <vector>

#include "internal.cuh"

namespace pbsgpu {

namespace {

constexpr int SCAN_THREADS = 512;
constexpr int ENC_WARPS = 8;                         // blocks per CTA of K9b
constexpr uint32_t NWORDS = ZFRAME_BLOCK / 32;       // m bitmap words per block
constexpr uint32_t CAND_WORDS = ZFRAME_BLOCK + 4;    // cand per position; also holds the <= S/4 sequences + 1 (16 B each)

// Predefined FSE tables (RFC 8878 3.1.1.3.2.2) in encoder form plus the code tables, filled on the host
struct LzTables {
    uint8_t enc_ll[36][64], enc_ml[53][64], enc_of[29][32];   // [symbol][decoder's next state] -> state of the symbol
    uint8_t nb_ll[64], nb_ml[64], nb_of[32];                  // per state: nbBits
    uint8_t base_ll[64], base_ml[64], base_of[32];            // per state: baseline
    uint8_t first_ll[36], first_ml[53], first_of[29];         // lowest state of each symbol (start of the last sequence)
    uint8_t code_ll[64], code_ml[128];                        // LL code of lengths < 64, ML code of (length - 3) < 128
    uint32_t lbase_ll[36], lbase_ml[53];                      // code -> baseline value
    uint8_t lbits_ll[36], lbits_ml[53];                       // code -> extra bits
};
__constant__ LzTables c_lz;

const int8_t LL_NORM[36] = {4, 3, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 1, 1, 1, 2, 2, 2, 2, 2, 2, 2, 2, 2, 3, 2, 1, 1, 1, 1, 1, -1, -1, -1, -1};
const int8_t ML_NORM[53] = {1, 4, 3, 2, 2, 2, 2, 2, 2, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1,
                            1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, -1, -1, -1, -1, -1, -1, -1};
const int8_t OF_NORM[29] = {1, 1, 1, 1, 1, 1, 2, 2, 2, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, -1, -1, -1, -1, -1};
const uint32_t LL_BASE[36] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 18, 20, 22, 24, 28, 32, 40, 48, 64,
                              128, 256, 512, 1024, 2048, 4096, 8192, 16384, 32768, 65536};
const uint8_t LL_BITS[36] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 3, 3, 4, 6, 7, 8, 9, 10, 11, 12,
                             13, 14, 15, 16};
const uint32_t ML_BASE[53] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22, 23, 24, 25, 26, 27, 28,
                              29, 30, 31, 32, 33, 34, 35, 37, 39, 41, 43, 47, 51, 59, 67, 83, 99, 131, 259, 515, 1027, 2051,
                              4099, 8195, 16387, 32771, 65539};
const uint8_t ML_BITS[53] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0,
                             1, 1, 1, 1, 2, 2, 3, 3, 4, 4, 5, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16};

// RFC 8878 4.1.1 decoding table -> per state nbBits / baseline, and the inverse the encoder needs
void fse_tables(const int8_t *norm, int nsym, int log, uint8_t *enc /*[nsym][1 << log]*/, uint8_t *nb, uint8_t *base, uint8_t *first) {
    const int size = 1 << log;
    std::vector<int> sym(size), next(nsym);
    int high = size - 1;
    for (int s = 0; s < nsym; s++)
        if (norm[s] == -1) sym[high--] = s;
    int pos = 0;
    const int step = (size >> 1) + (size >> 3) + 3;
    for (int s = 0; s < nsym; s++)
        for (int i = 0; i < norm[s]; i++) {
            sym[pos] = s;
            do pos = (pos + step) & (size - 1); while (pos > high);
        }
    for (int s = 0; s < nsym; s++) { next[s] = norm[s] == -1 ? 1 : norm[s]; first[s] = 0xFF; }
    for (int u = 0; u < size; u++) {
        const int s = sym[u], x = next[s]++;
        int hb = 31 - __builtin_clz((unsigned)x);
        nb[u] = (uint8_t)(log - hb);
        base[u] = (uint8_t)((x << nb[u]) - size);
        if (first[s] == 0xFF) first[s] = (uint8_t)u;
        for (int t = base[u]; t < base[u] + (1 << nb[u]); t++) enc[s * size + t] = (uint8_t)u;
    }
}

const LzTables &host_tables() {
    static const LzTables t = [] {
        LzTables h{};
        fse_tables(LL_NORM, 36, 6, &h.enc_ll[0][0], h.nb_ll, h.base_ll, h.first_ll);
        fse_tables(ML_NORM, 53, 6, &h.enc_ml[0][0], h.nb_ml, h.base_ml, h.first_ml);
        fse_tables(OF_NORM, 29, 5, &h.enc_of[0][0], h.nb_of, h.base_of, h.first_of);
        for (int c = 0; c < 36; c++) { h.lbase_ll[c] = LL_BASE[c]; h.lbits_ll[c] = LL_BITS[c]; }
        for (int c = 0; c < 53; c++) { h.lbase_ml[c] = ML_BASE[c]; h.lbits_ml[c] = ML_BITS[c]; }
        for (uint32_t v = 0, c = 0; v < 64; v++) { while (c + 1 < 36 && LL_BASE[c + 1] <= v) c++; h.code_ll[v] = (uint8_t)c; }
        for (uint32_t v = 0, c = 0; v < 128; v++) { while (c + 1 < 53 && ML_BASE[c + 1] <= v + 3) c++; h.code_ml[v] = (uint8_t)c; }
        return h;
    }();
    return t;
}

__device__ __forceinline__ uint32_t highbit(uint32_t v) { return 31 - __clz(v); }

// 4 bytes at p, little endian, reading only the aligned words that hold them
__device__ __forceinline__ uint32_t load4(const uint8_t *p) {
    const uint32_t mis = (uint32_t)((uintptr_t)p & 3);
    const uint32_t *w = (const uint32_t *)(p - mis);
    const uint32_t a0 = __ldg(w);
    return mis ? __funnelshift_r(a0, __ldg(w + 1), mis * 8) : a0;
}

// forward bitstream, LSB first; a field never straddles the 64-bit accumulator
struct BitWriter {
    uint8_t *dst;
    uint32_t pos, cap;
    uint64_t acc = 0;
    uint32_t nbits = 0;
    bool overflow = false;
    __device__ void flush() {
        const uint32_t nbytes = nbits >> 3;
        if (pos + 8 > cap) overflow = true;
        else
            for (uint32_t k = 0; k < nbytes; k++) dst[pos + k] = (uint8_t)(acc >> (8 * k));
        pos += nbytes;
        acc = nbytes == 8 ? 0 : acc >> (8 * nbytes);
        nbits &= 7;
    }
    __device__ void put(uint32_t v, uint32_t nb) {
        if (nbits + nb > 64) flush();
        acc |= (uint64_t)(v & ((1u << nb) - 1)) << nbits;   // nb <= 17
        nbits += nb;
    }
    __device__ void close() {
        put(1, 1);
        flush();
        if (nbits) {
            if (pos + 1 > cap) overflow = true;
            else dst[pos] = (uint8_t)acc;
            pos++;
        }
    }
};

}  // namespace

struct Seq { uint32_t lit_src, lit_dst, ml, off; };   // literal run [lit_src, next match) lands at lit_dst

// K9a: one CTA per block of the pass -> the m bitmap and cand of every match start, in the block's scratch region
__global__ void __launch_bounds__(SCAN_THREADS) k_zlz_scan(const uint8_t *base, const uint64_t *blk_src, const uint32_t *blk_size,
                                                           uint32_t *cand_scratch, uint32_t *bitmap_scratch) {
    extern __shared__ uint32_t table[];   // [1 << ZLZ_HLOG]: 1 + the last inserted position, 0 = none
    const uint32_t tid = threadIdx.x, lane = tid & 31;
    const uint8_t *src = base + blk_src[blockIdx.x];
    const uint32_t S = blk_size[blockIdx.x];
    uint32_t *cand = cand_scratch + (uint64_t)blockIdx.x * CAND_WORDS;
    uint32_t *bitmap = bitmap_scratch + (uint64_t)blockIdx.x * NWORDS;
    for (uint32_t i = tid; i < (1u << ZLZ_HLOG); i += SCAN_THREADS) table[i] = 0;
    __syncthreads();
    const uint32_t nseg = (S + ZLZ_SEG - 1) / ZLZ_SEG;
    for (uint32_t sg = 0; sg < nseg; sg++) {
        uint32_t h[ZLZ_SEG / SCAN_THREADS];
#pragma unroll
        for (int k = 0; k < ZLZ_SEG / SCAN_THREADS; k++) {
            const uint32_t p = sg * ZLZ_SEG + k * SCAN_THREADS + tid;
            bool m = false;
            h[k] = ~0u;
            if (p + 4 <= S) {
                const uint32_t u = load4(src + p);
                h[k] = (u * 0x9E3779B1u) >> (32 - ZLZ_HLOG);
                const uint32_t c1 = table[h[k]];
                if (c1 && load4(src + c1 - 1) == u) { m = true; cand[p] = c1 - 1; }
            }
            const uint32_t word = __ballot_sync(0xFFFFFFFFu, m);
            if (lane == 0) bitmap[p >> 5] = word;
        }
        __syncthreads();   // every lookup of the segment precedes its inserts
#pragma unroll
        for (int k = 0; k < ZLZ_SEG / SCAN_THREADS; k++)
            if (h[k] != ~0u) atomicMax(&table[h[k]], sg * ZLZ_SEG + k * SCAN_THREADS + tid + 1);
        __syncthreads();
    }
}

// K9b: one warp per block of the pass -> walk, literal runs, FSE; info[b] as in internal.cuh
__global__ void __launch_bounds__(ENC_WARPS * 32) k_zlz_encode(const uint8_t *base, const uint64_t *blk_src, const uint32_t *blk_size,
                                                               uint32_t n, uint8_t *slots, uint32_t *info,
                                                               uint32_t *cand_scratch, const uint32_t *bitmap_scratch) {
    const uint32_t lane = threadIdx.x & 31, b = blockIdx.x * ENC_WARPS + (threadIdx.x >> 5);
    if (b >= n) return;
    const uint8_t *src = base + blk_src[b];
    const uint32_t S = blk_size[b];
    uint8_t *slot = slots + (uint64_t)b * ZLZ_SLOT;
    const uint32_t *cand = cand_scratch + (uint64_t)b * CAND_WORDS;
    const uint32_t *bitmap = bitmap_scratch + (uint64_t)b * NWORDS;
    // sequence k goes to cand words [4k, 4k + 4): every sequence covers >= 4 bytes, so the walk has passed them for good
    Seq *seqs = (Seq *)(cand_scratch + (uint64_t)b * CAND_WORDS);
    const uint32_t nw = (S + ZLZ_SEG - 1) / ZLZ_SEG * (ZLZ_SEG / 32);
    uint32_t p = 0, nseq = 0, lit = 0;
    while (true) {   // the greedy walk
        uint32_t q = ~0u, w = p >> 5;
        if (w < nw) {
            const uint32_t first = bitmap[w] & (~0u << (p & 31));
            if (first) q = (w << 5) + __ffs(first) - 1;
            for (w++; q == ~0u && w < nw; w += 32) {   // 32 bitmap words = 1024 positions per ballot
                const uint32_t x = w + lane < nw ? bitmap[w + lane] : 0u;
                const uint32_t any = __ballot_sync(0xFFFFFFFFu, x != 0);
                if (any) {
                    const uint32_t l0 = __ffs(any) - 1;
                    q = ((w + l0) << 5) + __ffs(__shfl_sync(0xFFFFFFFFu, x, l0)) - 1;
                }
            }
        }
        if (q == ~0u) break;
        const uint32_t c = cand[q], lim = S - q;
        uint32_t L = ZLZ_MINMATCH;
        while (L < lim) {   // 128 bytes per step
            const uint32_t k = L + lane * 4;
            uint32_t diff = 0;
            if (k + 4 <= lim) diff = load4(src + c + k) ^ load4(src + q + k);
            else
                for (uint32_t j = 0; k + j < lim; j++) diff |= (uint32_t)(src[c + k + j] ^ src[q + k + j]) << (8 * j);
            const uint32_t any = __ballot_sync(0xFFFFFFFFu, diff != 0);
            if (any) {
                const uint32_t l0 = __ffs(any) - 1;
                L += l0 * 4 + (__ffs(__shfl_sync(0xFFFFFFFFu, diff, l0)) - 1) / 8;
                break;
            }
            L += 128;
        }
        if (L > lim) L = lim;
        __syncwarp();   // every lane has read cand[q] before lane 0 may overwrite it
        if (lane == 0) seqs[nseq] = Seq{p, lit, L, q - c};
        lit += q - p;
        nseq++;
        p = q + L;
    }
    if (lane == 0) seqs[nseq] = Seq{p, lit, 0, 0};   // the trailing literals
    __syncwarp();
    const uint32_t nlit = lit + (S - p);
    const uint32_t lhs = nlit <= 31 ? 1 : nlit <= 4095 ? 2 : 3;
    // a block without a match, or whose literals alone leave no gain, stays raw
    if (nseq == 0 || lhs + nlit + 2 + (nseq >= 128) + (nseq >= 0x7F00) >= S) {
        if (lane == 0) info[b] = 0;
        return;
    }
    // literal runs: the content starts at slot + 3 - lhs so that the literals always start at slot + 3
    uint8_t *lits = slot + 3;
    for (uint32_t r = 0; r <= nseq; r++) {
        const Seq s = seqs[r];
        const uint32_t len = r < nseq ? seqs[r + 1].lit_dst - s.lit_dst : S - s.lit_src;
        for (uint32_t j = lane; j < len; j += 32) lits[s.lit_dst + j] = src[s.lit_src + j];
    }
    if (lane != 0) return;
    // headers and the FSE bitstream
    uint8_t *content = slot + 3 - lhs;
    if (lhs == 1) content[0] = (uint8_t)(nlit << 3);
    else if (lhs == 2) { const uint32_t v = 0x4u | (nlit << 4); content[0] = (uint8_t)v; content[1] = (uint8_t)(v >> 8); }
    else { const uint32_t v = 0xCu | (nlit << 4); content[0] = (uint8_t)v; content[1] = (uint8_t)(v >> 8); content[2] = (uint8_t)(v >> 16); }
    uint32_t pos = 3 + nlit;
    if (nseq < 128) slot[pos++] = (uint8_t)nseq;
    else if (nseq < 0x7F00) { slot[pos++] = (uint8_t)((nseq >> 8) + 128); slot[pos++] = (uint8_t)nseq; }
    else { slot[pos++] = 255; slot[pos++] = (uint8_t)(nseq - 0x7F00); slot[pos++] = (uint8_t)((nseq - 0x7F00) >> 8); }
    slot[pos++] = 0;   // Symbol_Compression_Modes: LL, OF, ML Predefined_Mode
    BitWriter bw{slot, pos, ZLZ_SLOT};
    uint32_t sll = 0, sml = 0, sof = 0;
    // the decoder reads backward: start at the last sequence, end with the initial states
    for (int32_t r = (int32_t)nseq - 1; r >= 0; r--) {
        const Seq s = seqs[r];
        const uint32_t ll = seqs[r + 1].lit_dst - s.lit_dst, ml = s.ml, ofv = s.off + 3;
        const uint32_t llc = ll < 64 ? c_lz.code_ll[ll] : highbit(ll) + 19;
        const uint32_t mlc = ml - 3 < 128 ? c_lz.code_ml[ml - 3] : highbit(ml - 3) + 36;
        const uint32_t ofc = highbit(ofv);
        if (r == (int32_t)nseq - 1) {
            sll = c_lz.first_ll[llc]; sml = c_lz.first_ml[mlc]; sof = c_lz.first_of[ofc];
        } else {
            uint32_t x = c_lz.enc_of[ofc][sof]; bw.put(sof - c_lz.base_of[x], c_lz.nb_of[x]); sof = x;
            x = c_lz.enc_ml[mlc][sml]; bw.put(sml - c_lz.base_ml[x], c_lz.nb_ml[x]); sml = x;
            x = c_lz.enc_ll[llc][sll]; bw.put(sll - c_lz.base_ll[x], c_lz.nb_ll[x]); sll = x;
        }
        bw.put(ll - c_lz.lbase_ll[llc], c_lz.lbits_ll[llc]);
        bw.put(ml - c_lz.lbase_ml[mlc], c_lz.lbits_ml[mlc]);
        bw.put(ofv - (1u << ofc), ofc);
    }
    bw.put(sml, 6); bw.put(sof, 5); bw.put(sll, 6);
    bw.close();
    const uint32_t size = bw.pos - (3 - lhs);
    info[b] = (bw.overflow || size >= S) ? 0u : (size | ((3 - lhs) << 24));
}

uint64_t zlz_scratch_bytes_per_block() { return (uint64_t)(CAND_WORDS + NWORDS) * 4; }

cudaError_t launch_zlz(const uint8_t *base, const uint64_t *blk_src, const uint32_t *blk_size, uint32_t n_blk, uint8_t *slots,
                       uint32_t *info, void *scratch, uint32_t pass_blocks, cudaStream_t st) {
    if (n_blk == 0) return cudaSuccess;
    const int smem = (1 << ZLZ_HLOG) * 4;
    cudaError_t e = cudaFuncSetAttribute(k_zlz_scan, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e == cudaSuccess) e = cudaMemcpyToSymbolAsync(c_lz, &host_tables(), sizeof(LzTables), 0, cudaMemcpyHostToDevice, st);
    uint32_t *cand = (uint32_t *)scratch;
    uint32_t *bitmap = cand + (uint64_t)pass_blocks * CAND_WORDS;
    for (uint32_t lo = 0; e == cudaSuccess && lo < n_blk; lo += pass_blocks) {
        const uint32_t cnt = std::min(pass_blocks, n_blk - lo);
        k_zlz_scan<<<cnt, SCAN_THREADS, smem, st>>>(base, blk_src + lo, blk_size + lo, cand, bitmap);
        k_zlz_encode<<<(cnt + ENC_WARPS - 1) / ENC_WARPS, ENC_WARPS * 32, 0, st>>>(base, blk_src + lo, blk_size + lo, cnt,
                                                                                  slots + (uint64_t)lo * ZLZ_SLOT, info + lo, cand, bitmap);
        e = cudaGetLastError();
    }
    return e;
}

}  // namespace pbsgpu
