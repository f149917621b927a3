// pbs_plus_b200/csrc/capi_aux.cu -- C ABI of the "next" rows of SURVEY.md section 8: dynamic index images (f1), the commit
// walk's per-file XXH3-64 (f2) and DataBlob framing + CRC-32 for new chunks (f3).
#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "host.hpp"

using namespace pbsgpu;

// ---------------------------------------------------------------------------
// f1: dynamic index images
// ---------------------------------------------------------------------------
static const uint8_t DIDX_MAGIC[8] = {28, 145, 78, 165, 25, 186, 179, 205};
extern "C" int pbsgpu_sha256_batch(pbsgpu_ctx *, const void *, const uint64_t *, const uint64_t *, uint32_t, uint8_t *);

extern "C" uint64_t pbsgpu_didx_size(uint64_t n) { return 4096 + n * 40; }

extern "C" int pbsgpu_didx_build(pbsgpu_ctx *ctx, const pbsgpu_chunk *chunks, uint64_t n, const uint8_t uuid[16],
                                 int64_t ctime, uint8_t *out, uint64_t cap) {
    if (!ctx || (n && !chunks) || !out || !uuid) return PBSGPU_EINVAL;
    if (cap < pbsgpu_didx_size(n)) return fail(ctx, PBSGPU_ERANGE, "didx buffer too small: %llu < %llu", (unsigned long long)cap, (unsigned long long)pbsgpu_didx_size(n));
    memset(out, 0, 4096);
    memcpy(out, DIDX_MAGIC, 8);
    memcpy(out + 8, uuid, 16);
    for (int i = 0; i < 8; i++) out[24 + i] = (uint8_t)((uint64_t)ctime >> (8 * i));
    uint64_t total = 0, prev_end = 0;
    uint32_t prev_stream = 0;
    for (uint64_t i = 0; i < n; i++) {
        if (i == 0 || chunks[i].stream != prev_stream) prev_end = 0;
        if (chunks[i].end_off < prev_end) return fail(ctx, PBSGPU_EINVAL, "chunk records not ordered by (stream, end_off) at %llu", (unsigned long long)i);
        total += chunks[i].end_off - prev_end;
        prev_end = chunks[i].end_off; prev_stream = chunks[i].stream;
        uint8_t *e = out + 4096 + i * 40;
        for (int k = 0; k < 8; k++) e[k] = (uint8_t)(total >> (8 * k));
        memcpy(e + 8, chunks[i].digest, 32);
    }
    uint64_t off0 = 0, len0 = n * 40;
    return pbsgpu_sha256_batch(ctx, out + 4096, &off0, &len0, 1, out + 32);   // index_csum (GPU)
}

extern "C" int pbsgpu_didx_parse(pbsgpu_ctx *ctx, const uint8_t *didx, uint64_t size, uint64_t *ends, uint8_t *digests,
                                 uint64_t cap, uint64_t *n_entries, int verify) {
    if (!didx || !n_entries) return PBSGPU_EINVAL;
    if (size < 4096 || (size - 4096) % 40 || memcmp(didx, DIDX_MAGIC, 8) != 0)
        return fail(ctx, PBSGPU_EINVAL, "not a dynamic index image");
    uint64_t n = (size - 4096) / 40;
    *n_entries = n;
    if (ends || digests) {
        if (cap < n) return fail(ctx, PBSGPU_ERANGE, "output capacity %llu < %llu entries", (unsigned long long)cap, (unsigned long long)n);
        uint64_t prev = 0;
        for (uint64_t i = 0; i < n; i++) {
            const uint8_t *e = didx + 4096 + i * 40;
            uint64_t end = 0;
            for (int k = 0; k < 8; k++) end |= (uint64_t)e[k] << (8 * k);
            if (end < prev) return fail(ctx, PBSGPU_EINVAL, "index offsets not monotonic at entry %llu", (unsigned long long)i);
            prev = end;
            if (ends) ends[i] = end;
            if (digests) memcpy(digests + i * 32, e + 8, 32);
        }
    }
    if (verify) {
        if (!ctx) return PBSGPU_EINVAL;
        uint8_t csum[32];
        uint64_t off0 = 0, len0 = n * 40;
        int rc = pbsgpu_sha256_batch(ctx, didx + 4096, &off0, &len0, 1, csum);
        if (rc) return rc;
        if (memcmp(csum, didx + 32, 32) != 0) return fail(ctx, PBSGPU_EINVAL, "index checksum mismatch");
    }
    return PBSGPU_OK;
}

// ---------------------------------------------------------------------------
// f3: DataBlob checksums
// ---------------------------------------------------------------------------
static const uint8_t BLOB_MAGIC_UNCOMPRESSED[8] = {66, 171, 56, 7, 190, 131, 112, 161};

extern "C" void pbsgpu_blob_header(uint32_t crc, uint8_t out[12]) {
    memcpy(out, BLOB_MAGIC_UNCOMPRESSED, 8);
    for (int i = 0; i < 4; i++) out[8 + i] = (uint8_t)(crc >> (8 * i));
}

extern "C" int pbsgpu_crc32_batch(pbsgpu_ctx *ctx, const void *base, const uint64_t *off, const uint64_t *len,
                                  uint32_t n, uint32_t *crc_out) {
    if (!ctx || (n && (!off || !len || !crc_out))) return PBSGPU_EINVAL;
    Guard g(ctx);
    if (n == 0) return PBSGPU_OK;
    cudaStream_t st = ctx->streams[0];
    if (!ctx->d_crc_tables) {
        std::vector<uint8_t> h(crc_tables_bytes());
        crc_fill_tables_host(h.data());
        CK(cudaMalloc(&ctx->d_crc_tables, h.size()));
        // a pageable cudaMemcpy may return before its DMA lands, and the kernels run on non-blocking streams: wait here
        CK(cudaMemcpyAsync(ctx->d_crc_tables, h.data(), h.size(), cudaMemcpyHostToDevice, st));
        CK(cudaStreamSynchronize(st));
    }
    const int crc_variant = ctx->crc_variant;   // 0 = TMA-tiled kernel (default), 1 = simple lane-strided kernel (PBSGPU_CRC_VARIANT at open)
    uint64_t hi = 0;
    for (uint32_t i = 0; i < n; i++) hi = std::max(hi, off[i] + len[i]);
    const bool on_dev = !hi || pbsgpu_is_device_ptr(base);
    Scoped staged(ctx->dev, on_dev ? 0 : hi + 16);
    if (!staged) return fail(ctx, PBSGPU_ENOMEM, "staging of %llu bytes failed", (unsigned long long)hi);
    const uint8_t *dbase = on_dev ? (const uint8_t *)base : staged.as<uint8_t>();
    // work units: 128 KiB warp blocks (simple) or <= 576 KiB regions of the 16 B aligned body (tiled)
    const uint64_t UNIT = crc_variant ? crc_wb_bytes() : crc_region_bytes();
    std::vector<uint64_t> wb_first(n + 1);
    uint64_t total = 0;
    for (uint32_t i = 0; i < n; i++) {
        wb_first[i] = total;
        if (crc_variant) total += (len[i] + UNIT - 1) / UNIT;
        else if (len[i]) {
            uint64_t head = (16 - ((uintptr_t)(dbase + off[i]) & 15)) & 15;
            uint64_t body = len[i] > head ? len[i] - head : 0;
            total += std::max<uint64_t>(1, (body + UNIT - 1) / UNIT);
        }
    }
    wb_first[n] = total;
    Scoped d_off(ctx->dev, n * 8), d_len(ctx->dev, n * 8), d_first(ctx->dev, (n + 1) * 8), d_part(ctx->dev, (total + 1) * 4), d_out(ctx->dev, (uint64_t)n * 4);
    if (!d_off || !d_len || !d_first || !d_part || !d_out) return fail(ctx, PBSGPU_ENOMEM, "device allocation failed");
    cudaError_t e = on_dev ? cudaSuccess : cudaMemcpyAsync(staged.p, base, hi, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_off.p, off, n * 8, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_len.p, len, n * 8, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_first.p, wb_first.data(), (n + 1) * 8, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess)
        e = crc_variant ? launch_crc32(dbase, d_off.as<uint64_t>(), d_len.as<uint64_t>(), d_first.as<uint64_t>(), n, total, ctx->d_crc_tables,
                                       d_part.as<uint32_t>(), d_out.as<uint32_t>(), ctx->sm_count, st)
                        : launch_crc32_tiled(dbase, d_off.as<uint64_t>(), d_len.as<uint64_t>(), d_first.as<uint64_t>(), n, total,
                                             ctx->d_crc_tables, d_part.as<uint32_t>(), d_out.as<uint32_t>(), ctx->sm_count, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(crc_out, d_out.p, (uint64_t)n * 4, cudaMemcpyDeviceToHost, st);
    cudaError_t es = cudaStreamSynchronize(st);   // always: scoped blocks must be idle before they return to the pool
    if (e == cudaSuccess) e = es;
    if (e != cudaSuccess) { (void)cudaGetLastError(); return fail(ctx, PBSGPU_ECUDA, "crc32 batch: %s", cudaGetErrorString(e)); }
    return PBSGPU_OK;
}

uint64_t pbsgpu_blob_size_impl(uint64_t payload) { return payload + 12; }
extern "C" uint64_t pbsgpu_blob_size(uint64_t payload_len) { return pbsgpu_blob_size_impl(payload_len); }

// f3: complete uncompressed DataBlobs for the NEW chunks of a batch in one call (upstream pbs-datastore data_blob.rs:
// magic[8] | crc32 LE over the payload | payload; uploaded by POST /dynamic_chunk, reference
// internal/server/backup/log_cleanup.go:19-31).  The CRCs come from K6 on the device; payload bytes are copied once
// (device -> host for resident data, host -> host otherwise) straight into their place behind the header.
extern "C" int pbsgpu_blob_encode_batch(pbsgpu_ctx *ctx, const void *base, const uint64_t *off, const uint64_t *len, uint32_t n,
                                        uint8_t *out, const uint64_t *out_off, uint32_t *crc_out) {
    if (!ctx || (n && (!off || !len || !out || !out_off || !base))) return PBSGPU_EINVAL;
    Guard g(ctx);
    if (n == 0) return PBSGPU_OK;
    std::vector<uint32_t> crc(n);
    int rc = pbsgpu_crc32_batch(ctx, base, off, len, n, crc.data());
    if (rc) return rc;
    const bool on_dev = pbsgpu_is_device_ptr(base);
    cudaStream_t st = ctx->copy_stream;
    for (uint32_t i = 0; i < n; i++) {
        uint8_t *b = out + out_off[i];
        pbsgpu_blob_header(crc[i], b);
        if (!len[i]) continue;
        if (on_dev) {
            cudaError_t e = cudaMemcpyAsync(b + 12, (const uint8_t *)base + off[i], len[i], cudaMemcpyDeviceToHost, st);
            if (e != cudaSuccess) { (void)cudaGetLastError(); cudaStreamSynchronize(st); return fail(ctx, PBSGPU_ECUDA, "blob payload copy: %s", cudaGetErrorString(e)); }
        } else memcpy(b + 12, (const uint8_t *)base + off[i], len[i]);
    }
    if (on_dev) CK(cudaStreamSynchronize(st));
    if (crc_out) memcpy(crc_out, crc.data(), (size_t)n * 4);
    return PBSGPU_OK;
}

// f3, compressed form: DataBlobs whose payload is a zstd frame when that is smaller than the raw bytes (upstream
// `DataBlob::encode` keeps the compressed form only then).  The frame is built on the device from RLE_Blocks (128 KiB
// blocks of one repeated byte) and Raw_Blocks (zframe.cu), and with `lz` also from Compressed_Blocks (K9, zlz.cu) where
// those come out smaller than the block; the CRC (K6) covers the frame.
static const uint8_t BLOB_MAGIC_COMPRESSED[8] = {49, 185, 88, 66, 111, 182, 163, 127};

static int blob_encode_zstd(pbsgpu_ctx *ctx, const void *base, const uint64_t *off, const uint64_t *len, uint32_t n,
                            uint8_t *out, const uint64_t *out_off, uint64_t *out_len, uint32_t *crc_out, bool lz) {
    if (!ctx || (n && (!off || !len || !out || !out_off || !out_len || !base))) return PBSGPU_EINVAL;
    Guard g(ctx);
    if (n == 0) return PBSGPU_OK;
    cudaStream_t st = ctx->streams[0];
    uint64_t hi = 0;
    for (uint32_t i = 0; i < n; i++) {
        if (len[i] >= (1ull << 40)) return fail(ctx, PBSGPU_EINVAL, "blob %u longer than 2^40 bytes", i);
        hi = std::max(hi, off[i] + len[i]);
    }
    const bool on_dev = !hi || pbsgpu_is_device_ptr(base);
    Scoped staged(ctx->dev, on_dev ? 0 : hi + 16);
    if (!staged) return fail(ctx, PBSGPU_ENOMEM, "staging of %llu bytes failed", (unsigned long long)hi);
    const uint8_t *dbase = on_dev ? (const uint8_t *)base : staged.as<uint8_t>();
    if (!on_dev) CK(cudaMemcpyAsync(staged.p, base, hi, cudaMemcpyHostToDevice, st));
    // K8a: which 128 KiB blocks are one repeated byte
    std::vector<uint64_t> blk_first(n + 1);
    uint64_t n_blocks = 0;
    for (uint32_t i = 0; i < n; i++) { blk_first[i] = n_blocks; n_blocks += (len[i] + ZFRAME_BLOCK - 1) / ZFRAME_BLOCK; }
    blk_first[n] = n_blocks;
    if (n_blocks >= (1ull << 31)) return fail(ctx, PBSGPU_EINVAL, "too many 128 KiB blocks in one call (%llu)", (unsigned long long)n_blocks);
    std::vector<uint32_t> flags(n_blocks);
    {
        Scoped d_off(ctx->dev, n * 8), d_len(ctx->dev, n * 8), d_first(ctx->dev, (n + 1) * 8), d_flags(ctx->dev, (n_blocks + 1) * 4);
        if (!d_off || !d_len || !d_first || !d_flags) return fail(ctx, PBSGPU_ENOMEM, "device allocation failed");
        cudaError_t e = cudaMemcpyAsync(d_off.p, off, n * 8, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_len.p, len, n * 8, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_first.p, blk_first.data(), (n + 1) * 8, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = launch_zblock_scan(dbase, d_off.as<uint64_t>(), d_len.as<uint64_t>(), d_first.as<uint64_t>(), n, n_blocks, d_flags.as<uint32_t>(), st);
        if (e == cudaSuccess && n_blocks) e = cudaMemcpyAsync(flags.data(), d_flags.p, n_blocks * 4, cudaMemcpyDeviceToHost, st);
        cudaError_t es = cudaStreamSynchronize(st);
        if (e == cudaSuccess) e = es;
        if (e != cudaSuccess) { (void)cudaGetLastError(); return fail(ctx, PBSGPU_ECUDA, "zstd block scan: %s", cudaGetErrorString(e)); }
    }
    // K9: every block that is not one repeated byte -> a Compressed_Block in its slot, or raw (lz_info 0)
    std::vector<uint32_t> lz_info(lz ? n_blocks : 0, 0), lz_slot(lz ? n_blocks : 0, 0);
    std::vector<uint64_t> l_src;
    std::vector<uint32_t> l_size;
    for (uint32_t i = 0; lz && i < n; i++)
        for (uint64_t b = 0; b < blk_first[i + 1] - blk_first[i]; b++)
            if (!(flags[blk_first[i] + b] & 0x100u)) {
                lz_slot[blk_first[i] + b] = (uint32_t)l_src.size();
                l_src.push_back(off[i] + b * ZFRAME_BLOCK);
                l_size.push_back((uint32_t)std::min<uint64_t>(ZFRAME_BLOCK, len[i] - b * ZFRAME_BLOCK));
            }
    const uint32_t nl = (uint32_t)l_src.size();
    Scoped lz_stage(ctx->dev, nl ? (uint64_t)nl * ZLZ_SLOT : 0);
    if (nl) {
        if (!lz_stage) return fail(ctx, PBSGPU_ENOMEM, "match stage output of %llu bytes failed", (unsigned long long)nl * ZLZ_SLOT);
        // 16 walking warps per SM (K9b); the pass's scratch is ~528 KiB per block, ~1 GiB at 124 bulk SMs
        const uint32_t pass = std::min<uint32_t>(nl, 16 * (uint32_t)ctx->sm_count);
        Scoped d_src(ctx->dev, nl * 8ull), d_size(ctx->dev, nl * 4ull), d_info(ctx->dev, nl * 4ull),
            scratch(ctx->dev, pass * zlz_scratch_bytes_per_block());
        if (!d_src || !d_size || !d_info || !scratch) return fail(ctx, PBSGPU_ENOMEM, "device allocation failed");
        std::vector<uint32_t> info(nl);
        cudaError_t e = cudaMemcpyAsync(d_src.p, l_src.data(), nl * 8ull, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_size.p, l_size.data(), nl * 4ull, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = launch_zlz(dbase, d_src.as<uint64_t>(), d_size.as<uint32_t>(), nl, lz_stage.as<uint8_t>(), d_info.as<uint32_t>(), scratch.p, pass, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(info.data(), d_info.p, nl * 4ull, cudaMemcpyDeviceToHost, st);
        cudaError_t es = cudaStreamSynchronize(st);
        if (e == cudaSuccess) e = es;
        if (e != cudaSuccess) { (void)cudaGetLastError(); return fail(ctx, PBSGPU_ECUDA, "zstd match stage: %s", cudaGetErrorString(e)); }
        for (uint64_t g = 0; g < n_blocks; g++)
            if (!(flags[g] & 0x100u)) lz_info[g] = info[lz_slot[g]];
    }
    // per block: 1 byte (RLE), the Compressed_Block (K9) or the raw bytes
    auto content_bytes = [&](uint64_t g, uint64_t size) -> uint64_t {
        if (flags[g] & 0x100u) return 1;
        return lz && lz_info[g] ? (lz_info[g] & 0xFFFFFFu) : size;
    };
    // frame sizes; the chunks that come out smaller get a place in the stage and one emit entry per block
    std::vector<uint8_t> comp(n, 0);
    std::vector<uint64_t> frame_len(n, 0), frame_off, content, e_src, e_dst;
    std::vector<uint32_t> e_hdr, comp_idx;
    uint64_t cursor = 0;
    for (uint32_t i = 0; i < n; i++) {
        const uint64_t nb = blk_first[i + 1] - blk_first[i];
        uint64_t fl = ZFRAME_HEADER;
        for (uint64_t b = 0; b < nb; b++) {
            const uint64_t size = std::min<uint64_t>(ZFRAME_BLOCK, len[i] - b * ZFRAME_BLOCK);
            fl += 3 + content_bytes(blk_first[i] + b, size);
        }
        frame_len[i] = fl;
        if (len[i] == 0 || fl >= len[i]) continue;
        comp[i] = 1;
        comp_idx.push_back(i);
        frame_off.push_back(cursor);
        content.push_back(len[i]);
        uint64_t pos = cursor + ZFRAME_HEADER;
        for (uint64_t b = 0; b < nb; b++) {
            const uint64_t size = std::min<uint64_t>(ZFRAME_BLOCK, len[i] - b * ZFRAME_BLOCK);
            const uint64_t g = blk_first[i] + b;
            const uint32_t f = flags[g];
            const bool rle = (f & 0x100u) != 0, cmp = !rle && lz && lz_info[g];
            const uint64_t bytes = content_bytes(g, size);
            // Block_Size is the repeat count for RLE, the content size otherwise
            e_src.push_back(cmp ? (uint64_t)lz_slot[g] * ZLZ_SLOT + (lz_info[g] >> 24) : off[i] + b * ZFRAME_BLOCK);
            e_dst.push_back(pos);
            e_hdr.push_back((uint32_t)(b + 1 == nb) | ((rle ? 1u : cmp ? 2u : 0u) << 1) | ((uint32_t)(rle ? size : bytes) << 3) |
                            ((f & 0xFFu) << 24));
            pos += 3 + bytes;
        }
        cursor = (pos + 15) & ~15ull;
    }
    const uint32_t nc = (uint32_t)comp_idx.size();
    Scoped stage(ctx->dev, nc ? cursor + 16 : 0);
    if (!stage) return fail(ctx, PBSGPU_ENOMEM, "frame staging of %llu bytes failed", (unsigned long long)cursor);
    std::vector<uint32_t> crc(n, 0);
    if (nc) {
        const uint64_t ne = e_hdr.size();
        Scoped d_src(ctx->dev, ne * 8), d_dst(ctx->dev, ne * 8), d_hdr(ctx->dev, ne * 4), d_foff(ctx->dev, nc * 8), d_clen(ctx->dev, nc * 8);
        if (!d_src || !d_dst || !d_hdr || !d_foff || !d_clen) return fail(ctx, PBSGPU_ENOMEM, "device allocation failed");
        cudaError_t e = cudaMemcpyAsync(d_src.p, e_src.data(), ne * 8, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_dst.p, e_dst.data(), ne * 8, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_hdr.p, e_hdr.data(), ne * 4, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_foff.p, frame_off.data(), nc * 8, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_clen.p, content.data(), nc * 8, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = launch_zframe_hdr(stage.as<uint8_t>(), d_foff.as<uint64_t>(), d_clen.as<uint64_t>(), nc, st);
        if (e == cudaSuccess) e = launch_zframe_emit(dbase, nl ? lz_stage.as<uint8_t>() : nullptr, stage.as<uint8_t>(), d_src.as<uint64_t>(), d_dst.as<uint64_t>(), d_hdr.as<uint32_t>(), ne, st);
        cudaError_t es = cudaStreamSynchronize(st);
        if (e == cudaSuccess) e = es;
        if (e != cudaSuccess) { (void)cudaGetLastError(); return fail(ctx, PBSGPU_ECUDA, "zstd frame emit: %s", cudaGetErrorString(e)); }
        // CRC over the frames
        std::vector<uint64_t> flen(nc);
        std::vector<uint32_t> fcrc(nc);
        for (uint32_t k = 0; k < nc; k++) flen[k] = frame_len[comp_idx[k]];
        int rc = pbsgpu_crc32_batch(ctx, stage.p, frame_off.data(), flen.data(), nc, fcrc.data());
        if (rc) return rc;
        for (uint32_t k = 0; k < nc; k++) crc[comp_idx[k]] = fcrc[k];
    }
    if (nc < n) {   // CRC over the raw payloads of the rest
        std::vector<uint64_t> roff, rlen;
        std::vector<uint32_t> ridx;
        for (uint32_t i = 0; i < n; i++) if (!comp[i]) { ridx.push_back(i); roff.push_back(off[i]); rlen.push_back(len[i]); }
        std::vector<uint32_t> rcrc(ridx.size());
        int rc = pbsgpu_crc32_batch(ctx, hi ? (const void *)dbase : base, roff.data(), rlen.data(), (uint32_t)ridx.size(), rcrc.data());
        if (rc) return rc;
        for (size_t k = 0; k < ridx.size(); k++) crc[ridx[k]] = rcrc[k];
    }
    // assemble in the caller's memory
    cudaStream_t cs = ctx->copy_stream;
    uint32_t k = 0;
    cudaError_t e = cudaSuccess;
    for (uint32_t i = 0; i < n && e == cudaSuccess; i++) {
        uint8_t *b = out + out_off[i];
        memcpy(b, comp[i] ? BLOB_MAGIC_COMPRESSED : BLOB_MAGIC_UNCOMPRESSED, 8);
        for (int q = 0; q < 4; q++) b[8 + q] = (uint8_t)(crc[i] >> (8 * q));
        if (comp[i]) {
            e = cudaMemcpyAsync(b + 12, stage.as<uint8_t>() + frame_off[k++], frame_len[i], cudaMemcpyDeviceToHost, cs);
            out_len[i] = 12 + frame_len[i];
        } else {
            out_len[i] = 12 + len[i];
            if (!len[i]) continue;
            if (on_dev) e = cudaMemcpyAsync(b + 12, (const uint8_t *)base + off[i], len[i], cudaMemcpyDeviceToHost, cs);
            else memcpy(b + 12, (const uint8_t *)base + off[i], len[i]);
        }
    }
    cudaError_t es = cudaStreamSynchronize(cs);
    if (e == cudaSuccess) e = es;
    if (e != cudaSuccess) { (void)cudaGetLastError(); return fail(ctx, PBSGPU_ECUDA, "blob assembly copy: %s", cudaGetErrorString(e)); }
    if (crc_out) memcpy(crc_out, crc.data(), (size_t)n * 4);
    return PBSGPU_OK;
}

extern "C" int pbsgpu_blob_encode_batch_z(pbsgpu_ctx *ctx, const void *base, const uint64_t *off, const uint64_t *len, uint32_t n,
                                          uint8_t *out, const uint64_t *out_off, uint64_t *out_len, uint32_t *crc_out) {
    return blob_encode_zstd(ctx, base, off, len, n, out, out_off, out_len, crc_out, false);
}

extern "C" int pbsgpu_blob_encode_batch_lz(pbsgpu_ctx *ctx, const void *base, const uint64_t *off, const uint64_t *len, uint32_t n,
                                           uint8_t *out, const uint64_t *out_off, uint64_t *out_len, uint32_t *crc_out) {
    return blob_encode_zstd(ctx, base, off, len, n, out, out_off, out_len, crc_out, true);
}

// ---------------------------------------------------------------------------
// f2: XXH3-64 of n byte ranges (the commit walk's per-file content hash, commit.go:717-725, :957-976).
// Blocks are hashed in passes of at most PBSGPU_XXH3_CAP_BLOCKS (default 8 Mi = 8 GiB of input, 512 MiB
// of per-block sums); a pass takes the same block window of EVERY stream so the chains stay parallel.
// xxh3_enqueue only enqueues (all passes, no host wait) so the fused batch call can put it on a job's
// stream; xxh3_collect waits for the stream and brings the n hashes back.
// ---------------------------------------------------------------------------

void pbsgpu_xxh3_release(pbsgpu_ctx *ctx, XxhRun *r) {
    ctx->dev.put(r->d_off); ctx->dev.put(r->d_len); ctx->dev.put(r->d_first); ctx->dev.put(r->d_out);
    ctx->dev.put(r->d_state); ctx->dev.put(r->d_S);
    *r = XxhRun();
}

int pbsgpu_xxh3_enqueue(pbsgpu_ctx *ctx, const uint8_t *dbase, const uint64_t *off, const uint64_t *len, uint32_t n,
                        cudaStream_t st, XxhRun *r) {
    if (!ctx->d_xxh_tab) {
        std::vector<uint8_t> h(xxh3_tables_bytes());
        xxh3_fill_tables_host(h.data());
        CK(cudaMalloc(&ctx->d_xxh_tab, h.size()));
        // as for the CRC tables: the table must have landed before any stream's kernel reads it
        CK(cudaMemcpyAsync(ctx->d_xxh_tab, h.data(), h.size(), cudaMemcpyHostToDevice, st));
        CK(cudaStreamSynchronize(st));
    }
    const uint64_t cap_blocks = ctx->xxh3_cap_blocks;
    uint64_t total_all = 0, max_nb = 0, n_long = 0;
    std::vector<uint64_t> nb(n);
    for (uint32_t i = 0; i < n; i++) {
        nb[i] = len[i] > 240 ? (len[i] - 1) >> 10 : 0;
        total_all += nb[i]; max_nb = std::max(max_nb, nb[i]); n_long += nb[i] != 0;
    }
    const bool one = total_all <= cap_blocks;
    const uint64_t win = one ? std::max<uint64_t>(max_nb, 1) : std::max<uint64_t>(1, cap_blocks / n_long);
    const uint64_t s_blocks = one ? total_all : std::min(total_all, n_long * win);
    const uint64_t passes = (max_nb + win - 1) / win;
    r->n = n;
    r->d_off = (uint64_t *)ctx->dev.get(n * 8); r->d_len = (uint64_t *)ctx->dev.get(n * 8);
    r->d_first = (uint64_t *)ctx->dev.get(std::max<uint64_t>(passes, 1) * (n + 1) * 8);
    r->d_out = (uint64_t *)ctx->dev.get((uint64_t)n * 8); r->d_state = (uint64_t *)ctx->dev.get((uint64_t)n * 64);
    r->d_S = (uint64_t *)ctx->dev.get(std::max<uint64_t>(s_blocks, 1) * 64);
    if (!r->d_off || !r->d_len || !r->d_first || !r->d_out || !r->d_state || !r->d_S) {
        pbsgpu_xxh3_release(ctx, r);
        return fail(ctx, PBSGPU_ENOMEM, "xxh3: device allocation failed");
    }
    cudaError_t e = cudaMemcpyAsync(r->d_off, off, n * 8, cudaMemcpyHostToDevice, st);   // pageable sources are staged before return
    if (e == cudaSuccess) e = cudaMemcpyAsync(r->d_len, len, n * 8, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = launch_xxh3_small(dbase, r->d_off, r->d_len, n, ctx->d_xxh_tab, r->d_out, st);
    std::vector<uint64_t> first(n + 1);
    uint64_t pass = 0;
    for (uint64_t lo = 0; e == cudaSuccess && lo < max_nb; lo += win, pass++) {
        uint64_t total = 0;
        for (uint32_t i = 0; i < n; i++) {
            first[i] = total;
            if (nb[i] > lo) total += std::min(nb[i] - lo, win);
        }
        first[n] = total;
        uint64_t *df = r->d_first + pass * (n + 1);
        e = cudaMemcpyAsync(df, first.data(), (n + 1) * 8, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = launch_xxh3_pass(dbase, r->d_off, r->d_len, df, n, total, lo, win, ctx->d_xxh_tab, r->d_S, r->d_state, r->d_out, st);
    }
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        cudaStreamSynchronize(st);
        pbsgpu_xxh3_release(ctx, r);
        return fail(ctx, PBSGPU_ECUDA, "xxh3: %s", cudaGetErrorString(e));
    }
    return PBSGPU_OK;
}

int pbsgpu_xxh3_collect(pbsgpu_ctx *ctx, XxhRun *r, uint64_t *hash_out, cudaStream_t st) {
    if (!r->d_out) return PBSGPU_OK;
    cudaError_t e = cudaMemcpyAsync(hash_out, r->d_out, (uint64_t)r->n * 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    pbsgpu_xxh3_release(ctx, r);
    if (e != cudaSuccess) { (void)cudaGetLastError(); return fail(ctx, PBSGPU_ECUDA, "xxh3: %s", cudaGetErrorString(e)); }
    return PBSGPU_OK;
}

extern "C" int pbsgpu_xxh3_batch(pbsgpu_ctx *ctx, const void *base, const uint64_t *off, const uint64_t *len,
                                 uint32_t n, uint64_t *hash_out) {
    if (!ctx || (n && (!off || !len || !hash_out))) return PBSGPU_EINVAL;
    Guard g(ctx);
    if (n == 0) return PBSGPU_OK;
    cudaStream_t st = ctx->streams[0];
    uint64_t hi = 0;
    for (uint32_t i = 0; i < n; i++) hi = std::max(hi, off[i] + len[i]);
    const bool on_dev = !hi || pbsgpu_is_device_ptr(base);
    Scoped staged(ctx->dev, on_dev ? 0 : hi + 16);
    if (!staged) return fail(ctx, PBSGPU_ENOMEM, "staging of %llu bytes failed", (unsigned long long)hi);
    const uint8_t *dbase = on_dev ? (const uint8_t *)base : staged.as<uint8_t>();
    if (!on_dev) {
        cudaError_t e = cudaMemcpyAsync(staged.p, base, hi, cudaMemcpyHostToDevice, st);
        if (e != cudaSuccess) { (void)cudaGetLastError(); cudaStreamSynchronize(st); return fail(ctx, PBSGPU_ECUDA, "H2D copy: %s", cudaGetErrorString(e)); }
    }
    XxhRun run;
    int rc = pbsgpu_xxh3_enqueue(ctx, dbase, off, len, n, st, &run);
    if (rc == PBSGPU_OK) rc = pbsgpu_xxh3_collect(ctx, &run, hash_out, st);
    else cudaStreamSynchronize(st);
    return rc;
}
