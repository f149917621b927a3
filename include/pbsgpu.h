/*
 * pbsgpu.h -- C ABI of libpbsgpu.so, the B200-native chunk + digest + probe engine.
 *
 * This is the drop-in boundary for the ONE hot path of pbs-plus that this repo
 * accelerates (SURVEY.md section 8): content-defined chunking (buzhash), per-chunk
 * SHA-256 and the known-digest probe.  The reference (pbs-plus @ 26d6969) is pure
 * Go with CGO disabled and has NO existing FFI for this path; the arithmetic sits
 * behind Go call sites into github.com/pbs-plus/pxar v0.19.2 (reference go.mod:28).
 * Every entry point below names the reference interface it replaces
 * (paths relative to the reference tree).  The cgo binding a maintainer would add
 * is in go/gpuchunk/ and INTEGRATION.md.
 *
 * Conventions: plain C, plain pointers and sizes, no C++/torch types.  Every
 * function returns 0 on success or a negative PBSGPU_E* code; pbsgpu_strerror(ctx)
 * returns the message of the last failure on that context.  No thread-local state:
 * a ctx may be used from any OS thread (goroutines migrate), one call at a time per
 * ctx; different ctxs are independent.  There is NO CPU fallback: if no CUDA device
 * is usable pbsgpu_open fails.
 */
#ifndef PBSGPU_H
#define PBSGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PBSGPU_VERSION 201 /* 0.2.0 */

/* error codes (negative errno values) */
#define PBSGPU_OK 0
#define PBSGPU_EINVAL (-22)  /* bad argument (avg not a power of two, NULL, ...)      */
#define PBSGPU_ENOMEM (-12)  /* host or device allocation failed                      */
#define PBSGPU_ERANGE (-34)  /* caller's output array too small; *n_out = needed      */
#define PBSGPU_ECUDA (-5)    /* CUDA runtime/driver error, see pbsgpu_strerror        */
#define PBSGPU_ENODEV (-19)  /* no usable CUDA device                                 */
#define PBSGPU_ESTATE (-77)  /* call not valid in this state (stream finished, ...)   */

typedef struct pbsgpu_ctx pbsgpu_ctx;
typedef struct pbsgpu_set pbsgpu_set;
typedef struct pbsgpu_job pbsgpu_job;
typedef struct pbsgpu_stream pbsgpu_stream;

/* Chunker parameters.  Replaces buzhash.Config as built by buzhash.NewConfig(4096)
 * at internal/pxarmount/commit.go:302-305 and handed to backupproxy.NewPBSStore at
 * commit.go:296-305.  Derivation = upstream PBS ChunkerImpl::new. */
typedef struct pbsgpu_cfg {
    uint32_t avg;       /* average chunk size, BYTES, power of two, 256 .. 2^29 */
    uint32_t min;       /* avg >> 2                                            */
    uint32_t max;       /* avg << 2                                            */
    uint32_t mask;      /* 2*avg - 1                                           */
    uint32_t break_min; /* mask - 2 : cut iff (h & mask) >= break_min           */
    uint32_t window;    /* 64                                                  */
    uint32_t table[256];
} pbsgpu_cfg;

/* One finished chunk.  Replaces the (end offset, digest) pair the reference's
 * dedup writer appends to the dynamic index for every chunk produced inside
 * transfer.ArchiveWriter.WriteEntryReader (commit.go:720, :858). */
typedef struct pbsgpu_chunk {
    uint32_t stream;    /* index of the input stream in this call                */
    uint32_t flags;     /* PBSGPU_CHUNK_KNOWN: digest already in the set (skip upload) */
    uint64_t end_off;   /* exclusive end offset of the chunk within its stream   */
    uint8_t digest[32]; /* SHA-256 of the raw chunk bytes (CryptModeNone, commit.go:314) */
} pbsgpu_chunk;
#define PBSGPU_CHUNK_KNOWN 1u

typedef struct pbsgpu_devinfo {
    int32_t device;
    int32_t sm_count;
    int32_t cc_major, cc_minor;
    uint64_t total_mem, free_mem;
    char name[64];
} pbsgpu_devinfo;

/* Device-time breakdown of the last finished batch/job, CUDA events on the
 * launching stream (only filled when profiling is on). */
typedef struct pbsgpu_timing {
    float scan_ms, sort_ms, resolve_ms, sha_ms, set_ms, total_ms;
    /* kernel intervals in ms since the context was opened (same CUDA clock for all jobs of
     * a ctx): lets a caller merge overlapping jobs into "time a kernel class was active" */
    float scan_t0, scan_t1, sha_t0, sha_t1;
    float sha_long_ms, sha_bulk_ms; /* hybrid SHA launch: latency kernel (long chunks) / throughput kernel */
    uint64_t bytes, chunks, candidates;
    uint32_t scan_launches, sha_launches, other_launches, reruns;
} pbsgpu_timing;

/* ---- lifecycle -------------------------------------------------------------- */
int pbsgpu_version(void);
int pbsgpu_open(int device, pbsgpu_ctx **out);
void pbsgpu_close(pbsgpu_ctx *ctx);
const char *pbsgpu_strerror(const pbsgpu_ctx *ctx);
int pbsgpu_device_info(pbsgpu_ctx *ctx, pbsgpu_devinfo *out);
int pbsgpu_set_profiling(pbsgpu_ctx *ctx, int on);
/* SM partition in effect (CUDA green contexts; PBSGPU_PARTITION_SMS=n at open): SMs reserved for the
 * long-chunk latency kernels / SMs for everything else; both 0 when the GPU is not partitioned. */
int pbsgpu_partition_info(pbsgpu_ctx *ctx, int *long_sms, int *bulk_sms);
/* SMs that run only the front halves (K1 scan, sort, K2 resolve; PBSGPU_SCAN_SMS=n at open); 0 = they share the bulk SMs. */
int pbsgpu_scan_partition_sms(pbsgpu_ctx *ctx);
/* 0 = tuned kernels (default), 1 = simple cross-check kernels (same results) */
int pbsgpu_set_kernel_variant(pbsgpu_ctx *ctx, int variant);

/* ---- a1: configuration (replaces buzhash.NewConfig, commit.go:302-305) ------- */
/* avg in BYTES; table NULL = built-in default table. */
int pbsgpu_config(uint32_t avg_bytes, const uint32_t *table /*[256] or NULL*/, pbsgpu_cfg *out);
/* The reference passes 4096 = KiB in the upstream client's convention (4 MiB). */
int pbsgpu_config_kib(uint32_t avg_kib, const uint32_t *table, pbsgpu_cfg *out);
const uint32_t *pbsgpu_default_table(void);

/* ---- a2+a3(+a4): batch of independent streams ---------------------------------
 * Replaces, for n files at once, the per-file loop
 *     writer.WriteEntryReader(entry, reader, size)       (commit.go:720, :858)
 * i.e. [pull bytes -> buzhash scan -> cut -> SHA-256(chunk) -> known?].
 * Stream i is bytes [base+off[i], base+off[i]+len[i]).  `base` may be a DEVICE
 * pointer (data already resident in HBM) or a HOST pointer (pageable or pinned;
 * the library stages it through pinned buffers and overlaps H2D with compute).
 * Chunks are returned ordered by (stream, end_off).  If `set` is non-NULL every
 * chunk digest is probed against it in that order (a digest also counts as known
 * if an earlier chunk of the same call had it) and then inserted.
 * Returns PBSGPU_ERANGE with *n_out = required count if cap is too small. */
int pbsgpu_chunk_digest_batch(pbsgpu_ctx *ctx, const pbsgpu_cfg *cfg, const void *base, const uint64_t *off,
                              const uint64_t *len, uint32_t n, pbsgpu_set *set, pbsgpu_chunk *out, uint64_t cap,
                              uint64_t *n_out);

/* Asynchronous form for DEVICE-resident input: submit returns as soon as the
 * kernels are enqueued; several jobs may be in flight (they overlap on the GPU,
 * which hides the sequential tail of the longest chunk's SHA-256).  wait blocks,
 * copies the chunks out and frees the job -- except on PBSGPU_ERANGE, where the job stays
 * valid: call wait again with the capacity reported in *n_out, or pbsgpu_batch_free.
 * (A digest set can be attached with pbsgpu_batch_submit_ex.) */
int pbsgpu_batch_submit(pbsgpu_ctx *ctx, const pbsgpu_cfg *cfg, const void *base_dev, const uint64_t *off,
                        const uint64_t *len, uint32_t n, pbsgpu_job **job);
int pbsgpu_batch_wait(pbsgpu_job *job, pbsgpu_chunk *out, uint64_t cap, uint64_t *n_out, pbsgpu_timing *timing);

/* Extended batch form: everything the calls above take, plus
 *  - SUGGESTED BOUNDARIES (SURVEY.md section 8 a2 caveat): offsets at which the caller would like a cut -- the
 *    starts of the files' PAYLOAD headers when the stream is a pxar v2 payload stream (the bytes the production
 *    chunker sees: 16-byte PAYLOAD header + content per file, concatenated; internal/pxarmount/pxarfs.go:408-411,
 *    writer calls commit.go:720,:858).  Rule (upstream PBS `PayloadChunker`, restated for byte-wise arrival): with
 *    the running chunk starting at `base`, a boundary B with B - base < min is dropped; with min <= B - base <= max
 *    the chunk ends at B unless the hash test cuts earlier; with B - base > max the plain chunker decides and B
 *    stays pending.  Pairs (forced_stream[i], forced_off[i]) sorted by (stream, offset), offsets in (0, len);
 *    needs cfg->min >= 65 (avg >= 512).  Whether pbs-plus/pxar v0.19.2 applies such boundaries is UNVERIFIED;
 *    n_forced = 0 gives the plain chunker.
 *  - a digest set for the asynchronous form too: the probe + insert runs as kernels on the job's stream
 *    (jobs that share a set are ordered in submission order), flags come back with the records.
 *  - stream_xxh3[n] (may be NULL): as pbsgpu_chunk_digest_batch_xxh3 (synchronous form only).
 * `size` must be sizeof(pbsgpu_batch_opts) (forward compatibility). */
typedef struct pbsgpu_batch_opts {
    uint32_t size, flags;
    pbsgpu_set *set;
    const uint32_t *forced_stream;
    const uint64_t *forced_off;
    uint64_t n_forced;
    uint64_t *stream_xxh3;
} pbsgpu_batch_opts;
int pbsgpu_chunk_digest_batch_ex(pbsgpu_ctx *ctx, const pbsgpu_cfg *cfg, const void *base, const uint64_t *off,
                                 const uint64_t *len, uint32_t n, const pbsgpu_batch_opts *opts, pbsgpu_chunk *out,
                                 uint64_t cap, uint64_t *n_out);
int pbsgpu_batch_submit_ex(pbsgpu_ctx *ctx, const pbsgpu_cfg *cfg, const void *base_dev, const uint64_t *off,
                           const uint64_t *len, uint32_t n, const pbsgpu_batch_opts *opts, pbsgpu_job **job);
/* pbsgpu_batch_opts.flags for pbsgpu_batch_submit_ex.
 * PBSGPU_BATCH_EARLY_INPUT: give the input buffer back BEFORE the job is done.  A batch's results wait for the serial
 * SHA-256 chain of its longest chunk (~0.3 s for a 16 MiB chunk) -- ten times longer than the rest of a 16 GiB batch --
 * and until then the device reads the input.  With this flag the long chunks (about 11 % of the bytes on backup data)
 * are first copied into an arena inside the library (PBSGPU_ARENA_MB, default 32 GiB, halved until it fits; allocated on first use) and hashed
 * from there: pbsgpu_batch_wait_input returns as soon as the bulk pass and that copy are done, the caller may overwrite
 * or free the buffer and submit the next batch into it, and collects the records later with pbsgpu_batch_wait (in
 * submission order when a set is shared).  pbsgpu_batch_input_done is the non-blocking form (1 free, 0 not yet).
 * Results are identical with and without the flag; without it (or when no arena can be allocated) both calls simply
 * report the end of the job. */
#define PBSGPU_BATCH_EARLY_INPUT 1u
int pbsgpu_batch_wait_input(pbsgpu_job *job);
int pbsgpu_batch_input_done(pbsgpu_job *job);
/* Frees a job without collecting it (after a failed wait, or to abandon it); waits for its kernels. */
void pbsgpu_batch_free(pbsgpu_job *job);

/* Boundary scan only (a2): chunk END offsets per stream, no digests.
 * ends: caller array of cap u64; stream_first[i]..stream_first[i+1] index it
 * (stream_first has n+1 entries). */
int pbsgpu_scan_batch(pbsgpu_ctx *ctx, const pbsgpu_cfg *cfg, const void *base, const uint64_t *off,
                      const uint64_t *len, uint32_t n, uint64_t *ends, uint64_t cap, uint64_t *stream_first,
                      uint64_t *n_out);

/* Digest only (a3): SHA-256 of n arbitrary byte ranges; digests = n*32 bytes (host). */
int pbsgpu_sha256_batch(pbsgpu_ctx *ctx, const void *base, const uint64_t *off, const uint64_t *len, uint32_t n,
                        uint8_t *digests);

/* ---- streaming form -----------------------------------------------------------
 * Mirrors how the reference feeds ONE io.Reader of known size through the chunker
 * (scan() state carried across reads; commit.go:718-720).  Bytes are buffered on
 * the device; finished chunks become available from poll(); finish() emits the
 * final short chunk.  Results are identical to the batch call on the whole stream
 * no matter how the bytes are split across writes. */
int pbsgpu_stream_open(pbsgpu_ctx *ctx, const pbsgpu_cfg *cfg, pbsgpu_set *set, pbsgpu_stream **out);
int pbsgpu_stream_write(pbsgpu_stream *s, const void *host_data, uint64_t len);
int pbsgpu_stream_poll(pbsgpu_stream *s, pbsgpu_chunk *out, uint64_t cap, uint64_t *n_out);
int pbsgpu_stream_finish(pbsgpu_stream *s);
void pbsgpu_stream_close(pbsgpu_stream *s);
/* Zero-copy staging for the streaming form: reserve hands out up to pbsgpu_stream_slot_bytes() of PINNED memory owned
 * by the stream (a ring of 8 slots); the caller reads its io.Reader straight into it and commits the byte count, which
 * starts the DMA and returns at once.  reserve blocks only while every slot still waits for its DMA.  write() is
 * reserve + memcpy + commit for pageable memory and a direct DMA for pinned caller memory. */
int pbsgpu_stream_reserve(pbsgpu_stream *s, void **buf);
int pbsgpu_stream_commit(pbsgpu_stream *s, uint64_t len);
uint64_t pbsgpu_stream_slot_bytes(const pbsgpu_stream *s);
/* Suggested boundary at absolute stream offset `offset` (>= bytes written so far, strictly increasing): what the
 * payload-stream writer calls right before it writes a file's PAYLOAD header.  Rule as in pbsgpu_batch_opts. */
int pbsgpu_stream_suggest(pbsgpu_stream *s, uint64_t offset);
/* Bytes written so far (= the payload offset the next entry will get in the mpxar PAYLOAD_REF). */
uint64_t pbsgpu_stream_position(const pbsgpu_stream *s);

/* ---- a4: known-digest set -------------------------------------------------------
 * Replaces the known-chunk bookkeeping of the reference's dedup session:
 * seeded from the previous snapshot (backupproxy.PreviousBackupRef commit.go:286-294,
 * origPayloadIdx commit.go:324-329), "Only new chunks are uploaded"
 * (docs/pxar-mount.md:105).  Exact 32-byte comparison, device-resident table. */
int pbsgpu_set_create(pbsgpu_ctx *ctx, uint64_t capacity_hint, pbsgpu_set **out);
void pbsgpu_set_destroy(pbsgpu_set *set);
/* d32: n*32 bytes, HOST or DEVICE pointer.  hit (HOST, n bytes, may be NULL):
 * insert: 1 = already present before this call or earlier within it (then inserted);
 * probe : 1 = present in the set (plain membership, nothing inserted). */
int pbsgpu_set_insert(pbsgpu_set *set, const uint8_t *d32, uint64_t n, uint8_t *hit);
int pbsgpu_set_probe(pbsgpu_set *set, const uint8_t *d32, uint64_t n, uint8_t *hit);
int pbsgpu_set_count(pbsgpu_set *set, uint64_t *count);
/* Seed from a PBS dynamic index (.didx) image: 4096-byte header + 40-byte
 * {u64 end_le, digest[32]} entries (what origPayloadIdx holds, commit.go:324-329). */
int pbsgpu_set_seed_didx(pbsgpu_set *set, const uint8_t *didx, uint64_t size, uint64_t *n_entries);

/* ---- e: multi-GPU merge of the digest set (SURVEY.md section 8 e / 8 b) -----------------------------------------
 * One process (or thread) per GPU chunks its own shard of the files; the ONE exchange step is an NCCL all-gather of
 * every rank's new digests over NVLink, after which every rank inserts ALL gathered digests into its replica of the
 * set in global (rank, index) order.  hit[i] (HOST, n bytes, may be NULL) = this rank's digest i was known before the
 * call or occurs earlier in that global order -- so with files sharded in rank order the flags equal a single-GPU run.
 * Collective: every rank of the communicator must call it, in the same order.  d32 HOST or DEVICE, n may be 0.
 * `nccl_comm` is an ncclComm_t the caller owns (libnccl.so.2 is resolved with dlopen at first use; PBSGPU_NCCL_LIB
 * overrides the path); the three helpers below create one for callers without an NCCL binding of their own
 * (the 128-byte unique id travels by whatever channel the ranks share). */
int pbsgpu_set_allgather(pbsgpu_set *set, void *nccl_comm, const uint8_t *d32, uint64_t n, uint8_t *hit);
int pbsgpu_nccl_unique_id(uint8_t id[128]);
int pbsgpu_nccl_comm_create(pbsgpu_ctx *ctx, const uint8_t id[128], int nranks, int rank, void **comm);
void pbsgpu_nccl_comm_destroy(void *comm);

/* ---- f1 ("next" row of SURVEY.md section 8): PBS dynamic index (.didx) images ----------------
 * The (end offset, digest) list of a finished archive lands in `<name>.mpxar.didx` /
 * `<name>.ppxar.didx` (names at commit.go:321-322; parsed via datastore.ParseDynamicIndex,
 * internal/pxar/format.go:163).  Layout restated from upstream PBS (UNVERIFIED against the Go
 * module): 4096-byte header { magic[8] = 1c 91 4e a5 19 ba b3 cd, uuid[16], ctime i64 LE,
 * index_csum[32] = SHA-256 over the entry table, zero padding } followed by n entries
 * { u64 end_le, digest[32] }.  Offsets are cumulative over the records in the order given (the
 * archive stream is the concatenation of the streams).  The checksum is computed on the GPU. */
uint64_t pbsgpu_didx_size(uint64_t n_entries);
int pbsgpu_didx_build(pbsgpu_ctx *ctx, const pbsgpu_chunk *chunks, uint64_t n, const uint8_t uuid[16], int64_t ctime,
                      uint8_t *out, uint64_t cap);
/* ends / digests may be NULL to only count; verify != 0 recomputes index_csum (PBSGPU_EINVAL on mismatch). */
int pbsgpu_didx_parse(pbsgpu_ctx *ctx, const uint8_t *didx, uint64_t size, uint64_t *ends, uint8_t *digests,
                      uint64_t cap, uint64_t *n_entries, int verify);

/* ---- f3 ("next" row): DataBlob checksums for NEW chunks ---------------------------------------
 * A new chunk is uploaded as a PBS DataBlob { magic[8], crc32 LE of the payload, payload } (upstream
 * pbs-datastore data_blob.rs; POST /dynamic_chunk, reference internal/server/backup/log_cleanup.go:19-31).
 * pbsgpu_crc32_batch computes zlib-compatible CRC-32s of n byte ranges (HOST or DEVICE base) on the GPU;
 * pbsgpu_blob_header fills the 12-byte header of an unencrypted, uncompressed blob. */
int pbsgpu_crc32_batch(pbsgpu_ctx *ctx, const void *base, const uint64_t *off, const uint64_t *len, uint32_t n,
                       uint32_t *crc_out);
void pbsgpu_blob_header(uint32_t crc, uint8_t out[12]);
/* Complete uncompressed DataBlobs { magic[8], crc32 LE, payload } of n byte ranges (the NEW chunks of a batch) in one
 * call: blob i is written to out + out_off[i] (HOST memory, 12 + len[i] bytes; pbsgpu_blob_size gives that), the CRCs
 * come from K6, payload bytes are copied from `base` (HOST or DEVICE).  crc_out (may be NULL) also receives the CRCs. */
uint64_t pbsgpu_blob_size(uint64_t payload_len);
int pbsgpu_blob_encode_batch(pbsgpu_ctx *ctx, const void *base, const uint64_t *off, const uint64_t *len, uint32_t n,
                             uint8_t *out, const uint64_t *out_off, uint32_t *crc_out);
/* The same with the COMPRESSED form where it is smaller (upstream `DataBlob::encode` keeps a zstd payload only then):
 * blob i = { compressed-blob magic, crc32 LE of the frame, zstd frame } or the uncompressed blob as above; out_len[i]
 * receives its size (<= pbsgpu_blob_size(len[i]), which is what the caller reserves at out_off[i]).  The frame is a
 * standard zstd frame (RFC 8878) built on the device from RLE_Blocks -- 128 KiB blocks that are one repeated byte, i.e.
 * the zero runs of disk images and sparse files -- and Raw_Blocks; there is NO match / entropy stage, so data without
 * such runs stays uncompressed.  Any zstd decoder reads the result; it is not byte-identical to libzstd's output for the
 * same input (no two zstd encoders are). */
int pbsgpu_blob_encode_batch_z(pbsgpu_ctx *ctx, const void *base, const uint64_t *off, const uint64_t *len, uint32_t n,
                               uint8_t *out, const uint64_t *out_off, uint64_t *out_len, uint32_t *crc_out);
/* pbsgpu_blob_encode_batch_z plus zstd's match stage (K9): the same arguments, reservation and blob-level rule, and the
 * same frame and 128 KiB block grid, but a block that is not one repeated byte becomes a Compressed_Block wherever
 * that is smaller than the block (Raw_Block otherwise).  The Compressed_Block holds the sequences of a greedy LZ parse
 * confined to its own block (4-byte minimum match, 2^14-entry hash table) with Raw_Literals and the three predefined
 * FSE tables; it omits Huffman-coded literals, FSE-compressed or repeated tables, repeat offsets, lazy parsing and
 * matches across blocks, so it compresses less than libzstd level 1 and costs more GPU time than the _z call.  Text,
 * logs and repeated records shrink; any zstd decoder reads the result. */
int pbsgpu_blob_encode_batch_lz(pbsgpu_ctx *ctx, const void *base, const uint64_t *off, const uint64_t *len, uint32_t n,
                                uint8_t *out, const uint64_t *out_off, uint64_t *out_len, uint32_t *crc_out);

/* ---- f2 ("next" row): the commit walk's per-file content hash ----------------------------------
 * emitBackedFile tees every new file through `xxh3.New()` and keeps `h.Sum64()` (reference
 * internal/pxarmount/commit.go:717-725); verifyBackedFileHashes later re-reads every file to recompute
 * it (commit.go:957-976).  XXH3-64, seed 0, default secret (github.com/zeebo/xxh3, go.mod; the published
 * xxHash v0.8 algorithm -- tests pin it against libxxhash).
 * pbsgpu_xxh3_batch hashes n byte ranges (HOST or DEVICE base) on the GPU.
 * pbsgpu_chunk_digest_batch_xxh3 is pbsgpu_chunk_digest_batch plus stream_xxh3[n] (may be NULL): the
 * XXH3-64 of every stream computed from the SAME staged bytes the chunker and SHA-256 read, so the
 * batched commit walk needs no second pass over the file on the host. */
int pbsgpu_xxh3_batch(pbsgpu_ctx *ctx, const void *base, const uint64_t *off, const uint64_t *len, uint32_t n,
                      uint64_t *hash_out);
int pbsgpu_chunk_digest_batch_xxh3(pbsgpu_ctx *ctx, const pbsgpu_cfg *cfg, const void *base, const uint64_t *off,
                                   const uint64_t *len, uint32_t n, pbsgpu_set *set, pbsgpu_chunk *out, uint64_t cap,
                                   uint64_t *n_out, uint64_t *stream_xxh3);

/* ---- pinned staging owned by C, filled by the Go side ----------------------------- */
void *pbsgpu_host_alloc(pbsgpu_ctx *ctx, uint64_t bytes);
void pbsgpu_host_free(pbsgpu_ctx *ctx, void *p);

/* ---- measurement aid: synthetic corpus generated on the device ------------------
 * Same integer recipe as oracle/oracle.c:orc_corpus_fill (SURVEY.md section 8d).
 * Writes files [first_file, first_file+n_files), each file_len bytes, at
 * dst_dev + i*stride. */
typedef struct pbsgpu_corpus {
    uint64_t seed, file_len, block_len;
    uint32_t run_blocks, dup_permille, edit_mode, edit_thresh16;
    uint64_t edit_seed;
} pbsgpu_corpus;
int pbsgpu_corpus_fill(pbsgpu_ctx *ctx, const pbsgpu_corpus *c, uint64_t first_file, uint32_t n_files,
                       void *dst_dev, uint64_t stride);

#ifdef __cplusplus
}
#endif
#endif /* PBSGPU_H */
