/*
 * cryogpu.h -- C ABI of libcryogpu.so, the B200 (sm_100a) block codec for pg_cryogen.
 *
 * libcryogpu.so replaces the arithmetic behind the reference's block codec
 * (reference compression.c:61-159, declared in compression.h:13-24), i.e. the
 * calls the reference makes into liblz4 / libzstd:
 *
 *   LZ4_compressBound    compression.c:67      -> cryogpu_compress_bound
 *   LZ4_compress_fast    compression.c:70-72   -> cryogpu_compress_{device,host}  (method 0)
 *   LZ4_decompress_safe  compression.c:84      -> cryogpu_decompress_{device,host} (method 0)
 *   ZSTD_compressBound   compression.c:99      -> cryogpu_compress_bound
 *   ZSTD_compress        compression.c:102-104 -> cryogpu_compress_{device,host}  (method 1)
 *   ZSTD_decompress      compression.c:116     -> cryogpu_decompress_{device,host} (method 1)
 *
 * The stream formats are the reference's on-disk formats, unchanged: method 0 is
 * one raw LZ4 block, method 1 is one standard zstd frame (storage.h:64,
 * SURVEY.md A.3).  The drop-in compression.c that keeps the reference's
 * compression.h API on top of this library is pg_cryogen_b200/host/compression.c;
 * INTEGRATION.md shows the binding.
 *
 * Conventions: extern "C"; plain pointers and integers; no exceptions, no
 * palloc/elog, no longjmp across the boundary.  Every entry point returns a
 * call-level code (CRYOGPU_OK or CRYOGPU_E_*); per-block outcomes are written to
 * the caller's status[] array so that one bad block never fails a batch
 * (cache.c:178-179 maps a failed block to CRYO_ERR_DECOMPRESSION_FAILED).
 * There is no CPU fallback: without a usable CUDA device every call fails with
 * CRYOGPU_E_CUDA.
 */
#ifndef CRYOGPU_H
#define CRYOGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CRYOGPU_VERSION 100

/* compression.h:7-11 -- stored on disk as a 4-byte int (storage.h:64) */
#define CRYOGPU_LZ4  0
#define CRYOGPU_ZSTD 1

/* storage.h:18 */
#define CRYOGPU_BLCKSZ (1u << 20)

/* call-level return codes */
#define CRYOGPU_OK          0
#define CRYOGPU_E_CUDA     (-1)   /* CUDA runtime error; cryogpu_last_error() has the text */
#define CRYOGPU_E_ARG      (-2)   /* bad argument (NULL, misaligned device pointer, size) */
#define CRYOGPU_E_NOMEM    (-3)
#define CRYOGPU_E_METHOD   (-4)   /* unknown compression method (compression.c:137, :157) */

/* per-block status[] values */
#define CRYOGPU_ST_OK            0
#define CRYOGPU_ST_INPUT         1   /* truncated stream / input not consumed exactly */
#define CRYOGPU_ST_OUTPUT        2   /* output would exceed the block capacity */
#define CRYOGPU_ST_OFFSET        3   /* match offset 0 or before the start of the output */
#define CRYOGPU_ST_FORMAT        4   /* bad magic, reserved value, invalid entropy table */
#define CRYOGPU_ST_SIZE          5   /* zstd frame content size does not match */
#define CRYOGPU_ST_METHOD        6   /* unknown per-block method */
#define CRYOGPU_ST_UNSUPPORTED   7   /* valid but outside what this build handles */
/* page-chain calls only (cache.c:112-129 returns CRYO_ERR_EMPTY_BLOCK / CRYO_ERR_WRONG_STARTING_BLOCK there) */
#define CRYOGPU_ST_EMPTY_BLOCK   8   /* the first page is new (pd_upper == 0), or the chain is empty */
#define CRYOGPU_ST_WRONG_START   9   /* the first page of the chain is not the first page of its cryo block */
#define CRYOGPU_ST_CHAIN        10   /* the pages do not form the chain of one block, or it is shorter than
                                      * compressed_size needs (the reference fails in cryo_decompress then) */

typedef struct cryogpu_ctx cryogpu_ctx;

int         cryogpu_version(void);
const char *cryogpu_last_error(void);
const char *cryogpu_status_string(int status);

/* Number of usable CUDA devices (0 when there is none; never throws). */
int         cryogpu_device_count(void);

/*
 * Lazy, per-process, per-device context (stream, scratch, pinned staging).
 * Safe to call after fork() in a PostgreSQL backend (pg_cryogen.c:169-176):
 * nothing touches CUDA before the first cryogpu_init.
 */
int         cryogpu_init(int device, cryogpu_ctx **ctx);
void        cryogpu_shutdown(cryogpu_ctx *ctx);
int         cryogpu_device(const cryogpu_ctx *ctx);

/* LZ4_compressBound / ZSTD_compressBound for one block of block_size bytes. */
uint64_t    cryogpu_compress_bound(int method, uint64_t block_size);

/* Pinned host memory for the *_host calls (pageable pointers work too, slower). */
void       *cryogpu_host_alloc(size_t bytes);
void        cryogpu_host_free(void *p);

/*
 * Batched decompression, everything device-resident.
 *
 *   d_methods[i]   CRYOGPU_LZ4 / CRYOGPU_ZSTD, per block (storage.h:64: the method
 *                  is a per-block header field)
 *   d_src          base of the compressed bytes; block i is
 *                  d_src[d_src_off[i] .. d_src_off[i] + d_src_size[i]); the buffer
 *                  must be readable up to the next 16-byte boundary
 *   d_dst          output; block i is written to d_dst + i * dst_stride, capacity
 *                  block_size (CRYO_BLCKSZ in the reference: compression.c:84, :116);
 *                  d_dst and dst_stride must be multiples of 16
 *   d_out_size[i]  bytes produced (the reference only Asserts == CRYO_BLCKSZ,
 *                  compression.c:88, :120)
 *   d_status[i]    CRYOGPU_ST_*; a block whose status is not CRYOGPU_ST_OK leaves its
 *                  block_size bytes of d_dst unspecified (as ZSTD_decompress / LZ4_decompress_safe
 *                  do when they fail part-way: the zstd pipeline writes runs ahead of the decode)
 *   stream         a cudaStream_t (NULL = the context's own stream); the call only
 *                  enqueues work, it does not synchronise
 *
 * Ordering: the kernels' work areas belong to the context, so the device-resident calls of ONE
 * context execute one after the other on the device whatever streams they are given (each call's
 * stream first waits for an event recorded at the end of the previous call).  Use one context per
 * stream for calls that should overlap.  Work areas grow on demand (the first call of a given size
 * allocates, which waits for the device); a steady-state call only enqueues.
 */
int cryogpu_decompress_device(cryogpu_ctx *ctx, size_t n,
                              const int32_t *d_methods,
                              const uint8_t *d_src, const uint64_t *d_src_off,
                              const uint32_t *d_src_size,
                              uint8_t *d_dst, uint64_t dst_stride, uint32_t block_size,
                              uint32_t *d_out_size, int32_t *d_status, void *stream);

/*
 * Batched compression, everything device-resident.  Block i is read from
 * d_src + i * src_stride (block_size bytes) and written to d_dst + i * dst_stride
 * (capacity dst_cap >= cryogpu_compress_bound).  level_or_accel is
 * lz4_acceleration (compression.c:72) or zstd_compression_level (compression.c:104).
 * A block's stream depends only on its bytes, the method and level_or_accel: not on
 * the other blocks of the batch, its place in it, or the bytes after it in its slot.
 */
int cryogpu_compress_device(cryogpu_ctx *ctx, size_t n, int method, int level_or_accel,
                            const uint8_t *d_src, uint64_t src_stride, uint32_t block_size,
                            uint8_t *d_dst, uint64_t dst_stride, uint32_t dst_cap,
                            uint32_t *d_dst_size, int32_t *d_status, void *stream);

/*
 * Host-pointer variants: H2D copy, kernels, D2H copy, synchronous.  This is what
 * the drop-in compression.c calls with n = 1 (pg_cryogen.c:726, cache.c:178) and
 * what a batched cache fill / COPY flush calls with n > 1.
 */
int cryogpu_decompress_host(cryogpu_ctx *ctx, size_t n, const int32_t *methods,
                            const void *const *src, const uint32_t *src_size,
                            void *const *dst, uint32_t block_size,
                            uint32_t *out_size, int32_t *status);

int cryogpu_compress_host(cryogpu_ctx *ctx, size_t n, int method, int level_or_accel,
                          const void *const *src, uint32_t block_size,
                          void *const *dst, uint32_t dst_cap,
                          uint32_t *dst_size, int32_t *status);

/*
 * The host decompress call returns a sparse block as its non-zero 4 KiB pages and fills the rest of the
 * caller's block with zeros itself.  on != 0: the caller declares that its destination blocks are PRIVATE
 * ANONYMOUS memory (malloc, palloc, .bss -- the reference's per-backend cache, cache.c:49, is; shared_buffers
 * and file mappings are NOT), and the library then returns the whole OS pages of a zero run to the kernel
 * (madvise MADV_DONTNEED: they read as zeros again, on demand) instead of writing them.  Off by default;
 * CRYOGPU_ZERO_UNMAP=1 in the environment turns it on for every context.  Ignored for pinned destinations.
 */
int cryogpu_set_zero_by_unmap(cryogpu_ctx *ctx, int on);

/*
 * Bytes the last cryogpu_decompress_host call on this context moved over the bus.  The call
 * returns only the 4 KiB pages of a decoded block that hold a non-zero byte and zero-fills the
 * rest of the caller's block on the host (a cryo block of narrow rows is ~98 % zeros,
 * storage.c:18); CRYOGPU_SPARSE_D2H=0 restores the plain copy, CRYOGPU_HOST_THREADS sets the
 * number of host threads that place the pages (default: min(cores, 16)).
 */
void cryogpu_last_transfer_bytes(const cryogpu_ctx *ctx, uint64_t *h2d, uint64_t *d2h);

/*
 * zstd frames of the last cryogpu_decompress_device call on this context: how many the
 * phase-split pipeline was given, and how many of them it handed to the one-warp-per-frame
 * decoder (irregular or malformed frames, see zstd_decode_p.cuh).  Waits for the device.
 * Diagnostics for tests and benchmarks; the reference has no counterpart.
 */
int cryogpu_zstd_pipeline_stats(cryogpu_ctx *ctx, uint64_t *frames, uint64_t *fallback_frames);

/*
 * LZ4 blocks of the last cryogpu_decompress_device call on this context when the batch had more than
 * two blocks per SM: how many blocks the call had, and how many of them the one-warp-per-block decoder
 * handed to the CTA-per-block decoder (lz4_decode_c.cuh) because they had more sequences than a warp
 * should walk (lz4_decode_w.cuh); smaller batches go to that decoder whole and report 0 / 0.  Waits
 * for the device.  Diagnostics.
 */
int cryogpu_lz4_route_stats(cryogpu_ctx *ctx, uint64_t *blocks, uint64_t *cta_blocks);

/*
 * ------------------------------------------------------------------ page chains
 *
 * On disk a compressed cryo block is a chain of 8 KiB PostgreSQL pages (reference storage.h:49-67:
 * CryoPageHeader 32 bytes with first / next block numbers; the first page's CryoFirstPageHeader, 48 bytes,
 * adds created_xid, compression_method, compressed_size, npages).  These calls take and give the pages
 * themselves, so the reference's host-side copies on either side of the codec disappear:
 *
 *   cryogpu_decompress_pages_*  replaces the gather loop of cryo_read_decompress (cache.c:151-176) plus the
 *                               cryo_decompress call after it (cache.c:178): method and compressed size are
 *                               read from the first page's header on the device;
 *   cryogpu_compress_pages_*    replaces cryo_compress (pg_cryogen.c:726) plus the split loop of cryo_preserve
 *                               (pg_cryogen.c:761-805): the output is the page images, headers filled in
 *                               (first, next, pd_lower / pd_upper / pd_special, and on the first page npages,
 *                               compression_method, compressed_size, created_xid).  pd_lsn and pd_checksum are
 *                               the buffer manager's (GenericXLogFinish, PageSetChecksumInplace) and stay zero.
 *
 * A chain is described by the host, which has to walk `next` anyway to fetch the pages:
 *   page_slot[e]   (device call) index of entry e's page in d_pages
 *   page_blkno[e]  its block number in the relation
 *   chain_off[i]   block i's chain is the entries [chain_off[i], chain_off[i + 1]), first page first
 * The device checks every page's first / next against that description (CRYOGPU_ST_CHAIN otherwise).
 */
#define CRYOGPU_PAGE_SIZE 8192u

/* cryo_pages_needed, pg_cryogen.c:692-704 */
uint32_t cryogpu_pages_needed(uint64_t compressed_size);

/* d_methods[i] (out): compression_method as the header has it; d_comp_size[i] (out, may be NULL): compressed_size */
int cryogpu_decompress_pages_device(cryogpu_ctx *ctx, size_t n, const uint8_t *d_pages,
                                    const uint32_t *d_page_slot, const uint32_t *d_page_blkno,
                                    const uint32_t *d_chain_off, size_t total_entries,
                                    uint8_t *d_dst, uint64_t dst_stride, uint32_t block_size,
                                    uint32_t *d_out_size, int32_t *d_status, int32_t *d_methods,
                                    uint32_t *d_comp_size, void *stream);

/*
 * d_page_blkno: n x cap_pages block numbers reserved for the blocks' pages (block i uses the first
 * d_npages[i] of its row); cap_pages >= cryogpu_pages_needed(cryogpu_compress_bound(method, block_size)).
 * d_pages: n x cap_pages x 8 KiB; block i's page k is written at (i * cap_pages + k) * 8192.
 */
int cryogpu_compress_pages_device(cryogpu_ctx *ctx, size_t n, int method, int level_or_accel,
                                  const uint8_t *d_src, uint64_t src_stride, uint32_t block_size,
                                  const uint32_t *d_page_blkno, uint32_t cap_pages, uint32_t created_xid,
                                  uint8_t *d_pages, uint32_t *d_npages, uint32_t *d_comp_size,
                                  int32_t *d_status, void *stream);

/* host pointers: pages[e] = the 8 KiB page of chain entry e where it lies (buffer pool) */
int cryogpu_decompress_pages_host(cryogpu_ctx *ctx, size_t n, const void *const *pages,
                                  const uint32_t *page_blkno, const uint32_t *chain_off,
                                  void *const *dst, uint32_t block_size, uint32_t *out_size,
                                  int32_t *status, int32_t *methods, uint32_t *comp_size);

/* pages_out[i * cap_pages + k]: where block i's page k goes (only the first npages[i] are written) */
int cryogpu_compress_pages_host(cryogpu_ctx *ctx, size_t n, int method, int level_or_accel,
                                const void *const *src, uint32_t block_size,
                                const uint32_t *page_blkno, uint32_t cap_pages, uint32_t created_xid,
                                void *const *pages_out, uint32_t *npages, uint32_t *comp_size,
                                int32_t *status);

/*
 * The flush of a batch of blocks as cryo_preserve does it (pg_cryogen.c:726-805), for blocks whose first
 * page number was reserved when the block was started (cryo_reserve_blockno, pg_cryogen.c:588-601):
 * compress all blocks, then call alloc(arg) once for every further page a block needs -- block by block,
 * page by page, the order of the reference's ReadBuffer(P_NEW) calls -- then cut the page images on the
 * device and copy each to page_ptr(arg, blkno) (BufferGetPage of that block).
 */
typedef uint32_t (*cryogpu_alloc_page_fn)(void *arg);
typedef void *(*cryogpu_page_ptr_fn)(void *arg, uint32_t blkno);
int cryogpu_compress_pages_alloc_host(cryogpu_ctx *ctx, size_t n, int method, int level_or_accel,
                                      const void *const *src, uint32_t block_size,
                                      const uint32_t *first_blkno, cryogpu_alloc_page_fn alloc,
                                      cryogpu_page_ptr_fn page_ptr, void *arg, uint32_t created_xid,
                                      uint32_t *npages, uint32_t *comp_size, int32_t *status);

/*
 * ------------------------------------------------------------ cryo blocks from packed tuples
 *
 * The write-side mirror of the batched tuple fetch below: tuples in the layout it returns -- entry e is
 * (tup_off[e], tup_len[e]) into data, block i takes entries [block_first[i], block_first[i + 1]) in insertion
 * order -- and block i out as cryo_init_page + cryo_storage_insert (storage.c:15-50) build it, byte for byte:
 * header {lower, upper}, item j {off, len} at byte 8 + 8j, tuple j at block_size - sum over k <= j of
 * MAXALIGN(len_k), every other byte zero.  block_size must be a multiple of 8 (else CRYOGPU_E_ARG).
 *
 *   status[i]   CRYOGPU_ST_FORMAT: block_first[i + 1] < block_first[i], or an entry with tup_off == UINT64_MAX (the
 *               fetch's "not found"), len > block_size, or bytes outside [0, data_size).  CRYOGPU_ST_OUTPUT:
 *               storage_insert would not take every entry (more than 290 items, or a tuple that does not fit).
 *               A failed block is not written.
 *
 * Bytes: read sum len + 12 per entry; write n * block_size.
 */

/* Blocks from tuples, everything in HBM (d_data any alignment; d_dst, dst_stride multiples of 16).  Enqueues work on
 * `stream` only; calls on one context are ordered as the other device-resident calls are. */
int cryogpu_build_blocks_device(cryogpu_ctx *ctx, size_t n, const uint8_t *d_data, uint64_t data_size,
                                const uint64_t *d_tup_off, const uint32_t *d_tup_len, const uint64_t *d_block_first,
                                uint32_t block_size, uint8_t *d_dst, uint64_t dst_stride, int32_t *d_status,
                                void *stream);

/* The COPY flush from tuples: as cryogpu_compress_pages_alloc_host, but the blocks are built on the device, so only
 * the entries and the bytes of data they cover cross the bus (straight from pinned memory where the caller's is).
 * A block whose build failed has that status, asks alloc for no page and writes nothing.  block_first must not
 * decrease (else CRYOGPU_E_ARG).  cryogpu_last_transfer_bytes reports the bytes moved. */
int cryogpu_compress_tuples_pages_alloc_host(cryogpu_ctx *ctx, size_t n, int method, int level_or_accel,
                                             const void *data, uint64_t data_size, const uint64_t *tup_off,
                                             const uint32_t *tup_len, const uint64_t *block_first, uint32_t block_size,
                                             const uint32_t *first_blkno, cryogpu_alloc_page_fn alloc,
                                             cryogpu_page_ptr_fn page_ptr, void *arg, uint32_t created_xid,
                                             uint32_t *npages, uint32_t *comp_size, int32_t *status);

/*
 * ------------------------------------------------------------ tuple-level work
 *
 * The item walk of a sequential scan (cryo_getnextslot, pg_cryogen.c:293-307, over cryo_storage_fetch,
 * storage.c:55-68) on decoded blocks that are still in HBM: per block the number of tuples, the sum of
 * their lengths, and whether every CryoItemId lies inside the block.  d_status (may be NULL): blocks whose
 * decode status is not CRYOGPU_ST_OK are skipped (0 / 0 / 0).  Enqueues one kernel on `stream`.
 */
int cryogpu_tuple_stats_device(cryogpu_ctx *ctx, size_t n, const uint8_t *d_blocks, uint64_t stride,
                               uint32_t block_size, const int32_t *d_status, uint32_t *d_ntuples,
                               uint64_t *d_tuple_bytes, int32_t *d_valid, void *stream);

/*
 * Count pushdown: compressed blocks in host memory in; per block ntuples, tuple_bytes and status out.  The
 * decoded blocks stay on the device, so the call moves csize + 24 bytes per block over the bus instead of
 * csize + block_size.  A block that decodes but whose item ids point outside it gets CRYOGPU_ST_FORMAT.
 */
int cryogpu_decompress_count_host(cryogpu_ctx *ctx, size_t n, const int32_t *methods,
                                  const void *const *src, const uint32_t *src_size, uint32_t block_size,
                                  uint32_t *ntuples, uint64_t *tuple_bytes, int32_t *status);

/*
 * ------------------------------------------------------------ batched tuple fetch
 *
 * The random-read path (index fetch, bitmap heap scan, row lock, analyze: cryo_storage_fetch, storage.c:55-68):
 * the tuples a caller names by TID (block, 1-based item position), packed, instead of whole decoded blocks.
 *
 *   item walk   as cryogpu_tuple_stats_device: ntuples = the largest cur with cur * 8 < lower; item p is the
 *               CryoItemId {off, len} at byte 8 * p.  The table is valid iff lower >= 8, lower <= upper <=
 *               block_size and every item lies inside [upper, block_size).
 *   selection   sel_off == NULL: every item of every block in position order.  Else block i takes the positions
 *               sel_pos[sel_off[i] .. sel_off[i + 1]) in that order; repeats are copied again; position 0 means
 *               every item of the block (a lossy bitmap page).
 *   output      the entries of all blocks in block order, then selection order.  Entry e: tup_off[e] (byte offset
 *               into data, a multiple of 8: a HeapTupleHeader pointer into data is MAXALIGNed), tup_len[e] (the
 *               item's len); the pad bytes up to MAXALIGN(len) are zero.  A position outside 1..ntuples gives
 *               tup_off = UINT64_MAX, tup_len = 0 ("not found").  Block i's entries are
 *               [block_first[i], block_first[i + 1]) (n + 1 values).
 *   status[i]   the decoder's / chain check's status passes through (no entries); a decoded block whose item table
 *               is invalid: CRYOGPU_ST_FORMAT (no entries).  Entries and bytes are placed by prefix sum over the
 *               blocks; a block whose range would cross tup_cap or data_cap gets CRYOGPU_ST_OUTPUT and writes
 *               nothing (its range stays reserved in block_first).
 *   need[2]     {bytes, entries} the whole batch needs, whatever the capacities: size a retry with it.
 *
 * Bytes: read 8 + 8 * ntuples + the selected tuples per block; write sum MAXALIGN(len) + 12 per entry.
 */

/* Decoded blocks in HBM (block i at d_blocks + i * stride; d_blocks, stride 8-byte aligned; d_data 16-byte aligned).
 * d_block_status (may be NULL): the decode's status[].  Enqueues work on `stream` only, like
 * cryogpu_tuple_stats_device; calls on one context are ordered as the other device-resident calls are. */
int cryogpu_tuples_device(cryogpu_ctx *ctx, size_t n, const uint8_t *d_blocks, uint64_t stride, uint32_t block_size,
                          const int32_t *d_block_status, const uint64_t *d_sel_off, const uint32_t *d_sel_pos,
                          uint8_t *d_data, uint64_t data_cap, uint64_t *d_tup_off, uint32_t *d_tup_len, uint64_t tup_cap,
                          uint64_t *d_block_first, int32_t *d_status, uint64_t *d_need, void *stream);

/* Compressed streams in host memory in, tuples out: csize in, the tuples and per-block metadata back.  Synchronous;
 * large batches go in chunks (offsets are global); pinned data / tup_off / tup_len are written straight by the
 * copies.  cryogpu_last_transfer_bytes reports the bytes moved. */
int cryogpu_decompress_tuples_host(cryogpu_ctx *ctx, size_t n, const int32_t *methods, const void *const *src,
                                   const uint32_t *src_size, uint32_t block_size, const uint64_t *sel_off,
                                   const uint32_t *sel_pos, void *data, uint64_t data_cap, uint64_t *tup_off,
                                   uint32_t *tup_len, uint64_t tup_cap, uint64_t *block_first, int32_t *status,
                                   uint64_t *need);

/* Page chains in (as cryogpu_decompress_pages_host describes them), tuples out; methods[i] / comp_size[i] (may be
 * NULL): compression_method and compressed_size of the first page's header. */
int cryogpu_decompress_pages_tuples_host(cryogpu_ctx *ctx, size_t n, const void *const *pages, const uint32_t *page_blkno,
                                         const uint32_t *chain_off, uint32_t block_size, const uint64_t *sel_off,
                                         const uint32_t *sel_pos, void *data, uint64_t data_cap, uint64_t *tup_off,
                                         uint32_t *tup_len, uint64_t tup_cap, uint64_t *block_first, int32_t *status,
                                         int32_t *methods, uint32_t *comp_size, uint64_t *need);

/*
 * Multi-GPU host variants: the batch is split into contiguous block ranges, one
 * per context (one host thread + stream per GPU, no collective; SURVEY.md 8(e)).
 */
int cryogpu_decompress_host_multi(cryogpu_ctx *const *ctxs, int nctx, size_t n,
                                  const int32_t *methods, const void *const *src,
                                  const uint32_t *src_size, void *const *dst,
                                  uint32_t block_size, uint32_t *out_size, int32_t *status);

int cryogpu_compress_host_multi(cryogpu_ctx *const *ctxs, int nctx, size_t n, int method,
                                int level_or_accel, const void *const *src,
                                uint32_t block_size, void *const *dst, uint32_t dst_cap,
                                uint32_t *dst_size, int32_t *status);

#ifdef __cplusplus
}
#endif
#endif /* CRYOGPU_H */
