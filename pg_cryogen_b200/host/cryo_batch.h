/*
 * cryo_batch.h -- the callers on either side of the codec, batched (SURVEY.md 8 f-2, f-3).
 *
 * The reference decompresses one cryo block per cache miss (cache.c:244-297 -> cryo_read_decompress ->
 * cryo_decompress, cache.c:178) and compresses one block per flush (flush_modify_state ->
 * cryo_preserve -> cryo_compress, pg_cryogen.c:726).  A GPU wants batches.  This module is the
 * host-side harness that makes them, with the reference's own vocabulary and error codes:
 *
 *   read side   a block cache with the interface of cache.h (cryo_read_data, cryo_cache_get_data,
 *               cryo_cache_get_xid, cryo_cache_get_pg_nblocks, CryoError), more slots than the
 *               reference's 16 (cache.c:17), and a fill that takes N block numbers: the page chains
 *               of all misses are walked on the host (it has to follow `next` to fetch the pages
 *               anyway) and go to the device in ONE cryogpu_decompress_pages_host call.  The
 *               sequential scan uses it for read-ahead: the iterator (scan_iterator.c:55-78) knows
 *               the next block numbers.
 *   write side  a modify state that keeps several full 1 MiB blocks (the reference flushes at the
 *               first full one, pg_cryogen.c:634-640) and hands them to ONE
 *               cryogpu_compress_tuples_pages_alloc_host call; the first page of every block is reserved when
 *               the block is started, as cryo_reserve_blockno does (pg_cryogen.c:588-601), because
 *               the item pointers of its tuples carry that number.  The blocks are kept as their tuples,
 *               packed, with storage_insert's two counters per block deciding where one ends: the device
 *               builds the block images, so only the tuple bytes cross the bus.
 *
 * PostgreSQL's buffer manager is reached through CryoRelOps, so the module builds and is tested
 * without a backend; INTEGRATION.md shows the ReadBuffer / BufferGetPage / P_NEW bindings.
 */
#ifndef CRYO_BATCH_H
#define CRYO_BATCH_H

#include <stddef.h>
#include <stdint.h>

#include "cryogpu.h"

#define CRYO_BATCH_BLCKSZ   (1u << 20)          /* CRYO_BLCKSZ, storage.h:18 */
#define CRYO_BATCH_PAGE     8192u               /* BLCKSZ */
#define CRYO_BATCH_MAXPAGES 132u                /* pages of one block at most (cryo_pages_needed of the bound) */

/* cache.h:13-20 */
typedef enum
{
    CRYO_ERR_SUCCESS = 0,
    CRYO_ERR_DECOMPRESSION_FAILED,
    CRYO_ERR_WRONG_STARTING_BLOCK,
    CRYO_ERR_EMPTY_BLOCK,
    CRYO_ERR_CACHE_IS_FULL
} CryoError;

typedef int CacheEntry;                         /* cache.h:23: position in the cache */
#define InvalidCacheEntry (-1)

/* the relation, as the buffer manager shows it */
typedef struct
{
    void       *rel;
    uint32_t  (*nblocks)(void *rel);                        /* RelationGetNumberOfBlocks */
    void     *(*read_page)(void *rel, uint32_t blkno);      /* ReadBuffer + BufferGetPage (8 KiB) */
    uint32_t  (*extend)(void *rel);                         /* ReadBuffer(rel, P_NEW): a new zeroed page, its number */
} CryoRelOps;

typedef struct CryoBatchCache CryoBatchCache;

CryoBatchCache *cryo_batch_cache_create(cryogpu_ctx *gpu, int nslots);
void        cryo_batch_cache_destroy(CryoBatchCache *c);
/* cache.c:244-297, for n blocks at once: the misses among blocknos[] are read, in one device call.
 * errs[i] is what cryo_read_data would have returned for blocknos[i]; entries[i] the slot (or InvalidCacheEntry).
 * A block number may repeat: a request for a block that an earlier request of the same call missed gets that
 * miss's outcome (its error, and its entry or InvalidCacheEntry) and is not counted as a hit. */
int         cryo_batch_read_data(CryoBatchCache *c, const CryoRelOps *ops, const uint32_t *blocknos, int n,
                                 CacheEntry *entries, CryoError *errs);
/* cache.h:33-36 */
uint32_t    cryo_batch_get_pg_nblocks(CryoBatchCache *c, CacheEntry e);
const uint32_t *cryo_batch_get_pg_blocks(CryoBatchCache *c, CacheEntry e);
char       *cryo_batch_get_data(CryoBatchCache *c, CacheEntry e);
uint32_t    cryo_batch_get_xid(CryoBatchCache *c, CacheEntry e);
void        cryo_batch_cache_invalidate(CryoBatchCache *c);
/* device calls made, blocks decompressed and requests served from the cache so far */
void        cryo_batch_cache_stats(const CryoBatchCache *c, uint64_t *calls, uint64_t *blocks, uint64_t *hits);

/* sequential scan with read-ahead (cryo_getnextslot's block loop, pg_cryogen.c:253-291, over the iterator of
 * scan_iterator.c): returns the next cryo block of the relation, decoded, or NULL at the end.  Empty blocks
 * are skipped (pg_cryogen.c:268-272); any other error ends the scan with *err set. */
typedef struct CryoBatchScan CryoBatchScan;
CryoBatchScan *cryo_batch_scan_begin(CryoBatchCache *c, const CryoRelOps *ops, int readahead);
char       *cryo_batch_scan_next(CryoBatchScan *s, uint32_t *blockno, uint32_t *xid, CryoError *err);
void        cryo_batch_scan_end(CryoBatchScan *s);

/* TID fetch: the random-read path (index fetch, bitmap heap scan, row lock, analyze; cryo_read_data + cryo_storage_fetch,
 * pg_cryogen.c:377-463, :862-895, :987-1034) for m TIDs at once.  Each distinct block's chain is walked once on the host
 * and all of them go to ONE cryogpu_decompress_pages_tuples_host call (a second one only when the tuples outgrow the
 * room guessed for them); only the selected tuples come back.  Not through the block cache. */
typedef struct
{
    CryoError  *err;            /* [m]: what cryo_read_data returns for the request's block */
    uint32_t   *xid;            /* [m]: the block's created_xid, for the visibility rule of pg_cryogen.c:282-290 */
    uint64_t   *first;          /* [m + 1]: request i's tuples are [first[i], first[i + 1]): one, or every item for 0 */
    const char **tuple;         /* the tuple's bytes (MAXALIGNed), NULL when the position does not exist */
    uint32_t   *len;
    uint64_t    ntuples;
    uint64_t    calls;          /* device calls made */
    void       *data_;          /* private: the packed tuples and their entries */
    uint64_t   *tup_off_;
    uint32_t   *tup_len_;
} CryoFetchResult;

/* tid_block[i], tid_pos[i]: ItemPointer i (the block of the cryo block's first page, a 1-based item position; 0 = every
 * item of the block, as a lossy bitmap page asks).  Returns 0 or a cryogpu call code; free the result either way. */
int         cryo_batch_fetch_tuples(cryogpu_ctx *gpu, const CryoRelOps *ops, const uint32_t *tid_block, const uint32_t *tid_pos,
                                    int m, CryoFetchResult *res);
void        cryo_fetch_result_free(CryoFetchResult *res);

/* write side */
typedef struct CryoBatchWriter CryoBatchWriter;
CryoBatchWriter *cryo_batch_writer_create(cryogpu_ctx *gpu, const CryoRelOps *ops, int method, int level_or_accel,
                                          int batch_blocks, uint32_t xid);
/* cryo_multi_insert_internal's loop body (pg_cryogen.c:626-650): the tuple goes into the current block; a full
 * block is queued (not flushed) and a new one started.  Returns 0 and the item pointer (block, 1-based
 * position), or -1 when the tuple cannot fit an empty block. */
int         cryo_batch_insert(CryoBatchWriter *w, const void *tuple, uint32_t len, uint32_t *tid_block, uint32_t *tid_pos);
int         cryo_batch_insert_many(CryoBatchWriter *w, const void *tuples, uint32_t len, uint32_t count);
/* flush_modify_state for everything queued plus the current block: one device call.  Returns 0 or a cryogpu call code. */
int         cryo_batch_flush(CryoBatchWriter *w);
void        cryo_batch_writer_stats(const CryoBatchWriter *w, uint64_t *calls, uint64_t *blocks, uint64_t *pages);
double      cryo_batch_writer_flush_seconds(const CryoBatchWriter *w);   /* time spent in the device calls */
void        cryo_batch_writer_destroy(CryoBatchWriter *w);

/* an in-memory relation for tests and benchmarks (a stand-in for the buffer manager) */
typedef struct CryoMemRel CryoMemRel;
CryoMemRel *cryo_memrel_create(uint32_t max_pages);
void        cryo_memrel_destroy(CryoMemRel *r);
CryoRelOps  cryo_memrel_ops(CryoMemRel *r);
uint8_t    *cryo_memrel_pages(CryoMemRel *r, uint32_t *nblocks);

#endif /* CRYO_BATCH_H */
