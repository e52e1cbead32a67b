/*
 * cryo_batch.c -- batched cache fill / read-ahead and batched flush around libcryogpu (cryo_batch.h).
 * Host logic only: every byte of codec work happens in libcryogpu's kernels.
 */
#define _POSIX_C_SOURCE 200809L     /* clock_gettime */
#include "cryo_batch.h"

#include <stdlib.h>
#include <string.h>
#include <time.h>

#define INVALID_BLOCK 0xFFFFFFFFu
/* page header fields, storage.h:26-67 */
#define OFF_PD_UPPER 14
#define OFF_FIRST    24
#define OFF_NEXT     28
#define OFF_XID      32
#define OFF_CSIZE    40

static uint32_t rd32(const uint8_t *p) { uint32_t v; memcpy(&v, p, 4); return v; }
static uint32_t rd16(const uint8_t *p) { uint16_t v; memcpy(&v, p, 2); return v; }

/* cryo_pages_needed, pg_cryogen.c:692-704: the pages a chain of compressed_size bytes has */
static uint32_t
pages_needed(uint64_t size)
{
    return size <= CRYO_BATCH_PAGE - 48u ? 1u
                                         : 1u + (uint32_t) ((size - (CRYO_BATCH_PAGE - 48u) + CRYO_BATCH_PAGE - 32u - 1u) / (CRYO_BATCH_PAGE - 32u));
}

/* ------------------------------------------------------------------ read side */

/*
 * The pages of the chain that starts at blk, following `next` as cache.c:151-176 does, until compressed_size is covered
 * (the reference never reads npages): the device needs the pages, the host finds them.  An empty or foreign first page
 * still goes to the device alone: it names the error (cache.c:112-129).
 * Fills pages[] / pblk[] (CRYO_BATCH_MAXPAGES at most) and returns their number; *xid: created_xid of a first page.
 */
static uint32_t
walk_chain(const CryoRelOps *ops, uint32_t blk, uint32_t relblocks, const void **pages, uint32_t *pblk, uint32_t *xid)
{
    const uint8_t *pg = ops->read_page(ops->rel, blk);
    uint32_t       want = 0, k = 0;

    if (pg && rd16(pg + OFF_PD_UPPER) != 0 && rd32(pg + OFF_FIRST) == blk)
    {
        want = pages_needed(rd32(pg + OFF_CSIZE));
        *xid = rd32(pg + OFF_XID);
    }
    while (pg && k < CRYO_BATCH_MAXPAGES)
    {
        pages[k] = pg;
        pblk[k++] = blk;
        if (k >= want)
            break;
        blk = rd32(pg + OFF_NEXT);
        if (blk == INVALID_BLOCK || blk >= relblocks)
            break;
        pg = ops->read_page(ops->rel, blk);
    }
    return k;
}

typedef struct
{
    uint32_t    blockno;        /* key (one relation per cache here; the reference keys by (relid, blockno)) */
    int         used;
    uint64_t    ts;             /* last use, for LRU (cache.c:37, :200-206) */
    uint64_t    miss;           /* the call (its stamp) that took the slot for a miss ... */
    int         req;            /* ... and that call's request that did */
    uint32_t    nblocks;        /* cache.c:39 */
    uint32_t    xid;            /* cache.c:40 */
    uint32_t    blocks[CRYO_BATCH_MAXPAGES];
    char       *data;           /* CRYO_BLCKSZ, pinned */
} Slot;

struct CryoBatchCache
{
    cryogpu_ctx *gpu;
    int         nslots;
    Slot       *slot;
    uint64_t    clock, calls, blocks, hits;
};

CryoBatchCache *
cryo_batch_cache_create(cryogpu_ctx *gpu, int nslots)
{
    CryoBatchCache *c = calloc(1, sizeof(*c));

    if (!c || nslots < 1)
        return NULL;
    c->gpu = gpu;
    c->nslots = nslots;
    c->slot = calloc((size_t) nslots, sizeof(Slot));
    for (int i = 0; c->slot && i < nslots; i++)
        if (!(c->slot[i].data = cryogpu_host_alloc(CRYO_BATCH_BLCKSZ)))
        {
            cryo_batch_cache_destroy(c);
            return NULL;
        }
    return c;
}

void
cryo_batch_cache_destroy(CryoBatchCache *c)
{
    if (!c)
        return;
    for (int i = 0; c->slot && i < c->nslots; i++)
        cryogpu_host_free(c->slot[i].data);
    free(c->slot);
    free(c);
}

void
cryo_batch_cache_invalidate(CryoBatchCache *c)
{
    for (int i = 0; i < c->nslots; i++)
        c->slot[i].used = 0;
}

static int
find_slot(CryoBatchCache *c, uint32_t blockno)
{
    for (int i = 0; i < c->nslots; i++)
        if (c->slot[i].used && c->slot[i].blockno == blockno)
            return i;
    return InvalidCacheEntry;
}

/* allocate_cache_slot, cache.c:184-230: a free slot, else the least recently used one that this call has
 * not handed out (`stamp`: slots touched by the current call carry it) */
static int
take_slot(CryoBatchCache *c, uint64_t stamp)
{
    int best = InvalidCacheEntry;

    for (int i = 0; i < c->nslots; i++)
    {
        if (!c->slot[i].used)
            return i;
        if (c->slot[i].ts >= stamp)
            continue;
        if (best == InvalidCacheEntry || c->slot[i].ts < c->slot[best].ts)
            best = i;
    }
    return best;
}

int
cryo_batch_read_data(CryoBatchCache *c, const CryoRelOps *ops, const uint32_t *blocknos, int n,
                     CacheEntry *entries, CryoError *errs)
{
    const uint32_t relblocks = ops->nblocks(ops->rel);
    const uint64_t stamp = ++c->clock;
    int         nmiss = 0;
    int        *miss = malloc(sizeof(int) * (size_t) (n > 0 ? n : 1));
    size_t      npages = 0;
    const void **pages = NULL;
    uint32_t   *pblk = NULL, *coff = NULL;
    int         rc = 0;

    if (!miss)
        return CRYOGPU_E_NOMEM;
    /* hits, and the page chains of the misses */
    for (int i = 0; i < n; i++)
    {
        entries[i] = InvalidCacheEntry;
        errs[i] = CRYO_ERR_SUCCESS;
        /* cache.c:256-260 */
        if (blocknos[i] >= relblocks || blocknos[i] == 0)
        {
            errs[i] = CRYO_ERR_WRONG_STARTING_BLOCK;
            continue;
        }
        int e = find_slot(c, blocknos[i]);

        if (e != InvalidCacheEntry)
        {
            c->slot[e].ts = stamp;
            entries[i] = e;
            if (c->slot[e].miss != stamp)       /* a repeat of this call's miss is not a hit: see below */
                c->hits++;
            continue;
        }
        e = take_slot(c, stamp);
        if (e == InvalidCacheEntry)
        {
            errs[i] = CRYO_ERR_CACHE_IS_FULL;          /* cache.c:272-273 */
            continue;
        }
        Slot *s = &c->slot[e];

        s->used = 1;
        s->blockno = blocknos[i];
        s->ts = stamp;
        s->miss = stamp;
        s->req = i;
        s->nblocks = 0;
        entries[i] = e;
        miss[nmiss++] = i;
    }
    if (nmiss)
    {
        size_t cap = (size_t) nmiss * CRYO_BATCH_MAXPAGES;

        pages = malloc(sizeof(void *) * cap);
        pblk = malloc(sizeof(uint32_t) * cap);
        coff = malloc(sizeof(uint32_t) * (size_t) (nmiss + 1));
        if (!pages || !pblk || !coff)
        {
            rc = CRYOGPU_E_NOMEM;
            goto done;
        }
        for (int m = 0; m < nmiss; m++)
        {
            Slot *s = &c->slot[entries[miss[m]]];

            coff[m] = (uint32_t) npages;
            s->nblocks = walk_chain(ops, s->blockno, relblocks, pages + npages, pblk + npages, &s->xid);
            memcpy(s->blocks, pblk + npages, sizeof(uint32_t) * s->nblocks);
            npages += s->nblocks;
        }
        coff[nmiss] = (uint32_t) npages;
        void    **dst = malloc(sizeof(void *) * (size_t) nmiss);
        uint32_t *osz = malloc(sizeof(uint32_t) * (size_t) nmiss * 3);
        int32_t  *st = malloc(sizeof(int32_t) * (size_t) nmiss * 2);

        if (!dst || !osz || !st)
            rc = CRYOGPU_E_NOMEM;
        else
        {
            for (int m = 0; m < nmiss; m++)
                dst[m] = c->slot[entries[miss[m]]].data;
            rc = cryogpu_decompress_pages_host(c->gpu, (size_t) nmiss, pages, pblk, coff, dst, CRYO_BATCH_BLCKSZ, osz, st,
                                               st + nmiss, osz + nmiss);
            c->calls++;
            c->blocks += (uint64_t) nmiss;
            for (int m = 0; rc == 0 && m < nmiss; m++)
            {
                int i = miss[m];

                if (st[m] == CRYOGPU_ST_OK && osz[m] == CRYO_BATCH_BLCKSZ)
                    continue;
                errs[i] = st[m] == CRYOGPU_ST_EMPTY_BLOCK ? CRYO_ERR_EMPTY_BLOCK
                          : st[m] == CRYOGPU_ST_WRONG_START ? CRYO_ERR_WRONG_STARTING_BLOCK
                          : CRYO_ERR_DECOMPRESSION_FAILED;
                c->slot[entries[i]].used = 0;           /* cache.c:283-286 */
                entries[i] = InvalidCacheEntry;
            }
        }
        free(dst);
        free(osz);
        free(st);
    }
done:
    if (rc != 0)
        for (int m = 0; m < nmiss; m++)
        {
            c->slot[entries[miss[m]]].used = 0;
            entries[miss[m]] = InvalidCacheEntry;
            errs[miss[m]] = CRYO_ERR_DECOMPRESSION_FAILED;
        }
    /* a block named again after its miss in this call gets that miss's outcome: its error, and its entry or none */
    for (int i = 0; i < n; i++)
    {
        const int e = entries[i];

        if (e != InvalidCacheEntry && c->slot[e].miss == stamp && c->slot[e].req != i)
        {
            errs[i] = errs[c->slot[e].req];
            entries[i] = entries[c->slot[e].req];
        }
    }
    free(miss);
    free(pages);
    free(pblk);
    free(coff);
    return rc;
}

uint32_t cryo_batch_get_pg_nblocks(CryoBatchCache *c, CacheEntry e) { return c->slot[e].nblocks; }
const uint32_t *cryo_batch_get_pg_blocks(CryoBatchCache *c, CacheEntry e) { return c->slot[e].blocks; }
char *cryo_batch_get_data(CryoBatchCache *c, CacheEntry e) { return c->slot[e].data; }
uint32_t cryo_batch_get_xid(CryoBatchCache *c, CacheEntry e) { return c->slot[e].xid; }

void
cryo_batch_cache_stats(const CryoBatchCache *c, uint64_t *calls, uint64_t *blocks, uint64_t *hits)
{
    if (calls)
        *calls = c->calls;
    if (blocks)
        *blocks = c->blocks;
    if (hits)
        *hits = c->hits;
}

/* ---- sequential scan with read-ahead ---- */

struct CryoBatchScan
{
    CryoBatchCache *c;
    const CryoRelOps *ops;
    int         readahead;
    uint32_t    cursor;         /* next block number the iterator hands out (scan_iterator.c:55: starts at 1) */
    uint8_t    *excluded;       /* scan_iterator.c:80-125 keeps ranges; one flag per block does the same here */
    uint32_t    relblocks;
    /* the window fetched by the last call */
    uint32_t   *win_block;
    CacheEntry *win_entry;
    CryoError  *win_err;
    int         win_n, win_pos;
};

CryoBatchScan *
cryo_batch_scan_begin(CryoBatchCache *c, const CryoRelOps *ops, int readahead)
{
    CryoBatchScan *s = calloc(1, sizeof(*s));

    if (!s)
        return NULL;
    if (readahead < 1)
        readahead = 1;
    if (readahead > c->nslots)
        readahead = c->nslots;
    s->c = c;
    s->ops = ops;
    s->readahead = readahead;
    s->cursor = 1;
    s->relblocks = ops->nblocks(ops->rel);
    s->excluded = calloc(s->relblocks + 1u, 1);
    s->win_block = malloc(sizeof(uint32_t) * (size_t) readahead);
    s->win_entry = malloc(sizeof(CacheEntry) * (size_t) readahead);
    s->win_err = malloc(sizeof(CryoError) * (size_t) readahead);
    return s;
}

/* the next `readahead` starting pages the iterator would reach: a page that belongs to the chain of an earlier
 * block is skipped, as it is in the reference once that block has been read (cryo_seqscan_iter_exclude, cache.c:171) */
static void
scan_fill(CryoBatchScan *s)
{
    s->win_n = 0;
    s->win_pos = 0;
    while (s->win_n < s->readahead && s->cursor < s->relblocks)
    {
        const uint32_t b = s->cursor++;

        if (s->excluded[b])
            continue;
        const uint8_t *pg = s->ops->read_page(s->ops->rel, b);

        /* follow the chain now, so that its later pages are not taken for starting pages */
        if (pg && rd16(pg + OFF_PD_UPPER) != 0 && rd32(pg + OFF_FIRST) == b)
        {
            uint32_t want = pages_needed(rd32(pg + OFF_CSIZE)), k = 1, nb = rd32(pg + OFF_NEXT);

            while (k < want && k < CRYO_BATCH_MAXPAGES && nb != INVALID_BLOCK && nb < s->relblocks)
            {
                s->excluded[nb] = 1;
                nb = rd32((const uint8_t *) s->ops->read_page(s->ops->rel, nb) + OFF_NEXT);
                k++;
            }
        }
        s->win_block[s->win_n++] = b;
    }
    if (s->win_n)
        cryo_batch_read_data(s->c, s->ops, s->win_block, s->win_n, s->win_entry, s->win_err);
}

char *
cryo_batch_scan_next(CryoBatchScan *s, uint32_t *blockno, uint32_t *xid, CryoError *err)
{
    *err = CRYO_ERR_SUCCESS;
    for (;;)
    {
        if (s->win_pos >= s->win_n)
        {
            scan_fill(s);
            if (s->win_n == 0)
                return NULL;
        }
        const int i = s->win_pos++;

        if (s->win_err[i] == CRYO_ERR_EMPTY_BLOCK)
            continue;                           /* pg_cryogen.c:268-272 */
        if (s->win_err[i] != CRYO_ERR_SUCCESS)
        {
            *err = s->win_err[i];
            *blockno = s->win_block[i];
            return NULL;
        }
        *blockno = s->win_block[i];
        *xid = cryo_batch_get_xid(s->c, s->win_entry[i]);
        return cryo_batch_get_data(s->c, s->win_entry[i]);
    }
}

void
cryo_batch_scan_end(CryoBatchScan *s)
{
    if (!s)
        return;
    free(s->excluded);
    free(s->win_block);
    free(s->win_entry);
    free(s->win_err);
    free(s);
}

/* ---- TID fetch ---- */

static int
cmp_u64(const void *a, const void *b)
{
    const uint64_t x = *(const uint64_t *) a, y = *(const uint64_t *) b;

    return x < y ? -1 : x > y;
}

static CryoError
fetch_error(int32_t st)
{
    return st == CRYOGPU_ST_OK ? CRYO_ERR_SUCCESS
           : st == CRYOGPU_ST_EMPTY_BLOCK ? CRYO_ERR_EMPTY_BLOCK
           : st == CRYOGPU_ST_WRONG_START ? CRYO_ERR_WRONG_STARTING_BLOCK
           : CRYO_ERR_DECOMPRESSION_FAILED;
}

#define FETCH_GUESS_TUPLE   8192u       /* output room guessed per single position: a heap page */
#define FETCH_GUESS_ITEMS   290u        /* entries guessed per position 0: storage.c's limit per block */

int
cryo_batch_fetch_tuples(cryogpu_ctx *gpu, const CryoRelOps *ops, const uint32_t *tid_block, const uint32_t *tid_pos, int m,
                        CryoFetchResult *res)
{
    const uint32_t relblocks = ops->nblocks(ops->rel);
    uint64_t   *key = malloc(sizeof(uint64_t) * (size_t) (m > 0 ? m : 1));
    int         nk = 0, nb = 0, rc = 0;
    uint32_t   *blk = NULL, *pblk = NULL, *coff = NULL, *sel_pos = NULL, *bxid = NULL;
    uint64_t   *sel_off = NULL, *bf = NULL, *rfirst = NULL, *rcount = NULL, dcap = 0, tcap = 0, need[2] = {0, 0};
    int32_t    *st = NULL, *me = NULL;
    const void **pages = NULL;
    size_t      npages = 0;

    memset(res, 0, sizeof(*res));
    res->err = calloc((size_t) (m > 0 ? m : 1), sizeof(CryoError));
    res->xid = calloc((size_t) (m > 0 ? m : 1), sizeof(uint32_t));
    res->first = calloc((size_t) m + 1, sizeof(uint64_t));
    rfirst = calloc((size_t) (m > 0 ? m : 1), sizeof(uint64_t));
    rcount = calloc((size_t) (m > 0 ? m : 1), sizeof(uint64_t));
    if (!key || !res->err || !res->xid || !res->first || !rfirst || !rcount)
    {
        rc = CRYOGPU_E_NOMEM;
        goto done;
    }
    /* cache.c:256-260: the metapage and blocks past the end; the others grouped by block, in request order */
    for (int i = 0; i < m; i++)
        if (tid_block[i] >= relblocks || tid_block[i] == 0)
            res->err[i] = CRYO_ERR_WRONG_STARTING_BLOCK;
        else
            key[nk++] = (uint64_t) tid_block[i] << 32 | (uint32_t) i;
    qsort(key, (size_t) nk, sizeof(uint64_t), cmp_u64);
    for (int k = 0; k < nk; k++)
        nb += k == 0 || (key[k] >> 32) != (key[k - 1] >> 32);
    blk = malloc(sizeof(uint32_t) * (size_t) (nb + 1));
    bxid = calloc((size_t) nb + 1, sizeof(uint32_t));
    coff = malloc(sizeof(uint32_t) * (size_t) (nb + 1));
    sel_off = malloc(sizeof(uint64_t) * (size_t) (nb + 1));
    bf = malloc(sizeof(uint64_t) * (size_t) (nb + 1));
    sel_pos = malloc(sizeof(uint32_t) * (size_t) (nk + 1));
    st = malloc(sizeof(int32_t) * (size_t) (nb + 1));
    me = malloc(sizeof(int32_t) * (size_t) (nb + 1));
    pages = malloc(sizeof(void *) * (size_t) (nb + 1) * CRYO_BATCH_MAXPAGES);
    pblk = malloc(sizeof(uint32_t) * (size_t) (nb + 1) * CRYO_BATCH_MAXPAGES);
    if (!blk || !bxid || !coff || !sel_off || !bf || !sel_pos || !st || !me || !pages || !pblk)
    {
        rc = CRYOGPU_E_NOMEM;
        goto done;
    }
    /* one walk per distinct block; its positions in request order (repeats and all) */
    nb = 0;
    for (int k = 0; k < nk; k++)
    {
        const uint32_t b = (uint32_t) (key[k] >> 32), pos = tid_pos[(uint32_t) key[k]];

        if (k == 0 || b != blk[nb - 1])
        {
            blk[nb] = b;
            sel_off[nb] = (uint64_t) k;
            coff[nb] = (uint32_t) npages;
            npages += walk_chain(ops, b, relblocks, pages + npages, pblk + npages, &bxid[nb]);
            nb++;
        }
        sel_pos[k] = pos;
        tcap += pos ? 1u : FETCH_GUESS_ITEMS;
        dcap += pos ? FETCH_GUESS_TUPLE : CRYO_BATCH_BLCKSZ;
    }
    sel_off[nb] = (uint64_t) nk;
    coff[nb] = (uint32_t) npages;
    /* one device call; a second one only when the guessed room was short (need says how much there is to fetch) */
    for (int attempt = 0; nb && attempt < 2; attempt++)
    {
        free(res->data_);
        free(res->tup_off_);
        free(res->tup_len_);
        res->data_ = malloc(dcap ? dcap : 1);
        res->tup_off_ = malloc(sizeof(uint64_t) * (tcap ? tcap : 1));
        res->tup_len_ = malloc(sizeof(uint32_t) * (tcap ? tcap : 1));
        if (!res->data_ || !res->tup_off_ || !res->tup_len_)
        {
            rc = CRYOGPU_E_NOMEM;
            goto done;
        }
        rc = cryogpu_decompress_pages_tuples_host(gpu, (size_t) nb, pages, pblk, coff, CRYO_BATCH_BLCKSZ, sel_off, sel_pos,
                                                  res->data_, dcap, res->tup_off_, res->tup_len_, tcap, bf, st, me, NULL, need);
        res->calls++;
        if (rc != 0 || (need[0] <= dcap && need[1] <= tcap))
            break;
        dcap = need[0];
        tcap = need[1];
    }
    if (rc != 0)
        goto done;
    /* per request: its block's error and xid, and its entries (a position 0 has the block's ntuples of them) */
    for (int d = 0, k = 0; d < nb; d++)
    {
        const CryoError e = fetch_error(st[d]);
        uint64_t        zeros = 0, ent = bf[d];

        for (uint64_t s = sel_off[d]; s < sel_off[d + 1]; s++)
            zeros += sel_pos[s] == 0;
        const uint64_t nt = zeros ? (bf[d + 1] - bf[d] - (sel_off[d + 1] - sel_off[d] - zeros)) / zeros : 0;

        for (; k < nk && (uint32_t) (key[k] >> 32) == blk[d]; k++)
        {
            const uint32_t i = (uint32_t) key[k];

            res->err[i] = e;
            if (e != CRYO_ERR_SUCCESS)
                continue;
            res->xid[i] = bxid[d];
            rfirst[i] = ent;
            rcount[i] = sel_pos[k] ? 1u : nt;
            ent += rcount[i];
        }
    }
    for (int i = 0; i < m; i++)
        res->first[i + 1] = res->first[i] + rcount[i];
    res->ntuples = res->first[m];
    res->tuple = malloc(sizeof(char *) * (size_t) (res->ntuples ? res->ntuples : 1));
    res->len = malloc(sizeof(uint32_t) * (size_t) (res->ntuples ? res->ntuples : 1));
    if (!res->tuple || !res->len)
    {
        rc = CRYOGPU_E_NOMEM;
        goto done;
    }
    for (int i = 0; i < m; i++)
        for (uint64_t j = 0; j < rcount[i]; j++)
        {
            const uint64_t e = rfirst[i] + j, t = res->first[i] + j;

            res->tuple[t] = res->tup_off_[e] == UINT64_MAX ? NULL : (const char *) res->data_ + res->tup_off_[e];
            res->len[t] = res->tup_len_[e];
        }
done:
    if (rc != 0)
        for (int i = 0; i < m; i++)
            if (res->err)
                res->err[i] = CRYO_ERR_DECOMPRESSION_FAILED;
    free(key);
    free(blk);
    free(bxid);
    free(coff);
    free(sel_off);
    free(bf);
    free(sel_pos);
    free(st);
    free(me);
    free(pages);
    free(pblk);
    free(rfirst);
    free(rcount);
    return rc;
}

void
cryo_fetch_result_free(CryoFetchResult *res)
{
    free(res->err);
    free(res->xid);
    free(res->first);
    free(res->tuple);
    free(res->len);
    free(res->data_);
    free(res->tup_off_);
    free(res->tup_len_);
    memset(res, 0, sizeof(*res));
}

/* ----------------------------------------------------------------- write side */

struct CryoBatchWriter
{
    cryogpu_ctx *gpu;
    const CryoRelOps *ops;
    int         method, level, batch;
    uint32_t    xid;
    /* the tuples of the queued blocks and the current one, appended MAXALIGNed, and their entries; pinned, sized at
     * create for batch + 1 blocks (a block holds under CRYO_BATCH_BLCKSZ bytes of tuples and at most 290 items) */
    uint8_t    *tup;
    uint64_t   *tup_off, *block_first;  /* block_first[k]: the first entry of queued block k */
    uint32_t   *tup_len;
    uint64_t    nent, nbytes;
    uint32_t    lower, upper;           /* storage.c's two counters of the current block */
    uint32_t   *target_block;   /* reserved first page of each (pg_cryogen.c:588-601) */
    int         nfull;
    int         started;        /* the current block has a reserved page */
    uint64_t    calls, blocks, pages;
    double      flush_seconds;  /* spent in the device calls (build + compress + split + copies), for benchmarks */
};

/* cryo_storage_insert, storage.c:26-50, on the current block's counters: the device builds the block image from the
 * entries at flush time.  sizeof(ItemId) there is the size of a POINTER (ItemId is ItemIdData *): 8 bytes, which
 * happens to be sizeof(CryoItemId); MaxHeapTuplesPerPage = 291 for 8 KiB pages. */
static int
storage_insert(CryoBatchWriter *w, const void *tuple, uint32_t len)
{
    if (len + 8u > w->upper - w->lower || (w->lower - 8u) / 8u + 1u >= 291u)
        return -1;
    w->upper -= (len + 7u) & ~7u;               /* MAXALIGN */
    memcpy(w->tup + w->nbytes, tuple, len);
    w->tup_off[w->nent] = w->nbytes;
    w->tup_len[w->nent++] = len;
    w->nbytes += (len + 7u) & ~7u;
    w->lower += 8;                              /* d->lower += sizeof(ItemId), storage.c:47 */
    return (int) ((w->lower - 8u) / 8u);
}

CryoBatchWriter *
cryo_batch_writer_create(cryogpu_ctx *gpu, const CryoRelOps *ops, int method, int level_or_accel, int batch_blocks,
                         uint32_t xid)
{
    CryoBatchWriter *w = calloc(1, sizeof(*w));

    if (!w || batch_blocks < 1)
        return NULL;
    const size_t blocks = (size_t) batch_blocks + 1;

    w->gpu = gpu;
    w->ops = ops;
    w->method = method;
    w->level = level_or_accel;
    w->batch = batch_blocks;
    w->xid = xid;
    w->target_block = calloc(blocks, sizeof(uint32_t));
    w->block_first = calloc(blocks + 1, sizeof(uint64_t));
    w->tup = cryogpu_host_alloc(blocks * CRYO_BATCH_BLCKSZ);
    w->tup_off = cryogpu_host_alloc(blocks * 290 * sizeof(uint64_t));
    w->tup_len = cryogpu_host_alloc(blocks * 290 * sizeof(uint32_t));
    if (!w->target_block || !w->block_first || !w->tup || !w->tup_off || !w->tup_len)
    {
        cryo_batch_writer_destroy(w);
        return NULL;
    }
    return w;
}

/* init_modify_state, pg_cryogen.c:603-617: a fresh block (cryo_init_page's counters) and its reserved first page */
static void
start_block(CryoBatchWriter *w)
{
    w->lower = 8;
    w->upper = CRYO_BATCH_BLCKSZ;
    w->block_first[w->nfull] = w->nent;
    w->target_block[w->nfull] = w->ops->extend(w->ops->rel);
    w->started = 1;
}

static uint32_t alloc_cb(void *arg) { CryoBatchWriter *w = arg; return w->ops->extend(w->ops->rel); }
static void *ptr_cb(void *arg, uint32_t blkno) { CryoBatchWriter *w = arg; return w->ops->read_page(w->ops->rel, blkno); }

/* the n queued blocks, which hold every entry so far; the packed buffer starts over */
static int
flush_blocks(CryoBatchWriter *w, int n)
{
    if (n == 0)
        return 0;
    uint32_t *np = malloc(sizeof(uint32_t) * (size_t) n * 2);
    int32_t  *st = malloc(sizeof(int32_t) * (size_t) n);
    int       rc = CRYOGPU_E_NOMEM;

    w->block_first[n] = w->nent;
    if (np && st)
    {
        struct timespec t0, t1;

        clock_gettime(CLOCK_MONOTONIC, &t0);
        rc = cryogpu_compress_tuples_pages_alloc_host(w->gpu, (size_t) n, w->method, w->level, w->tup, w->nbytes, w->tup_off,
                                                      w->tup_len, w->block_first, CRYO_BATCH_BLCKSZ, w->target_block,
                                                      alloc_cb, ptr_cb, w, w->xid, np, np + n, st);
        clock_gettime(CLOCK_MONOTONIC, &t1);
        w->flush_seconds += (double) (t1.tv_sec - t0.tv_sec) + 1e-9 * (double) (t1.tv_nsec - t0.tv_nsec);
        w->calls++;
        for (int i = 0; rc == 0 && i < n; i++)
        {
            if (st[i] != CRYOGPU_ST_OK)
                rc = CRYOGPU_E_CUDA;
            w->pages += np[i];
        }
        w->blocks += (uint64_t) n;
    }
    w->nent = 0;
    w->nbytes = 0;
    free(np);
    free(st);
    return rc;
}

int
cryo_batch_insert(CryoBatchWriter *w, const void *tuple, uint32_t len, uint32_t *tid_block, uint32_t *tid_pos)
{
    int pos;

    if (!w->started)
        start_block(w);
    if ((pos = storage_insert(w, tuple, len)) < 0)
    {
        /* pg_cryogen.c:634-647: the block is full.  The reference compresses and writes it now; here it waits
         * for its batch. */
        w->nfull++;
        w->started = 0;
        if (w->nfull == w->batch)
        {
            int rc = flush_blocks(w, w->nfull);

            w->nfull = 0;
            if (rc != 0)
                return rc;
        }
        start_block(w);
        if ((pos = storage_insert(w, tuple, len)) < 0)
            return -1;                          /* "tuple is too large to fit the cryo block" */
    }
    *tid_block = w->target_block[w->nfull];
    *tid_pos = (uint32_t) pos;
    return 0;
}

/* `count` tuples of `len` bytes each, back to back at `tuples`: the loop of cryo_multi_insert_internal (pg_cryogen.c:626-650) */
int
cryo_batch_insert_many(CryoBatchWriter *w, const void *tuples, uint32_t len, uint32_t count)
{
    uint32_t tb, tp;

    for (uint32_t i = 0; i < count; i++)
    {
        int rc = cryo_batch_insert(w, (const char *) tuples + (size_t) i * len, len, &tb, &tp);

        if (rc != 0)
            return rc;
    }
    return 0;
}

int
cryo_batch_flush(CryoBatchWriter *w)
{
    int n = w->nfull + (w->started ? 1 : 0), rc = flush_blocks(w, n);

    w->nfull = 0;
    w->started = 0;
    return rc;
}

void
cryo_batch_writer_stats(const CryoBatchWriter *w, uint64_t *calls, uint64_t *blocks, uint64_t *pages)
{
    if (calls)
        *calls = w->calls;
    if (blocks)
        *blocks = w->blocks;
    if (pages)
        *pages = w->pages;
}

double
cryo_batch_writer_flush_seconds(const CryoBatchWriter *w)
{
    return w->flush_seconds;
}

void
cryo_batch_writer_destroy(CryoBatchWriter *w)
{
    if (!w)
        return;
    cryogpu_host_free(w->tup);
    cryogpu_host_free(w->tup_off);
    cryogpu_host_free(w->tup_len);
    free(w->block_first);
    free(w->target_block);
    free(w);
}

/* ------------------------------------------------------ in-memory relation */

struct CryoMemRel
{
    uint8_t    *pages;
    uint32_t    nblocks, max_pages;
};

static uint32_t mr_nblocks(void *r) { return ((CryoMemRel *) r)->nblocks; }
static void *mr_read(void *r, uint32_t b) { CryoMemRel *m = r; return b < m->nblocks ? m->pages + (size_t) b * CRYO_BATCH_PAGE : NULL; }
static uint32_t
mr_extend(void *r)
{
    CryoMemRel *m = r;

    if (m->nblocks >= m->max_pages)
        return INVALID_BLOCK;
    memset(m->pages + (size_t) m->nblocks * CRYO_BATCH_PAGE, 0, CRYO_BATCH_PAGE);
    return m->nblocks++;
}

CryoMemRel *
cryo_memrel_create(uint32_t max_pages)
{
    CryoMemRel *m = calloc(1, sizeof(*m));

    if (!m)
        return NULL;
    m->pages = calloc(max_pages, CRYO_BATCH_PAGE);
    m->max_pages = max_pages;
    m->nblocks = 1;                             /* block 0 is the metapage (CRYO_META_PAGE, storage.h:12) */
    return m;
}

void
cryo_memrel_destroy(CryoMemRel *m)
{
    if (m)
        free(m->pages);
    free(m);
}

CryoRelOps
cryo_memrel_ops(CryoMemRel *m)
{
    CryoRelOps o = {m, mr_nblocks, mr_read, mr_extend};

    return o;
}

uint8_t *
cryo_memrel_pages(CryoMemRel *m, uint32_t *nblocks)
{
    *nblocks = m->nblocks;
    return m->pages;
}
