/*
 * tests/cryogpu_stub.c -- TEST INFRASTRUCTURE ONLY (never linked into the product).
 *
 * A CPU stand-in for the five libcryogpu calls pg_cryogen_b200/host/cryo_batch.c makes, so that the batched callers'
 * host logic (block cache, read-ahead scan, TID fetch, COPY writer) runs in the CPU suite.  Each call restates what the
 * device does, from the plain restatements the repository already has:
 *
 *   gather + chain checks   pg_gather_block (csrc/cryo_pages.cuh): EMPTY_BLOCK, WRONG_START, CHAIN with the max_csize
 *                           bound and the first / next check of every page
 *   decode                  cryo_oracle_lz4_decode / cryo_oracle_zstd_decode (oracle/cryo_oracle.c)
 *   tuple selection         cryo_oracle_block_tuples (tests/tuple_oracle.c)
 *   block build             cryo_init_page + cryo_storage_insert (storage.c:15-50), as include/cryogpu.h states it
 *   compression             LZ4_compress_fast / ZSTD_compress (liblz4 / libzstd through the pg_shim headers)
 *   split                   cryo_preserve (pg_cryogen.c:761-805) as oracle/cryo_pages.c restates it; alloc is called
 *                           block by block, page by page, after every block of the batch is compressed
 *
 * tests/batch_scenarios.py compiles it with a private copy of cryo_batch.c into a temporary directory.
 */
#include <stdlib.h>
#include <string.h>

#include "cryogpu.h"
#include "cryo_oracle.h"
#include "lz4.h"
#include "zstd.h"

void cryo_oracle_block_tuples(const uint8_t *blocks, uint64_t stride, uint32_t n, uint32_t block_size,
                              const int32_t *block_status, const uint64_t *sel_off, const uint32_t *sel_pos,
                              uint8_t *data, uint64_t data_cap, uint64_t *tup_off, uint32_t *tup_len, uint64_t tup_cap,
                              uint64_t *block_first, int32_t *status, uint64_t need[2]);

#define PAGE        8192u
#define HDR         32u
#define HDR_FIRST   48u
#define INVALID     0xFFFFFFFFu

static uint32_t get16(const uint8_t *p) { return p[0] | ((uint32_t) p[1] << 8); }
static uint32_t get32(const uint8_t *p) { return get16(p) | (get16(p + 2) << 16); }
static void put16(uint8_t *p, uint32_t v) { p[0] = (uint8_t) v; p[1] = (uint8_t) (v >> 8); }
static void put32(uint8_t *p, uint32_t v) { put16(p, v & 0xFFFFu); put16(p + 2, v >> 16); }

void *cryogpu_host_alloc(size_t bytes) { return malloc(bytes ? bytes : 1); }
void cryogpu_host_free(void *p) { free(p); }

static uint32_t
pages_needed(uint64_t size)
{
    return size <= PAGE - HDR_FIRST ? 1u : 1u + (uint32_t) ((size - (PAGE - HDR_FIRST) + (PAGE - HDR) - 1) / (PAGE - HDR));
}

/* the largest stream either library writes for a block of this size (cryogpu_decompress_pages_device) */
static uint32_t
max_csize(uint32_t block_size)
{
    const uint64_t a = (uint64_t) LZ4_compressBound((int) block_size), b = ZSTD_compressBound(block_size);

    return (uint32_t) (a > b ? a : b);
}

/* pg_gather_block: the stream of the chain entries [c0, c1) into out; *method as the header has it */
static int
gather(const void *const *pages, const uint32_t *blkno, uint32_t c0, uint32_t c1, uint32_t maxc, uint8_t *out,
       uint32_t *csize, int32_t *method)
{
    *csize = 0;
    *method = 0;
    if (c1 <= c0)
        return CRYOGPU_ST_EMPTY_BLOCK;
    const uint8_t *p0 = pages[c0];

    if (get16(p0 + 14) == 0)
        return CRYOGPU_ST_EMPTY_BLOCK;
    if (get32(p0 + 24) != blkno[c0])
        return CRYOGPU_ST_WRONG_START;
    *method = (int32_t) get32(p0 + 36);
    const uint32_t cs = get32(p0 + 40);

    if (cs > maxc || pages_needed(cs) > c1 - c0)
        return CRYOGPU_ST_CHAIN;
    const uint32_t np = pages_needed(cs);
    uint32_t left = cs;
    int st = CRYOGPU_ST_OK;

    for (uint32_t k = 0; k < np; k++)
    {
        const uint8_t *pg = pages[c0 + k];
        const uint32_t hdr = k == 0 ? HDR_FIRST : HDR, l = PAGE - hdr < left ? PAGE - hdr : left;

        if (get32(pg + 24) != blkno[c0] || (k + 1 < np && get32(pg + 28) != blkno[c0 + k + 1]))
            st = CRYOGPU_ST_CHAIN;
        memcpy(out, pg + hdr, l);
        out += l;
        left -= l;
    }
    if (st == CRYOGPU_ST_OK)
        *csize = cs;
    return st;
}

static int
decode(int32_t method, const uint8_t *src, uint32_t size, uint8_t *dst, uint32_t cap, uint32_t *out_size)
{
    long r;

    *out_size = 0;
    if (method == CRYOGPU_LZ4)
        r = cryo_oracle_lz4_decode(src, size, dst, cap, NULL, NULL, NULL);
    else if (method == CRYOGPU_ZSTD)
        r = cryo_oracle_zstd_decode(src, size, dst, cap, NULL, NULL, NULL);
    else
        return CRYOGPU_ST_METHOD;
    if (r >= 0)
    {
        *out_size = (uint32_t) r;
        return CRYOGPU_ST_OK;
    }
    return r == CRYO_ORACLE_ERR_OUTPUT ? CRYOGPU_ST_OUTPUT : r == CRYO_ORACLE_ERR_OFFSET ? CRYOGPU_ST_OFFSET
           : r == CRYO_ORACLE_ERR_FORMAT ? CRYOGPU_ST_FORMAT : r == CRYO_ORACLE_ERR_SIZE ? CRYOGPU_ST_SIZE
           : CRYOGPU_ST_INPUT;
}

/* one block of a page-chain call: gather, then decode into dst */
static int
pages_block(const void *const *pages, const uint32_t *page_blkno, uint32_t c0, uint32_t c1, uint8_t *dst, uint32_t block_size,
            uint32_t *out_size, int32_t *method, uint32_t *comp_size)
{
    uint8_t *buf = malloc((size_t) (c1 > c0 ? c1 - c0 : 1) * PAGE);
    uint32_t cs;
    int      st = gather(pages, page_blkno, c0, c1, max_csize(block_size), buf, &cs, method);

    *out_size = 0;
    if (st == CRYOGPU_ST_OK)
        st = decode(*method, buf, cs, dst, block_size, out_size);
    *comp_size = cs;
    free(buf);
    return st;
}

int
cryogpu_decompress_pages_host(cryogpu_ctx *ctx, size_t n, const void *const *pages, const uint32_t *page_blkno,
                              const uint32_t *chain_off, void *const *dst, uint32_t block_size, uint32_t *out_size,
                              int32_t *status, int32_t *methods, uint32_t *comp_size)
{
    (void) ctx;
    for (size_t i = 0; i < n; i++)
    {
        uint32_t cs;

        status[i] = pages_block(pages, page_blkno, chain_off[i], chain_off[i + 1], dst[i], block_size, &out_size[i],
                                &methods[i], &cs);
        if (comp_size)
            comp_size[i] = cs;
    }
    return CRYOGPU_OK;
}

int
cryogpu_decompress_pages_tuples_host(cryogpu_ctx *ctx, size_t n, const void *const *pages, const uint32_t *page_blkno,
                                     const uint32_t *chain_off, uint32_t block_size, const uint64_t *sel_off,
                                     const uint32_t *sel_pos, void *data, uint64_t data_cap, uint64_t *tup_off,
                                     uint32_t *tup_len, uint64_t tup_cap, uint64_t *block_first, int32_t *status,
                                     int32_t *methods, uint32_t *comp_size, uint64_t *need)
{
    uint8_t *blocks = calloc(n ? n : 1, block_size);
    int32_t *dec = malloc(sizeof(int32_t) * (n ? n : 1));

    (void) ctx;
    if (!blocks || !dec)
    {
        free(blocks);
        free(dec);
        return CRYOGPU_E_NOMEM;
    }
    for (size_t i = 0; i < n; i++)
    {
        uint32_t osz, cs;

        dec[i] = pages_block(pages, page_blkno, chain_off[i], chain_off[i + 1], blocks + i * (size_t) block_size, block_size,
                             &osz, &methods[i], &cs);
        if (comp_size)
            comp_size[i] = cs;
    }
    cryo_oracle_block_tuples(blocks, block_size, (uint32_t) n, block_size, dec, sel_off, sel_pos, data, data_cap, tup_off,
                             tup_len, tup_cap, block_first, status, need);
    free(blocks);
    free(dec);
    return CRYOGPU_OK;
}

/* cryo_init_page + cryo_storage_insert for the entries [e0, e1): the status of include/cryogpu.h's block build */
static int
build_block(const uint8_t *data, uint64_t data_size, const uint64_t *tup_off, const uint32_t *tup_len, uint64_t e0,
            uint64_t e1, uint32_t block_size, uint8_t *blk)
{
    uint32_t lower = 8, upper = block_size;

    memset(blk, 0, block_size);
    for (uint64_t e = e0; e < e1; e++)
    {
        const uint64_t off = tup_off[e];
        const uint32_t len = tup_len[e];

        if (off == UINT64_MAX || len > block_size || off > data_size || len > data_size - off)
            return CRYOGPU_ST_FORMAT;
    }
    for (uint64_t e = e0; e < e1; e++)
    {
        const uint32_t len = tup_len[e];

        if ((uint64_t) len + 8u > upper - lower || (lower - 8u) / 8u + 1u >= 291u)
            return CRYOGPU_ST_OUTPUT;
        upper -= (len + 7u) & ~7u;
        memcpy(blk + upper, data + tup_off[e], len);
        put32(blk + lower, upper);
        put32(blk + lower + 4, len);
        lower += 8;
    }
    put32(blk, lower);
    put32(blk + 4, upper);
    return CRYOGPU_ST_OK;
}

int
cryogpu_compress_tuples_pages_alloc_host(cryogpu_ctx *ctx, size_t n, int method, int level_or_accel, const void *data,
                                         uint64_t data_size, const uint64_t *tup_off, const uint32_t *tup_len,
                                         const uint64_t *block_first, uint32_t block_size, const uint32_t *first_blkno,
                                         cryogpu_alloc_page_fn alloc, cryogpu_page_ptr_fn page_ptr, void *arg,
                                         uint32_t created_xid, uint32_t *npages, uint32_t *comp_size, int32_t *status)
{
    const uint32_t bound = max_csize(block_size);
    uint8_t  *blk = malloc(block_size), *comp = malloc((size_t) (n ? n : 1) * bound);
    uint32_t *blkno = NULL;
    int       rc = CRYOGPU_OK;

    (void) ctx;
    if (method != CRYOGPU_LZ4 && method != CRYOGPU_ZSTD)
        rc = CRYOGPU_E_METHOD;
    else if (!blk || !comp)
        rc = CRYOGPU_E_NOMEM;
    /* compress every block of the batch ... */
    for (size_t i = 0; rc == CRYOGPU_OK && i < n; i++)
    {
        uint8_t *c = comp + i * (size_t) bound;

        npages[i] = 0;
        comp_size[i] = 0;
        status[i] = build_block(data, data_size, tup_off, tup_len, block_first[i], block_first[i + 1], block_size, blk);
        if (status[i] != CRYOGPU_ST_OK)
            continue;
        if (method == CRYOGPU_LZ4)
        {
            const int r = LZ4_compress_fast((const char *) blk, (char *) c, (int) block_size, (int) bound, level_or_accel);

            comp_size[i] = r > 0 ? (uint32_t) r : 0;
        }
        else
        {
            const size_t r = ZSTD_compress(c, bound, blk, block_size, level_or_accel);

            comp_size[i] = ZSTD_isError(r) ? 0 : (uint32_t) r;
        }
        if (comp_size[i] == 0)
            status[i] = CRYOGPU_ST_OUTPUT;
    }
    /* ... then the block numbers, block by block, page by page, and the page images */
    blkno = rc == CRYOGPU_OK ? malloc(sizeof(uint32_t) * (size_t) (n ? n : 1) * pages_needed(bound)) : NULL;
    if (rc == CRYOGPU_OK && !blkno)
        rc = CRYOGPU_E_NOMEM;
    for (size_t i = 0; rc == CRYOGPU_OK && i < n; i++)
    {
        uint32_t *b = blkno + i * pages_needed(bound);

        if (status[i] != CRYOGPU_ST_OK)
            continue;
        b[0] = first_blkno[i];
        for (uint32_t k = 1; k < pages_needed(comp_size[i]); k++)
            b[k] = alloc(arg);
    }
    for (size_t i = 0; rc == CRYOGPU_OK && i < n; i++)
    {
        const uint32_t *b = blkno + i * pages_needed(bound), np = pages_needed(comp_size[i]);
        const uint8_t *p = comp + i * (size_t) bound;
        uint32_t left = comp_size[i];

        if (status[i] != CRYOGPU_ST_OK)
            continue;
        for (uint32_t k = 0; k < np; k++)
        {
            uint8_t *pg = page_ptr(arg, b[k]);
            const uint32_t hdr = k == 0 ? HDR_FIRST : HDR, take = PAGE - hdr < left ? PAGE - hdr : left;

            if (!pg)
            {
                rc = CRYOGPU_E_ARG;
                break;
            }
            memset(pg, 0, PAGE);
            put32(pg + 24, b[0]);
            put32(pg + 28, k + 1 < np ? b[k + 1] : INVALID);
            if (k == 0)
            {
                put16(pg + 44, np);
                put32(pg + 36, (uint32_t) method);
                put32(pg + 40, comp_size[i]);
                put32(pg + 32, created_xid);
            }
            put16(pg + 14, PAGE);
            put16(pg + 12, hdr + take);
            put16(pg + 16, PAGE);
            memcpy(pg + hdr, p, take);
            p += take;
            left -= take;
        }
        npages[i] = np;
    }
    free(blk);
    free(comp);
    free(blkno);
    return rc;
}
