/*
 * cryo_tuples.cuh -- batched tuple fetch from decoded cryo blocks in HBM: the random-read path of the reference
 * (index fetch, bitmap heap scan, row lock, analyze: cryo_storage_fetch, storage.c:55-68, reached through
 * pg_cryogen.c:377-463, :862-895, :987-1034).  The caller names tuples by item position; only the selected tuples
 * cross the bus, packed, instead of whole 1 MiB blocks.
 *
 *   select  one warp per block: the item walk of k_tuple_stats (ntuples = the largest cur with cur * 8 < lower;
 *           item p is the CryoItemId {off, len} at byte 8 * p), the table's validity (lower >= 8,
 *           lower <= upper <= block_size, every item inside [upper, block_size)), and the selection: every item,
 *           or the caller's positions in the caller's order (repeats allowed; 0 = every item of the block).  Out:
 *           the block's entry count and its packed bytes (sum of MAXALIGN(len) over the entries).
 *   scan    one CTA: exclusive prefix sums of (entries, bytes) over the batch -> block_first[], the byte start of
 *           every block, the two totals; a block whose range would cross tup_cap or data_cap is CRYOGPU_ST_OUTPUT.
 *   gather  one warp per block walks the selection again: per group of 32 entries a warp scan places them, a
 *           tuple longer than TUP_LARGE is copied by the whole warp, shorter ones by 8-lane groups (an S tuple is
 *           61 bytes).  Reads touch the item table and the selected tuples only.
 *
 * Output: tuples start on 8-byte boundaries (a HeapTupleHeader pointer into the buffer is MAXALIGNed); the pad
 * bytes up to MAXALIGN(len) are zero.  A position outside 1..ntuples gives tup_off = TUP_NONE, tup_len = 0.
 * Blocks are 8-byte aligned (stride too); the data buffer is 16-byte aligned.
 *
 * The write side runs the other way (blk_build_block, the COPY flush from packed tuples): entries in the layout the
 * gather writes in, cryo blocks out, byte for byte what cryo_init_page + cryo_storage_insert (storage.c:15-50) build.
 */
#pragma once
#include "cryo_common.cuh"

#define TUP_NONE        0xFFFFFFFFFFFFFFFFull   /* tup_off of a position that does not exist */
#define TUP_MISSING     0xFFFFFFFFu             /* internal: no item behind the position */
#define TUP_LARGE       128u                    /* longer tuples: one warp each; shorter: one 8-lane group each */
#define TUP_SCAN_THREADS 256u
#define TUP_SCAN_ITEMS  4u                      /* blocks per thread and tile of the scan */

typedef unsigned long long tup_u64;

CRYO_DEV tup_u64 tup_ld8(const uint8_t *p) { return *reinterpret_cast<const tup_u64 *>(p); }
CRYO_DEV void tup_st8(uint8_t *p, tup_u64 v) { *reinterpret_cast<tup_u64 *>(p) = v; }
CRYO_DEV uint32_t tup_maxalign(uint32_t len) { return (len + 7u) & ~7u; }

/* number of items, as k_tuple_stats counts them (block_size >= 16) */
CRYO_DEV uint32_t tup_count(const uint8_t *block, uint32_t block_size)
{
    const uint32_t lower = ld4(block);
    uint32_t n = lower ? (lower - 1u) / 8u : 0u;

    if ((tup_u64) n * 8u + 8u > block_size)
        n = block_size / 8u - 1u;
    return n;
}

CRYO_DEV uint2 tup_item(const uint8_t *block, uint32_t p)
{
    return *reinterpret_cast<const uint2 *>(block + 8u * p);
}

/*
 * Select, one warp, one block.  in_status: the decoder's / chain check's outcome (a failed block keeps it and gets
 * no entries).  sel_off == NULL: every item; else the positions sel_pos[sel_off[b] .. sel_off[b + 1]).
 */
CRYO_DEV void tup_select_block(const uint8_t *block, uint32_t block_size, int32_t in_status, const tup_u64 *sel_off,
                               const uint32_t *sel_pos, uint32_t b, tup_u64 *cnt, tup_u64 *bytes, int32_t *status,
                               uint32_t lane)
{
    int32_t st = in_status;
    tup_u64 c = 0, by = 0;

    if (st == ST_OK)
    {
        const uint32_t lower = ld4(block), upper = ld4(block + 4), n = tup_count(block, block_size);
        bool ok = lower >= 8u && lower <= upper && upper <= block_size;
        tup_u64 all = 0;

        for (uint32_t cur = 1u + lane; ok && cur <= n; cur += 32u)
        {
            const uint2 it = tup_item(block, cur);

            all += tup_maxalign(it.y);
            if (it.x < upper || it.x > block_size || it.y > block_size - it.x)
                ok = false;
        }
        ok = __all_sync(CRYO_FULL, ok);
#pragma unroll
        for (uint32_t d = 16; d; d >>= 1)
            all += __shfl_xor_sync(CRYO_FULL, all, d);
        if (!ok)
            st = ST_FORMAT;
        else if (!sel_off)
        {
            c = n;
            by = all;
        }
        else
        {
            for (tup_u64 i = sel_off[b] + lane; i < sel_off[b + 1]; i += 32u)
            {
                const uint32_t p = sel_pos[i];

                c += p == 0 ? n : 1u;
                by += p == 0 ? all : p <= n ? tup_maxalign(tup_item(block, p).y) : 0u;
            }
#pragma unroll
            for (uint32_t d = 16; d; d >>= 1)
            {
                c += __shfl_xor_sync(CRYO_FULL, c, d);
                by += __shfl_xor_sync(CRYO_FULL, by, d);
            }
        }
    }
    if (lane == 0)
    {
        *cnt = st == ST_OK ? c : 0u;
        *bytes = st == ST_OK ? by : 0u;
        *status = st;
    }
}

/*
 * Scan, one CTA of nthr threads (a multiple of 32, at most 32 warps).  ent0 / byte0: where this batch starts in the
 * caller's output (the host calls cut a batch into chunks); tup_cap / data_cap: the caller's capacities, global.
 * block_first[n + 1] and byte_first[n + 1] are global; need = {bytes, entries} of this batch.  smem: 2 x 32 words.
 */
CRYO_DEV void tup_scan(uint32_t n, const tup_u64 *cnt, const tup_u64 *bytes, int32_t *status, tup_u64 ent0, tup_u64 byte0,
                       tup_u64 tup_cap, tup_u64 data_cap, tup_u64 *block_first, tup_u64 *byte_first, tup_u64 *need,
                       tup_u64 *smem, uint32_t tid, uint32_t nthr)
{
    const uint32_t lane = tid & 31u, w = tid >> 5, nw = nthr >> 5;
    tup_u64 carry_e = 0, carry_b = 0;

    for (uint32_t base = 0; base < n; base += nthr * TUP_SCAN_ITEMS)
    {
        const uint32_t i0 = base + tid * TUP_SCAN_ITEMS;
        tup_u64 le = 0, lb = 0;

        for (uint32_t k = 0; k < TUP_SCAN_ITEMS; k++)
            if (i0 + k < n)
            {
                le += cnt[i0 + k];
                lb += bytes[i0 + k];
            }
        tup_u64 xe = le, xb = lb;

        for (uint32_t d = 1; d < 32u; d <<= 1)
        {
            const tup_u64 ye = __shfl_up_sync(CRYO_FULL, xe, d), yb = __shfl_up_sync(CRYO_FULL, xb, d);

            if (lane >= d)
            {
                xe += ye;
                xb += yb;
            }
        }
        if (lane == 31u)
        {
            smem[2 * w] = xe;
            smem[2 * w + 1] = xb;
        }
        __syncthreads();
        tup_u64 pe = carry_e, pb = carry_b, te = 0, tb = 0;

        for (uint32_t k = 0; k < nw; k++)
        {
            if (k < w)
            {
                pe += smem[2 * k];
                pb += smem[2 * k + 1];
            }
            te += smem[2 * k];
            tb += smem[2 * k + 1];
        }
        pe += xe - le;
        pb += xb - lb;
        for (uint32_t k = 0; k < TUP_SCAN_ITEMS; k++)
            if (i0 + k < n)
            {
                const uint32_t i = i0 + k;
                const tup_u64 e = ent0 + pe, by = byte0 + pb;

                block_first[i] = e;
                byte_first[i] = by;
                if (status[i] == ST_OK && cnt[i] && (e + cnt[i] > tup_cap || by + bytes[i] > data_cap))
                    status[i] = ST_OUTPUT;
                pe += cnt[i];
                pb += bytes[i];
            }
        carry_e += te;
        carry_b += tb;
        __syncthreads();
    }
    if (tid == 0)
    {
        block_first[n] = ent0 + carry_e;
        byte_first[n] = byte0 + carry_b;
        need[0] = carry_b;
        need[1] = carry_e;
    }
}

/*
 * Word k (bytes [8k, 8k + 8)) of the len-byte tuple at src, zero past len.  src has any alignment: the word is put
 * together from the aligned 8-byte words around it (the second only when it holds tuple bytes).
 */
CRYO_DEV tup_u64 tup_word(const uint8_t *src, uint32_t len, uint32_t k)
{
    const uint32_t sh = (uint32_t) ((uintptr_t) src & 7u), left = len - 8u * k;
    const uint8_t *a = src - sh + 8u * k;
    tup_u64 w = tup_ld8(a) >> (8u * sh);

    if (sh && 8u * k + 8u - sh < len)
        w |= tup_ld8(a + 8u) << (64u - 8u * sh);
    if (left < 8u)
        w &= (1ull << (8u * left)) - 1ull;
    return w;
}

/*
 * The tuple at src (any alignment) to dst (8-byte aligned), zero-padded to MAXALIGN(len), by a team of nt threads.
 * Where src and dst agree mod 16 the body moves as 16-byte vectors; otherwise (and at the ends) as aligned 8-byte
 * words, each shifted together from two aligned loads.
 */
CRYO_DEV void tup_copy(uint8_t *dst, const uint8_t *src, uint32_t len, uint32_t t, uint32_t nt)
{
    const uint32_t nw = (len + 7u) / 8u;
    uint32_t k0 = 0;

    if ((((uintptr_t) src ^ (uintptr_t) dst) & 15u) == 0)
    {
        const uint32_t h = ((uintptr_t) dst & 8u) ? 1u : 0u;     /* one word up to the first 16-byte boundary */
        const uint32_t nv = len >= 8u * h ? (len - 8u * h) / 16u : 0u;

        if (nv)
        {
            if (h && t == 0)
                tup_st8(dst, tup_ld8(src));
            for (uint32_t v = t; v < nv; v += nt)
                st16(dst + 8u * h + 16u * v, ld16(src + 8u * h + 16u * v));
            k0 = h + 2u * nv;
        }
    }
    for (uint32_t k = k0 + t; k < nw; k += nt)
        tup_st8(dst + 8u * k, tup_word(src, len, k));
}

/* Output pointers of the gather: entries / bytes are global; the arrays start at entry ent0 and byte byte0. */
struct TupOut
{
    uint8_t  *data;
    tup_u64  *tup_off;
    uint32_t *tup_len;
    tup_u64   ent0, byte0;
};

/*
 * One group of up to 32 entries, one per lane with act set, in lane order: so = the tuple's offset in the block
 * (TUP_MISSING: the position does not exist), len its length.  ent / boff: the next entry and byte, advanced.
 */
CRYO_DEV void tup_emit(bool act, uint32_t so, uint32_t len, const uint8_t *block, tup_u64 &ent, tup_u64 &boff,
                       TupOut o, uint32_t lane)
{
    const bool found = act && so != TUP_MISSING;
    const uint32_t sz = found ? tup_maxalign(len) : 0u;
    tup_u64 x = sz;

    for (uint32_t d = 1; d < 32u; d <<= 1)
    {
        const tup_u64 y = __shfl_up_sync(CRYO_FULL, x, d);

        if (lane >= d)
            x += y;
    }
    const tup_u64 total = __shfl_sync(CRYO_FULL, x, 31);
    const unsigned am = __ballot_sync(CRYO_FULL, act);
    const tup_u64 my = boff + x - sz;

    if (act)
    {
        const tup_u64 e = ent + (uint32_t) __popc(am & ((1u << lane) - 1u)) - o.ent0;

        o.tup_off[e] = found ? my : TUP_NONE;
        o.tup_len[e] = found ? len : 0u;
    }
    const bool big = found && len > TUP_LARGE, small = found && !big;
    unsigned bm = __ballot_sync(CRYO_FULL, big);

    while (bm)
    {
        const int l = __ffs((int) bm) - 1;
        const uint32_t ls = __shfl_sync(CRYO_FULL, so, l), ll = __shfl_sync(CRYO_FULL, len, l);
        const tup_u64 lo = __shfl_sync(CRYO_FULL, my, l);

        bm &= bm - 1u;
        tup_copy(o.data + (lo - o.byte0), block + ls, ll, lane, 32u);
    }
    if (__any_sync(CRYO_FULL, small))
    {
        const uint32_t g = lane >> 3;

        for (uint32_t j = 0; j < 8u; j++)
        {
            const int src = (int) (4u * j + g);
            const int sm = __shfl_sync(CRYO_FULL, small ? 1 : 0, src);
            const uint32_t ls = __shfl_sync(CRYO_FULL, so, src), ll = __shfl_sync(CRYO_FULL, len, src);
            const tup_u64 lo = __shfl_sync(CRYO_FULL, my, src);

            if (sm)
                tup_copy(o.data + (lo - o.byte0), block + ls, ll, lane & 7u, 8u);
        }
    }
    ent += (uint32_t) __popc(am);
    boff += total;
}

/* every item of the block, in position order */
CRYO_DEV void tup_emit_all(const uint8_t *block, uint32_t n, tup_u64 &ent, tup_u64 &boff, TupOut o, uint32_t lane)
{
    for (uint32_t c0 = 0; c0 < n; c0 += 32u)
    {
        const uint32_t cur = c0 + 1u + lane;
        const bool act = cur <= n;
        const uint2 it = act ? tup_item(block, cur) : make_uint2(0u, 0u);

        tup_emit(act, it.x, it.y, block, ent, boff, o, lane);
    }
}

/*
 * Gather, one warp, one block whose status after the scan is CRYOGPU_ST_OK.  ent / boff: the block's first entry
 * and byte (block_first[b], the scan's byte start).
 */
CRYO_DEV void tup_gather_block(const uint8_t *block, uint32_t block_size, const tup_u64 *sel_off, const uint32_t *sel_pos,
                               uint32_t b, tup_u64 ent, tup_u64 boff, TupOut o, uint32_t lane)
{
    const uint32_t n = tup_count(block, block_size);
    /* every item: a selection of one position 0 */
    const tup_u64 s0 = sel_off ? sel_off[b] : 0u, s1 = sel_off ? sel_off[b + 1] : 1u;

    for (tup_u64 i0 = s0; i0 < s1; i0 += 32u)
    {
        const bool have = i0 + lane < s1;
        const uint32_t p = !have ? 1u : sel_off ? sel_pos[i0 + lane] : 0u;
        unsigned zm = __ballot_sync(CRYO_FULL, have && p == 0);
        uint32_t cur = 0;

        /* runs of single positions, each followed by at most one 0 (every item) */
        for (;;)
        {
            const uint32_t z = zm ? (uint32_t) (__ffs((int) zm) - 1) : 32u;
            const bool act = have && lane >= cur && lane < z;
            uint32_t so = TUP_MISSING, len = 0;

            if (act && p >= 1u && p <= n)
            {
                const uint2 it = tup_item(block, p);

                so = it.x;
                len = it.y;
            }
            if (__any_sync(CRYO_FULL, act))
                tup_emit(act, so, len, block, ent, boff, o, lane);
            if (z == 32u)
                break;
            tup_emit_all(block, n, ent, boff, o, lane);
            zm &= zm - 1u;
            cur = z + 1u;
        }
    }
}

/* ---------------------------------------------------------------- block build */

#define BLK_THREADS     256u
#define BLK_MAX_ITEMS   290u                    /* storage.c: (lower - 8) / 8 + 1 >= MaxHeapTuplesPerPage (291) rejects */
#define BLK_SMEM        (BLK_MAX_ITEMS * 4u + 8u * 8u + 8u)     /* upper_j per entry | warp sums | two flags */

static_assert(2u * BLK_THREADS >= BLK_MAX_ITEMS, "the scan gives each thread two entries");

/*
 * One cryo block from its entries [block_first[b], block_first[b + 1]) of (tup_off, tup_len), in insertion order,
 * by one CTA of BLK_THREADS threads.  Tuple bytes are read at data + (tup_off - data_lo); an entry is malformed
 * (CRYOGPU_ST_FORMAT) when tup_off is TUP_NONE, len > block_size, or [tup_off, tup_off + len) is not inside
 * [data_lo, data_size).  A block storage.c would not take in full is CRYOGPU_ST_OUTPUT.  A failed block writes nothing.
 *
 * Acceptance is storage_insert's rule for every entry at once: with S_j = sum over k < j of MAXALIGN(len_k), before
 * entry j lower = 8 + 8j and upper = block_size - S_j, and j is taken iff len_j + 8 <= upper - lower and j < 290.
 *
 * block_size % 8 == 0 (the caller checks) keeps every lower and upper a multiple of 8, so a taken entry has
 * MAXALIGN(len_j) <= upper - lower - 8: its tuple [upper - MAXALIGN(len_j), upper) lies above its item
 * [lower, lower + 8), and the final block splits into disjoint ranges -- header [0, 8), items [8, lower), the zero
 * gap [lower, upper), tuples and their zero pad [upper, block_size).  The writes below rely on that: they go in any
 * order, by any thread, with no barrier between them.
 */
CRYO_DEV void blk_build_block(const uint8_t *data, tup_u64 data_lo, tup_u64 data_size, const tup_u64 *tup_off,
                              const uint32_t *tup_len, const tup_u64 *block_first, uint32_t b, uint32_t block_size,
                              uint8_t *dst, int32_t *status, uint32_t *smem, uint32_t tid)
{
    uint32_t *s_up = smem, *s_flag = smem + BLK_MAX_ITEMS + 16u;
    tup_u64  *s_warp = reinterpret_cast<tup_u64 *>(smem + BLK_MAX_ITEMS);
    const uint32_t lane = tid & 31u, w = tid >> 5;
    const tup_u64 e0 = block_first[b], e1 = block_first[b + 1];
    const tup_u64 cnt = e1 >= e0 ? e1 - e0 : 0u;
    bool bad = e1 < e0;

    if (tid == 0)
        s_flag[0] = s_flag[1] = 0u;
    for (tup_u64 k = tid; k < cnt; k += BLK_THREADS)
    {
        const tup_u64 off = tup_off[e0 + k], len = tup_len[e0 + k];

        if (off == TUP_NONE || len > block_size || off < data_lo || off > data_size || len > data_size - off)
            bad = true;
    }
    __syncthreads();
    if (bad)
        s_flag[0] = 1u;
    __syncthreads();
    if (s_flag[0] || cnt > BLK_MAX_ITEMS)
    {
        if (tid == 0)
            *status = s_flag[0] ? ST_FORMAT : ST_OUTPUT;
        return;
    }
    /* exclusive prefix sums of MAXALIGN(len): thread t holds entries 2t and 2t + 1 */
    const uint32_t j0 = 2u * tid, n = (uint32_t) cnt;
    const uint32_t l0 = j0 < n ? tup_len[e0 + j0] : 0u, l1 = j0 + 1u < n ? tup_len[e0 + j0 + 1u] : 0u;
    const tup_u64 a0 = tup_maxalign(l0), mine = a0 + tup_maxalign(l1);
    tup_u64 x = mine;

    for (uint32_t d = 1; d < 32u; d <<= 1)
    {
        const tup_u64 y = __shfl_up_sync(CRYO_FULL, x, d);

        if (lane >= d)
            x += y;
    }
    if (lane == 31u)
        s_warp[w] = x;
    __syncthreads();
    tup_u64 s = x - mine;

    for (uint32_t k = 0; k < w; k++)
        s += s_warp[k];
    /* entry j is taken iff len_j + 8 <= (block_size - S_j) - (8 + 8j); signed: past a refused entry it can go negative */
    bool refuse = false;

    for (uint32_t i = 0; i < 2u; i++)
    {
        const uint32_t j = j0 + i, len = i ? l1 : l0;

        if (j >= n)
            break;
        const long long room = (long long) block_size - (long long) s - 8ll - 8ll * j;

        if ((long long) len + 8ll > room)
            refuse = true;
        s += tup_maxalign(len);
        s_up[j] = (uint32_t) (block_size - s);         /* upper_j, meaningful when every entry is taken */
    }
    if (refuse)
        s_flag[1] = 1u;
    __syncthreads();
    if (s_flag[1])
    {
        if (tid == 0)
            *status = ST_OUTPUT;
        return;
    }
    const uint32_t lower = 8u + 8u * n, upper = n ? s_up[n - 1u] : block_size;

    /* header, items */
    if (tid == 0)
    {
        *status = ST_OK;
        tup_st8(dst, (tup_u64) upper << 32 | lower);
    }
    for (uint32_t i = 0; i < 2u && j0 + i < n; i++)
        tup_st8(dst + 8u + 8u * (j0 + i), (tup_u64) (i ? l1 : l0) << 32 | s_up[j0 + i]);
    /* the zero gap [lower, upper): 16-byte stores over its aligned middle, one 8-byte word at either end at most */
    {
        const uint32_t a = (lower + 15u) & ~15u, z = upper & ~15u;

        if (tid == 0 && lower < a && lower < upper)
            tup_st8(dst + lower, 0ull);
        if (tid == 1 && a <= upper && z < upper && z >= a)
            tup_st8(dst + z, 0ull);
        if (a < z)
            for (uint32_t v = tid; v < (z - a) / 16u; v += BLK_THREADS)
                st16(dst + a + 16u * v, make_uint4(0u, 0u, 0u, 0u));
    }
    /* tuples, zero-padded to MAXALIGN(len): one 8-lane group each (a team of 8 moves a 128-byte line per step) */
    for (uint32_t j = tid >> 3; j < n; j += BLK_THREADS / 8u)
        tup_copy(dst + s_up[j], data + (tup_off[e0 + j] - data_lo), tup_len[e0 + j], tid & 7u, 8u);
}
