/*
 * tests/tuple_oracle.c -- TEST INFRASTRUCTURE ONLY (never linked into the product).
 *
 * Plain-C restatement of the batched tuple fetch (cryogpu_tuples_device and the host calls over it) for the
 * parity tests: the item walk of cryo_getnextslot (pg_cryogen.c:293) and cryo_storage_fetch (storage.c:55-68),
 * applied to a batch of decoded blocks and a selection of item positions.  Built by tests/tuple_oracle.py.
 */
#include <stdint.h>
#include <string.h>

static uint32_t get32(const uint8_t *p) { return p[0] | ((uint32_t) p[1] << 8) | ((uint32_t) p[2] << 16) | ((uint32_t) p[3] << 24); }

/*
 * Batched tuple fetch (the random-read path: cryo_storage_fetch, storage.c:55-68, for the TIDs an index or bitmap
 * scan hands over): for n decoded blocks at blocks + i * stride, the selected tuples packed into one buffer.
 *
 *   item walk   ntuples = the largest cur with cur * 8 < lower (and 8 * cur + 8 <= block_size); item p is the
 *               CryoItemId {off, len} at byte 8 * p.  The table is valid iff lower >= 8, lower <= upper <=
 *               block_size and every item lies inside [upper, block_size); otherwise the block gets
 *               CRYOGPU_ST_FORMAT (4) and no entries.
 *   selection   sel_off == NULL: every item in position order; else the positions sel_pos[sel_off[i] ..
 *               sel_off[i + 1]) in that order, repeats copied again, 0 = every item of the block.
 *   output      entries in block order, then selection order; tuple bytes at tup_off[e] (8-byte aligned, zero
 *               padding up to MAXALIGN(len)), tup_len[e] = len; a position outside 1..ntuples gives
 *               tup_off = UINT64_MAX, tup_len = 0.  Block i's entries are [block_first[i], block_first[i + 1]).
 *   status      block_status[i] (may be NULL) passes through with no entries when it is not 0; a block whose
 *               entry or byte range would cross tup_cap / data_cap gets CRYOGPU_ST_OUTPUT (2), keeps its range
 *               in block_first and writes nothing.  need[0] = bytes, need[1] = entries the whole batch needs.
 */
void
cryo_oracle_block_tuples(const uint8_t *blocks, uint64_t stride, uint32_t n, uint32_t block_size,
                         const int32_t *block_status, const uint64_t *sel_off, const uint32_t *sel_pos,
                         uint8_t *data, uint64_t data_cap, uint64_t *tup_off, uint32_t *tup_len, uint64_t tup_cap,
                         uint64_t *block_first, int32_t *status, uint64_t need[2])
{
    uint64_t ent = 0, bytes = 0;

    for (uint32_t i = 0; i < n; i++)
    {
        const uint8_t *blk = blocks + (uint64_t) i * stride;
        const uint32_t lower = get32(blk), upper = get32(blk + 4);
        uint32_t nt = 0;
        uint64_t all = 0, cnt = 0, by = 0;
        int      st = block_status ? block_status[i] : 0, ok = lower >= 8 && lower <= upper && upper <= block_size;

        block_first[i] = ent;
        if (st == 0)
        {
            for (uint32_t cur = 1; (uint64_t) cur * 8u < lower && (uint64_t) cur * 8u + 8u <= block_size; cur++)
            {
                const uint32_t off = get32(blk + 8u * cur), len = get32(blk + 8u * cur + 4);

                nt++;
                all += (len + 7u) & ~7u;
                if (off < upper || off > block_size || len > block_size - off)
                    ok = 0;
            }
            if (!ok)
                st = 4;
        }
        if (st == 0)
        {
            const uint64_t s0 = sel_off ? sel_off[i] : 0, s1 = sel_off ? sel_off[i + 1] : 1;

            for (uint64_t s = s0; s < s1; s++)
            {
                const uint32_t p = sel_off ? sel_pos[s] : 0;

                if (p == 0)
                {
                    cnt += nt;
                    by += all;
                }
                else
                {
                    cnt++;
                    if (p <= nt)
                        by += (get32(blk + 8u * p + 4) + 7u) & ~7u;
                }
            }
            if (cnt && (ent + cnt > tup_cap || bytes + by > data_cap))
                st = 2;
        }
        status[i] = st;
        if (st == 0)
        {
            const uint64_t s0 = sel_off ? sel_off[i] : 0, s1 = sel_off ? sel_off[i + 1] : 1;
            uint64_t e = ent, at = bytes;

            for (uint64_t s = s0; s < s1; s++)
            {
                const uint32_t p = sel_off ? sel_pos[s] : 0;
                const uint64_t lo = p ? p : 1, hi = p ? p : nt;

                for (uint64_t q = lo; q <= hi; q++, e++)
                {
                    if (q > nt)
                    {
                        tup_off[e] = UINT64_MAX;
                        tup_len[e] = 0;
                        continue;
                    }
                    const uint32_t off = get32(blk + 8u * q), len = get32(blk + 8u * q + 4);
                    const uint32_t al = (len + 7u) & ~7u;

                    tup_off[e] = at;
                    tup_len[e] = len;
                    memcpy(data + at, blk + off, len);
                    memset(data + at + len, 0, al - len);
                    at += al;
                }
            }
        }
        ent += cnt;
        bytes += by;
    }
    block_first[n] = ent;
    need[0] = bytes;
    need[1] = ent;
}
