/*
 * lz4_encode.cuh -- batched LZ4 *block* compression, one CTA per cryo block.
 *
 * Replaces LZ4_compress_fast as called by the reference at compression.c:70-72
 * (lz4_compress, compression.c:61-77): CRYO_BLCKSZ plaintext bytes in, one raw LZ4
 * block out (no frame, no size prefix), lz4_acceleration (compression.c:72) steering
 * the search.  The output is a standard LZ4 block: it round-trips through
 * LZ4_decompress_safe byte-identically; it is not byte-identical to liblz4's output
 * (nothing on disk or in the regression suite depends on the compressed bytes,
 * SURVEY.md section 4), and its size stays within the tolerance stated in DESIGN.md.
 *
 * Parallel decomposition.  Greedy LZ4 matching is a serial walk (where the next
 * search starts depends on the match just found), so the block is cut into
 * LZ4E_SEGS segments and every warp walks its own segment with a private
 * 4 096-entry hash table in shared memory (liblz4's table size for 64 KiB inputs):
 *   - 32 consecutive search positions are probed at once, one per lane (hash of 4
 *     bytes, table lookup, 4-byte verify), the table is updated for all of them, and
 *     the first hit in scan order wins (ballot + ffs) -- the greedy choice;
 *   - matches are extended backwards and forwards 32 bytes per step (ballot of the
 *     first mismatch);
 *   - misses widen the stride exactly like liblz4's skip schedule:
 *     step = (acceleration << 6 + attempts) >> 6.
 * Every warp writes the body of its segment's sequences to a scratch stream.  A
 * literal run is just input bytes, so runs that straddle segment boundaries need no
 * fix-up pass: once the last segment of a block is done the final layout is a prefix
 * sum over at most LZ4E_SEGS pieces, and the warp that finished it copies "token +
 * extension + literals from the input + body from scratch" into place with coalesced
 * 16-byte stores.  Segments are work items of a queue (lz4_encode_worker): no CTA barrier.
 */
#pragma once
#include "cryo_common.cuh"

#define LZ4E_WARPS    16
#define LZ4E_THREADS  (32 * LZ4E_WARPS)
#define LZ4E_HASHLOG  12
#define LZ4E_HASH_BYTES ((1u << LZ4E_HASHLOG) * 2u)
#define LZ4E_MAXSEG   65536u          /* positions fit the u16 hash entries */
#define LZ4E_MAXSEGS  2048            /* block_size <= 128 MiB */
#define LZ4E_META     (LZ4E_WARPS * LZ4E_HASH_BYTES)
#define LZ4E_SMEM     (LZ4E_META + 64)
#define LZ4E_MFLIMIT  12u
#define LZ4E_LASTLIT  5u

struct Lz4eSeg
{
    uint32_t    first_match;    /* segment-relative start of the first match (len if none) */
    uint32_t    tail_start;     /* segment-relative end of the last match */
    uint32_t    body;           /* scratch bytes: first offset .. last match-length extension */
    int32_t     ml0;            /* first match length - 4, or -1 when the segment has no match */
    /* filled in by the layout pass */
    uint32_t    lit0;           /* input position of the first literal of this segment's piece */
    uint32_t    LL;             /* literal count of the piece's first token */
    uint32_t    at;             /* offset of the piece in dst, ~0u when the segment has no piece */
    uint32_t    pad;
};
#ifdef CRYO_EMU
#define CRYO_HD static inline
#else
#define CRYO_HD __host__ __device__ static inline
#endif
CRYO_HD size_t lz4e_nsegs(uint32_t n)
{
    size_t s = ((size_t) n + LZ4E_MAXSEG - 1) / LZ4E_MAXSEG;

    return s < LZ4E_WARPS ? LZ4E_WARPS : s;
}

/* scratch per block: segment streams (bound of every segment) + segment metadata */
CRYO_HD size_t lz4e_scratch_bytes(uint32_t n)
{
    size_t segs = lz4e_nsegs(n);

    return (((size_t) n + n / 255 + 96 * segs + 1024) + 15) / 16 * 16 + segs * sizeof(Lz4eSeg);
}

CRYO_DEV uint32_t lz4e_ld4(const uint8_t *p)
{
    uintptr_t a = (uintptr_t) p & ~(uintptr_t) 3;
    uint32_t  w0 = __ldg(reinterpret_cast<const uint32_t *>(a));
    uint32_t  w1 = __ldg(reinterpret_cast<const uint32_t *>(a + 4));

    return __funnelshift_r(w0, w1, ((uint32_t) (uintptr_t) p & 3u) * 8u);
}

CRYO_DEV uint32_t lz4e_extlen(uint32_t v)       /* bytes of length extension for a value >= 15 */
{
    return v < 15 ? 0u : (v - 15) / 255 + 1;
}

/* warp writes the extension bytes of `v` (v >= 15) at p: (v-15)/255 x 0xFF then the rest */
CRYO_DEV void lz4e_put_ext(uint8_t *p, uint32_t v, uint32_t lane)
{
    uint32_t r = v - 15, full = r / 255;

    for (uint32_t i = lane; i < full; i += 32)
        p[i] = 255;
    if (lane == 0)
        p[full] = (uint8_t) (r - full * 255);
}

/*
 * table[h] = v for every lane with `on`, by the whole warp.  Where lanes share a slot the highest lane (the latest
 * position, as liblz4's serial walk would leave it) writes alone: CUDA leaves unspecified which of several stores
 * to one address lands, and a table that depended on it would make a block's stream depend on how the warps were
 * scheduled, so on its neighbours in the batch.
 */
CRYO_DEV void lz4e_insert(uint16_t *table, uint32_t h, uint16_t v, bool on, uint32_t lane)
{
    const uint32_t peers = __match_any_sync(CRYO_FULL, on ? h : ~0u);

    if (on && lane == 31u - (uint32_t) __clz((int) peers))
        table[h] = v;
}

/*
 * One warp compresses in[0, len) (one segment) into the scratch stream `body`.
 * Matches never start after len - 12 and never cover the last 5 bytes (the LZ4 end
 * of block rules, applied to every segment so that any of them may be the last).
 */
CRYO_DEV void lz4e_segment(const uint8_t *in, uint32_t len, uint32_t hist, int accel, uint8_t *body,
                           uint16_t *table, Lz4eSeg *meta, uint32_t lane)
{
    uint32_t anchor = 0, p = 0, op = 0, lead = 0;
    int32_t  ml0 = -1;
    const uint32_t start_attempts = (uint32_t) accel << 6;
    uint32_t attempts = start_attempts;
    uint32_t cont_off = 0;          /* offset of a match that continues across the segment start */

    for (uint32_t i = lane; i < (1u << LZ4E_HASHLOG) / 8; i += 32)
        reinterpret_cast<uint4 *>(table)[i] = make_uint4(0, 0, 0, 0);
    __syncwarp();
    /*
     * History.  The table holds positions as 16 bits, counted from H bytes before the segment.  A block of
     * the usual size is cut into 64 KiB segments -- LZ4's whole window -- and H is 0; a small block (the
     * 64 KiB blocks of BASELINE.json's acceleration sweep become 4 KiB segments) would lose most of its
     * matches at the segment boundaries, so the warp first enters every position of the bytes before its
     * segment into the table (inserts only: cheap beside the search), most recent last, as liblz4's single
     * walk would have left them.
     */
    const uint32_t H = hist + len <= 65535u ? hist : (len < 65535u ? 65535u - len : 0u);

    if (len > LZ4E_MFLIMIT && H)
    {
        /* every hstep-th position: 1 up to acceleration 2, then wider, as liblz4's own walk skips more the higher
         * the acceleration; four loads in flight per lane */
        const uint32_t hstep = accel <= 2 ? 1u : accel <= 8 ? 2u : accel <= 16 ? 4u : 8u;

        for (uint32_t q0 = 0; q0 < H; q0 += 128u * hstep)
        {
            uint32_t v[4];

#pragma unroll
            for (uint32_t u = 0; u < 4; u++)
            {
                const uint32_t q = q0 + (32u * u + lane) * hstep;

                v[u] = q < H ? lz4e_ld4(in + (int32_t) q - (int32_t) H) : 0u;
            }
#pragma unroll
            for (uint32_t u = 0; u < 4; u++)
            {
                const uint32_t q = q0 + (32u * u + lane) * hstep;

                lz4e_insert(table, (v[u] * 2654435761u) >> (32 - LZ4E_HASHLOG), (uint16_t) q, q < H, lane);
            }
        }
        __syncwarp();
    }
    if (len > LZ4E_MFLIMIT)
    {
        const uint32_t mflimit = len - LZ4E_MFLIMIT;      /* last position a match may start at */
        const uint32_t matchlimit = len - LZ4E_LASTLIT;   /* matches end at or before this */

        /* a run or short period that continues from the previous segment (the zero run of a
         * sparse block spans many segments): try a few small offsets into the bytes before the
         * segment, so that the segment can open with a match instead of `step` literals */
        if (hist >= 64)
        {
            const uint32_t o = lane < 16 ? lane + 1 : (lane - 13) * 8;      /* 1..16, 24..144 */
            bool ok = true;

            for (uint32_t j = 0; j < 8; j++)
                ok = ok && in[j] == in[(int32_t) j - (int32_t) o];
            uint32_t mm = __ballot_sync(CRYO_FULL, ok);

            if (mm)
            {
                int kk = __ffs((int) mm) - 1;

                cont_off = kk < 16 ? (uint32_t) kk + 1 : (uint32_t) (kk - 13) * 8;
            }
        }
        while (p <= mflimit)
        {
            /* liblz4's probe schedule after an anchor: ip, ip + 1, then stride `step` */
            const uint32_t step = attempts >> 6;
            const uint32_t pos = lane == 0 ? p : p + 1 + (lane - 1) * step;
            const bool     valid = pos <= mflimit;
            uint32_t v = 0, h = 0;
            int32_t  cand = 0;              /* relative to the segment: negative = in the bytes before it */
            bool     hit = false;

            if (valid)
            {
                v = lz4e_ld4(in + pos);
                h = (v * 2654435761u) >> (32 - LZ4E_HASHLOG);
                cand = (int32_t) table[h] - (int32_t) H;
            }
            if (valid)
                hit = cand < (int32_t) pos && lz4e_ld4(in + cand) == v;
            /* the probes of one group cannot see each other through the table; a probe whose
             * 4 bytes repeat the previous probe's (runs, short periods) matches it directly */
            {
                uint32_t pv = __shfl_up_sync(CRYO_FULL, v, 1);

                if (valid && !hit && lane > 0 && pv == v)
                {
                    hit = true;
                    cand = (int32_t) (lane == 1 ? p : pos - step);
                }
            }
            uint32_t m = __ballot_sync(CRYO_FULL, hit);

            if (cont_off)
                m = 1;              /* forced: position 0 continues a match at offset cont_off */
            /* insert the probed positions up to and including the first hit; the ones behind
             * it will be probed again after the match and must still see older candidates */
            lz4e_insert(table, h, (uint16_t) (pos + H), valid && (m & ((1u << lane) - 1u)) == 0, lane);
            __syncwarp();
            if (m == 0)
            {
                p += 1 + 31 * step;
                attempts += 32;
                continue;
            }
            const int      k = __ffs((int) m) - 1;
            uint32_t       mpos = k == 0 ? p : p + 1 + (uint32_t) (k - 1) * step;
            int32_t        mcand = __shfl_sync(CRYO_FULL, cand, k);
            uint32_t       off = (uint32_t) ((int32_t) mpos - mcand);
            const bool     cont = cont_off != 0;

            if (cont)
            {
                off = cont_off;     /* source lies before the segment: no backward extension */
                mcand = 0;
                cont_off = 0;
            }

            /* extend backwards over bytes still in the literal run, 32 bytes per step */
            const uint32_t mpos0 = mpos;

            for (; !cont;)
            {
                bool eq = mpos >= anchor + 1 + lane && mcand - (int32_t) (1 + lane) >= -(int32_t) H &&
                          in[mpos - 1 - lane] == in[mcand - 1 - (int32_t) lane];
                uint32_t ne = ~__ballot_sync(CRYO_FULL, eq);
                uint32_t back = ne ? (uint32_t) __ffs((int) ne) - 1u : 32u;

                mpos -= back;
                mcand -= (int32_t) back;
                if (back < 32)
                    break;
            }
            /* extend forwards, 32 bytes per step */
            uint32_t ml = 4 + (mpos0 - mpos);

            for (;;)
            {
                uint32_t idx = mpos + ml + lane;
                bool     eq = idx < matchlimit && in[idx] == in[(int32_t) idx - (int32_t) off];
                uint32_t ne = ~__ballot_sync(CRYO_FULL, eq);

                if (ne == 0)
                {
                    ml += 32;
                    /* long runs (the ~1 MB zero run of a sparse cryo block): 512 bytes per step, the
                     * loads of a step issued together; stops at the first 128-byte group with a
                     * mismatch or within 8 bytes of the limit, the bytewise step above finishes */
                    for (bool stop = false; !stop;)
                    {
                        uint32_t x[4];

#pragma unroll
                        for (uint32_t u = 0; u < 4; u++)
                        {
                            const uint32_t i4 = mpos + ml + 128u * u + 4u * lane;

                            x[u] = i4 + 8u <= matchlimit ? (lz4e_ld4(in + i4) ^ lz4e_ld4(in + i4 - off)) : 1u;
                        }
#pragma unroll
                        for (uint32_t u = 0; u < 4; u++)
                        {
                            if (stop)
                                break;
                            if (__ballot_sync(CRYO_FULL, x[u] != 0) != 0)
                                stop = true;
                            else
                                ml += 128u;
                        }
                    }
                    continue;
                }
                ml += (uint32_t) __ffs((int) ne) - 1u;
                break;
            }
            /* emit: [token][ll ext][literals] are implicit for the first sequence */
            const uint32_t ll = mpos - anchor;

            if (ml0 < 0)
            {
                lead = ll;
                ml0 = (int32_t) (ml - 4);
            }
            else
            {
                if (lane == 0)
                    body[op] = (uint8_t) (((ll < 15 ? ll : 15u) << 4) | (ml - 4 < 15 ? ml - 4 : 15u));
                op += 1;
                if (ll >= 15)
                {
                    lz4e_put_ext(body + op, ll, lane);
                    op += lz4e_extlen(ll);
                }
                team_copy(body + op, in + anchor, ll, lane, 32);
                op += ll;
            }
            if (lane == 0)
            {
                body[op] = (uint8_t) off;
                body[op + 1] = (uint8_t) (off >> 8);
            }
            op += 2;
            if (ml - 4 >= 15)
            {
                lz4e_put_ext(body + op, ml - 4, lane);
                op += lz4e_extlen(ml - 4);
            }
            p = anchor = mpos + ml;
            attempts = start_attempts;
            /* like liblz4, remember the position two bytes before the end of the match */
            if (lane == 0 && p >= 2 && p - 2 <= mflimit)
                table[(lz4e_ld4(in + p - 2) * 2654435761u) >> (32 - LZ4E_HASHLOG)] = (uint16_t) (p - 2 + H);
            __syncwarp();
        }
    }
    if (lane == 0)
    {
        meta->first_match = ml0 < 0 ? len : lead;
        meta->tail_start = anchor;
        meta->body = op;
        meta->ml0 = ml0;
    }
}

/* segments of a block of n bytes: at most LZ4E_MAXSEG bytes each, at least LZ4E_WARPS of them when the block allows */
CRYO_HD uint32_t lz4e_seg_count(uint32_t n, uint32_t *seg_len)
{
    uint32_t nseg = (n + LZ4E_MAXSEG - 1) / LZ4E_MAXSEG;

    if (nseg < LZ4E_WARPS)
        nseg = n >= LZ4E_WARPS * 1024u ? LZ4E_WARPS : (n >= 1024u ? n / 1024u : 1u);
    const uint32_t seg = ((n + nseg - 1) / nseg + 15u) & ~15u;

    *seg_len = seg;
    return n ? (n + seg - 1) / seg : 1u;
}

/*
 * Layout and copy of one block whose segments are all done, by ONE warp.  A segment with a match owns one
 * piece = token + ll-ext + literals + body; its literals start where the previous piece's last match ended
 * (literal runs are plain input bytes, so runs that cross segment boundaries need no fix-up).
 */
CRYO_DEV void lz4e_finish_block(const uint8_t *src, uint32_t n, uint8_t *dst, uint32_t dst_cap, uint32_t *dst_size,
                                int32_t *status, uint8_t *scratch, uint32_t lane)
{
    uint32_t       seg;
    const uint32_t nseg = lz4e_seg_count(n, &seg);
    const size_t   stream_bytes = (((size_t) n + n / 255 + 96 * lz4e_nsegs(n) + 1024) + 15) / 16 * 16;
    Lz4eSeg       *meta = reinterpret_cast<Lz4eSeg *>(scratch + stream_bytes);
    const uint32_t seg_stride = seg + seg / 255 + 64;
    uint32_t       out = 0, carry_start = 0;

    /* positions: serial over at most nseg pieces, every lane the same arithmetic (the metadata is in L2) */
    for (uint32_t s = 0; s < nseg; s++)
    {
        const Lz4eSeg *ms = meta + s;

        if (ms->ml0 < 0)
            continue;
        const uint32_t LL = s * seg + ms->first_match - carry_start;

        out += 1 + lz4e_extlen(LL) + LL + ms->body;
        carry_start = s * seg + ms->tail_start;
    }
    const uint32_t total = out + 1 + lz4e_extlen(n - carry_start) + (n - carry_start);

    if (total > dst_cap)
    {
        if (lane == 0)
        {
            *dst_size = 0;
            *status = ST_OUTPUT;
        }
        return;
    }
    out = 0;
    carry_start = 0;
    for (uint32_t s = 0; s < nseg; s++)
    {
        const Lz4eSeg *ms = meta + s;

        if (ms->ml0 < 0)
            continue;
        const uint32_t LL = s * seg + ms->first_match - carry_start, m0 = (uint32_t) ms->ml0;
        uint8_t *d = dst + out;
        uint32_t o = 1;

        if (lane == 0)
            d[0] = (uint8_t) (((LL < 15 ? LL : 15u) << 4) | (m0 < 15 ? m0 : 15u));
        if (LL >= 15)
        {
            lz4e_put_ext(d + o, LL, lane);
            o += lz4e_extlen(LL);
        }
        team_copy(d + o, src + carry_start, LL, lane, 32);
        team_copy(d + o + LL, scratch + (size_t) s * seg_stride, ms->body, lane, 32);
        out += o + LL + ms->body;
        carry_start = s * seg + ms->tail_start;
    }
    {
        /* closing sequence: literals only (the last 5+ bytes of the block are in it) */
        const uint32_t LL = n - carry_start;
        uint8_t *d = dst + out;
        uint32_t o = 1;

        if (lane == 0)
            d[0] = (uint8_t) ((LL < 15 ? LL : 15u) << 4);
        if (LL >= 15)
        {
            lz4e_put_ext(d + o, LL, lane);
            o += lz4e_extlen(LL);
        }
        team_copy(d + o, src + carry_start, LL, lane, 32);
    }
    if (lane == 0)
    {
        *dst_size = total;
        *status = ST_OK;
    }
}

/*
 * The encoder's work loop, one warp.  Work items are (block, segment) pairs handed out in order from a
 * queue in global memory; the warp that finishes the last segment of a block lays the block out.  With one
 * CTA per block (round 1) fifteen warps waited at a barrier for the one whose segment holds the tuples of
 * a sparse cryo block (68 % of the stall samples, profiles/r01g_other_kernels_ncu_summary.txt); here they take
 * segments of the next blocks instead.
 *   queue[0]: next item; done[b]: finished segments of block b (both zeroed by the caller);
 *   scratch: lz4e_scratch_bytes(n) per block; table: this warp's LZ4E_HASH_BYTES of shared memory.
 */
CRYO_DEV void lz4_encode_worker(const uint8_t *src, uint64_t src_stride, uint32_t n, uint8_t *dst, uint64_t dst_stride,
                                uint32_t dst_cap, int accel, uint32_t *dst_size, int32_t *status, uint8_t *scratch,
                                uint64_t scratch_stride, uint32_t nblocks, uint32_t *queue, uint32_t *done,
                                uint16_t *table, uint32_t lane)
{
    if (accel < 1)
        accel = 1;                      /* liblz4: acceleration < 1 means 1 (SURVEY B.1) */
    if (accel > 65537)
        accel = 65537;
    /* 32 positions are probed per step here, so a denser schedule than liblz4's costs little: above
     * acceleration 2 the stride is half of liblz4's.  With liblz4's own stride the phase of the sparse
     * probes decides which matches are seen and small sparse blocks came out up to 1.24 x the
     * reference's size at accelerations 10..40 (profiles/r02_ratio_sweep.txt); halved, every block
     * kind stays within the 1.10 x tolerance of DESIGN.md section 1 at every acceleration. */
    if (accel > 2)
        accel = (accel + 1) / 2;
    uint32_t       seg;
    const uint32_t nseg = lz4e_seg_count(n, &seg);
    const size_t   stream_bytes = (((size_t) n + n / 255 + 96 * lz4e_nsegs(n) + 1024) + 15) / 16 * 16;
    const uint32_t seg_stride = seg + seg / 255 + 64;
    const uint64_t items = (uint64_t) nblocks * nseg;

    for (;;)
    {
        uint32_t w = 0;

        if (lane == 0)
            w = atomicAdd(queue, 1u);
        w = __shfl_sync(CRYO_FULL, w, 0);
        if (w >= items)
            return;
        const uint32_t b = w / nseg, s = w % nseg;
        const uint8_t *bsrc = src + b * src_stride;
        uint8_t       *bscr = scratch + b * scratch_stride;
        Lz4eSeg       *meta = reinterpret_cast<Lz4eSeg *>(bscr + stream_bytes);
        const uint32_t lo = s * seg, len = n - lo < seg ? n - lo : seg;

        lz4e_segment(bsrc + lo, len, lo, accel, bscr + (size_t) s * seg_stride, table, meta + s, lane);
        __syncwarp();
        __threadfence();                /* the segment's stream and metadata before the count */
        uint32_t fin = 0;

        if (lane == 0)
            fin = atomicAdd(done + b, 1u);
        fin = __shfl_sync(CRYO_FULL, fin, 0);
        if (fin == nseg - 1u)
        {
            __threadfence();            /* ... and the other warps' after it */
            lz4e_finish_block(bsrc, n, dst + b * dst_stride, dst_cap, dst_size + b, status + b, bscr, lane);
        }
    }
}
