/*
 * zstd_encode.cuh -- batched zstd *frame* compression, one CTA per cryo block.
 *
 * Replaces ZSTD_compress as called by the reference at compression.c:102-104
 * (zstd_compress, compression.c:93-109): CRYO_BLCKSZ plaintext bytes in, ONE standard
 * zstd frame out (magic, content size, no checksum, no dictionary -- SURVEY.md A.3),
 * zstd_compression_level (compression.c:104) steering the effort.  The output is a
 * standard RFC 8878 frame: it round-trips through ZSTD_decompress byte-identically; it
 * is not byte-identical to libzstd's output (nothing on disk or in the regression suite
 * depends on compressed bytes, SURVEY.md section 4), and its size stays within the
 * tolerance stated in DESIGN.md.
 *
 * Parallel decomposition.  The frame is cut into zstd blocks of ZSE_BLOCK = 64 KiB (the
 * format allows any size up to 128 KiB) and every warp of the CTA compresses its own
 * block start to finish with no CTA barrier:
 *
 *   RLE test      all bytes equal -> RLE_Block (the zero interior of a sparse cryo block)
 *   match finder  greedy, 32 probe positions per step (one per lane), private hash table
 *                 in shared memory, ballot picks the first hit in scan order, matches are
 *                 extended 32 bytes per step; emits (literal run, match length, offset)
 *   literals      histogram (shared-memory atomics) -> length-limited Huffman code ->
 *                 FSE-compressed (or direct) weights -> 1 or 4 streams; every lane packs
 *                 16 symbols per step, bit positions by warp scan, atomicOr into the block
 *   sequences     repeat-offset assignment that never depends on the previous block (the
 *                 history starts "unknown", a raw offset makes its slot known), LL/OF/ML
 *                 codes + histograms, normalised counts, per-table choice of predefined /
 *                 RLE / FSE_Compressed by estimated cost, the three FSE state chains run
 *                 on three lanes (they are independent), then all lanes pack the
 *                 interleaved bitstream by warp scan + atomicOr
 *
 * Blocks that do not shrink are stored Raw.  After a CTA barrier the block sizes are
 * prefix-summed and all warps copy header + body into place with coalesced stores.
 * Levels: negative levels = raw literals + strided probing (stride grows with -level), like
 * libzstd; level >= 1 (and 0) = Huffman literals, every position probed, min match 5.
 */
#pragma once
#include "cryo_common.cuh"
#include "zstd_format.cuh"
#include "zstd_decode_w.cuh"

#define ZSE_WARPS       16
#define ZSTDE_THREADS   (32 * ZSE_WARPS)
#define ZSE_BLOCK       65536u
#define ZSE_HASHLOG     12
#define ZSE_MAXSEQ      8192u
#define ZSE_PER_WARP    8192u
#define ZSE_CTL         (ZSE_WARPS * ZSE_PER_WARP)
#define ZSTDE_SMEM      (ZSE_CTL + 512)

/* global scratch per warp */
#define ZSE_SCR_SEQ     0u
#define ZSE_SCR_LIT     (ZSE_MAXSEQ * 16u)
#define ZSE_SCR_OUT     (ZSE_SCR_LIT + ZSE_BLOCK + 64u)
#define ZSE_SCR_PER_WARP (ZSE_SCR_OUT + ZSE_BLOCK + 1024u)

/* entropy-phase overlay of the per-warp shared memory (the hash table is dead by then) */
#define ZE_HIST      0        /* u32[256] literal histogram */
#define ZE_HCODE     1024     /* u16[256] Huffman code << 4 | length */
#define ZE_HLEN      1536     /* u8[256]  code lengths, then weights */
#define ZE_SORTED    1792     /* u16[256] symbols by ascending count */
#define ZE_NODEW     2304     /* u32[512] Huffman node weights */
#define ZE_PARENT    4352     /* u16[512] */
#define ZE_HDESC     5376     /* u8[192]  Huffman tree description */
#define ZE_WNORM     5568     /* i16[16] normalised counts of the weights */
#define ZE_WCELL     5600     /* u32[64] FSE cells of the weights table */
#define ZE_WENC      5856     /* u16[64] */
#define ZE_WMISC     5984     /* u16[96] scratch: cum[16] | next[16] | cumw[64] */
/* sequence-phase overlay */
#define ZQ_HIST      0        /* u32[3][64] */
#define ZQ_NORM      768      /* i16[3][64] */
#define ZQ_CUM       1152     /* u16[3][64] first enc slot of every symbol */
#define ZQ_ENC_LL    1536     /* u16[512] */
#define ZQ_ENC_OF    2560     /* u16[256] */
#define ZQ_ENC_ML    3072     /* u16[512] */
#define ZQ_CELL      4096     /* u32[512] decode-cell scratch */
#define ZQ_NEXT      6144     /* u16[64] */
#define ZQ_CUMW      6272     /* u16[66] */
#define ZQ_DESC      6416     /* u8[3][96] table descriptions */
#define ZQ_END       6704

#ifdef CRYO_EMU
#define ZSE_HD static inline
#else
#define ZSE_HD __host__ __device__ static inline
#endif
/* global scratch of one CTA (per warp: sequences, literals, the block's body) */
ZSE_HD size_t zstde_scratch_bytes(uint32_t block_size)
{
    (void) block_size;
    return (size_t) ZSE_WARPS * ZSE_SCR_PER_WARP;
}

struct ZseParams
{
    uint32_t    mm;             /* minimum match length, 4..8 */
    uint32_t    step;           /* distance between probe pairs: libzstd's stepSize (2 = every position) */
    bool        huffman;        /* compress literals */
};

CRYO_DEV ZseParams zse_params(int level)
{
    ZseParams p;

    if (level > 22)
        level = 22;
    if (level < -131072)
        level = -131072;
    if (level <= 0)
    {
        /* libzstd: negative levels = level-0 row of ZSTD_fast, targetLength = -level as
         * acceleration, literal compression off (SURVEY.md B.2); level 0 means the default 3 */
        if (level == 0)
        {
            p.mm = 5;
            p.step = 2;
            p.huffman = true;
        }
        else
        {
            /* raw literals cost 8 bits each, so matches of 5 pay; probes are denser than
             * libzstd's stepSize = 1 - level because the table only spans this 64 KiB block */
            p.mm = 5;
            p.step = 2u + ((uint32_t) (-level) - 1u) / 2u;
            p.huffman = false;
        }
    }
    else
    {
        p.mm = 5;
        p.step = 2;
        p.huffman = true;
    }
#ifdef CRYO_EMU
    if (getenv("ZSE_DBG_MM"))
        p.mm = (uint32_t) atoi(getenv("ZSE_DBG_MM"));
    if (getenv("ZSE_DBG_STEP"))
        p.step = (uint32_t) atoi(getenv("ZSE_DBG_STEP"));
#endif
    return p;
}

/* ---- small helpers ---------------------------------------------------------- */

CRYO_DEV uint32_t zse_ld4(const uint8_t *p)
{
    uintptr_t a = (uintptr_t) p & ~(uintptr_t) 3;
    uint32_t  w0 = __ldg(reinterpret_cast<const uint32_t *>(a));
    uint32_t  w1 = __ldg(reinterpret_cast<const uint32_t *>(a + 4));

    return __funnelshift_r(w0, w1, ((uint32_t) (uintptr_t) p & 3u) * 8u);
}

/* OR `nb` bits of v (v < 2^nb, nb <= 32) into the zeroed word array at bit position `bit` */
CRYO_DEV void zse_put(uint32_t *w, uint32_t bit, uint32_t v, uint32_t nb)
{
    if (nb == 0)
        return;
    uint32_t i = bit >> 5, s = bit & 31u;

    atomicOr(w + i, v << s);
    if (s + nb > 32u)
        atomicOr(w + i + 1, v >> (32u - s));
}

CRYO_DEV void zse_put_byte(uint32_t *w, uint32_t byte_pos, uint32_t v)
{
    atomicOr(w + (byte_pos >> 2), (v & 0xFFu) << (8u * (byte_pos & 3u)));
}

/* log2(x) * 256 for x >= 1 (8.8 fixed point, linear interpolation inside the octave) */
CRYO_DEV uint32_t zse_log2_fp(uint32_t x)
{
    int      h = zs_highbit(x);
    uint32_t m = h >= 8 ? (x >> (h - 8)) : (x << (8 - h));      /* 256..511 */
    uint32_t f = m - 256u;                                     /* 0..255 */

    /* log2(1+f/256)*256 ~ f + 22*f*(256-f)/4096  (max error < 2/256) */
    return ((uint32_t) h << 8) + f + ((22u * f * (256u - f)) >> 12);
}

CRYO_DEV uint32_t zse_ll_code(uint32_t ll)
{
    if (ll < 16)
        return ll;
    if (ll >= 64)
        return (uint32_t) zs_highbit(ll) + 19u;
    uint32_t c = 24;

    while (ZS_LL_BASE[c] > ll)
        c--;
    return c;
}

CRYO_DEV uint32_t zse_ml_code(uint32_t ml)         /* ml = real match length >= 3 */
{
    uint32_t b = ml - 3;

    if (b < 32)
        return b;
    if (b >= 128)
        return (uint32_t) zs_highbit(b) + 36u;
    uint32_t c = 42;

    while (ZS_ML_BASE[c] > ml)
        c--;
    return c;
}

/* warp inclusive scan */
CRYO_DEV uint32_t zse_scan_incl(uint32_t v, uint32_t lane)
{
#pragma unroll
    for (int d = 1; d < 32; d <<= 1)
    {
        uint32_t t = __shfl_up_sync(CRYO_FULL, v, d);

        if ((int) lane >= d)
            v += t;
    }
    return v;
}

/* ---- FSE: normalised counts, table description, encoding tables ------------- */

/*
 * Normalise hist[0..nsym) (total > 0, at least two symbols present) to a sum of 1 << log
 * with every present symbol >= 1.  Single lane.
 */
CRYO_DEV void zse_fse_normalize(const uint32_t *hist, int nsym, uint32_t total, int log, int16_t *norm)
{
    const uint32_t size = 1u << log;
    int32_t  rest = (int32_t) size;
    int      big = 0;
    uint32_t bigc = 0;

    for (int s = 0; s < nsym; s++)
    {
        uint32_t c = hist[s];
        int32_t  p = 0;

        if (c)
        {
            p = (int32_t) ((((uint64_t) c << log) + (total >> 1)) / total);
            if (p < 1)
                p = 1;
            if (c > bigc)
            {
                bigc = c;
                big = s;
            }
        }
        norm[s] = (int16_t) p;
        rest -= p;
    }
    if (rest > 0 || -rest < norm[big] / 2)
    {
        norm[big] = (int16_t) (norm[big] + rest);
        return;
    }
    /* too much was handed out to rare symbols: take it back from the largest, one at a time */
    while (rest < 0)
    {
        int m = 0;

        for (int s = 1; s < nsym; s++)
            if (norm[s] > norm[m])
                m = s;
        norm[m]--;
        rest++;
    }
}

/* RFC 8878 4.1.1 table description of norm[0..nsym) into dst; returns bytes.  Single lane. */
CRYO_DEV uint32_t zse_fse_write_ncount(const int16_t *norm, int nsym, int log, uint8_t *dst)
{
    uint64_t acc = (uint64_t) (log - 5);
    uint32_t nacc = 4, out = 0;
    int      remaining = 1 << log;          /* probability mass not yet described */
    int      s = 0;

    while (remaining > 0 && s < nsym)
    {
        const int bits = zs_highbit((uint32_t) remaining + 1u) + 1;
        const int lower = (1 << (bits - 1)) - 1;
        const int thr = (1 << bits) - 1 - (remaining + 1);
        const int p = norm[s++];
        int       v = p + 1;

        remaining -= p < 0 ? -p : p;
        if (v < thr)
        {
            acc |= (uint64_t) v << nacc;
            nacc += (uint32_t) bits - 1u;
        }
        else
        {
            if (v > lower)
                v += thr;
            acc |= (uint64_t) v << nacc;
            nacc += (uint32_t) bits;
        }
        if (p == 0)
        {
            /* run of further zero-probability symbols: 2-bit repeat counts */
            int z = 0;

            while (s + z < nsym && norm[s + z] == 0)
                z++;
            s += z;
            for (;;)
            {
                while (nacc >= 8)
                {
                    dst[out++] = (uint8_t) acc;
                    acc >>= 8;
                    nacc -= 8;
                }
                if (z >= 3)
                {
                    acc |= (uint64_t) 3 << nacc;
                    nacc += 2;
                    z -= 3;
                }
                else
                {
                    acc |= (uint64_t) z << nacc;
                    nacc += 2;
                    break;
                }
            }
        }
        while (nacc >= 8)
        {
            dst[out++] = (uint8_t) acc;
            acc >>= 8;
            nacc -= 8;
        }
    }
    if (nacc)
        dst[out++] = (uint8_t) acc;
    return out;
}

/* size in bits of the FSE coding of hist under norm (8.8 fixed point accumulated, rounded up) */
CRYO_DEV uint32_t zse_fse_cost_bits(const uint32_t *hist, const int16_t *norm, int nsym, int log)
{
    uint64_t c = 0;

    for (int s = 0; s < nsym; s++)
        if (hist[s])
        {
            uint32_t p = norm[s] < 0 ? 1u : (uint32_t) norm[s];

            c += (uint64_t) hist[s] * (((uint32_t) log << 8) - zse_log2_fp(p));
        }
    return (uint32_t) ((c + 255) >> 8);
}

/*
 * Encoding tables from normalised counts (warp).  enc[cum[s] + r] = the r-th cell (in cell
 * order) that decodes to symbol s; cum[] is written for nsym symbols.  cell/next/cumw are
 * scratch (u32[1<<log], u16[64], u16[66]).
 */
CRYO_DEV void zse_fse_build_enc(const int16_t *norm, int nsym, int log, uint16_t *enc, uint16_t *cum,
                                uint32_t *cell, uint16_t *next, uint16_t *cumw, uint32_t lane)
{
    const uint32_t size = 1u << log;

    fse_build_table_warp(cell, norm, nsym, log, next, cumw, lane);
    __syncwarp();
    if (lane == 0)
    {
        uint32_t a = 0;

        for (int s = 0; s < nsym; s++)
        {
            cum[s] = (uint16_t) a;
            a += norm[s] < 0 ? 1u : (uint32_t) norm[s];
        }
    }
    __syncwarp();
    for (uint32_t p = lane; p < size; p += 32)
    {
        uint32_t c = cell[p], s = c & 0xFFu, nb = (c >> 8) & 0xFFu, base = c >> 16;
        uint32_t nx = ((base + size) & 0xFFFFu) >> nb;       /* base is stored mod 2^16 */
        uint32_t cnt = norm[s] < 0 ? 1u : (uint32_t) norm[s];

        if (nb == 0 && log == 16)
            nx = size;                                        /* unreachable: log <= 9 */
        /* (base + size) < 2 * size <= 1024, so the mod-2^16 stored base is exact */
        enc[cum[s] + nx - cnt] = (uint16_t) p;
    }
    __syncwarp();
}

/* one FSE encoding step: emit the bits that lead from a cell of symbol s to state X */
CRYO_DEV uint32_t zse_fse_step(uint32_t &X, uint32_t s, const uint16_t *enc, const uint16_t *cum,
                               const int16_t *norm, int log)
{
    const uint32_t cnt = norm[s] < 0 ? 1u : (uint32_t) norm[s];
    const uint32_t x = X + (1u << log);
    int      nb = log - zs_highbit(cnt);

    if ((x >> nb) < cnt)
        nb -= 1;
    const uint32_t bits = x & ((1u << nb) - 1u);

    X = enc[cum[s] + (x >> nb) - cnt];
    return bits | ((uint32_t) nb << 12);
}

/* ---- match finder ------------------------------------------------------------ */

/*
 * Long runs: 512 bytes per step (4 groups of 4 bytes per lane, the 16 loads of a step issued
 * together), used once a match has already run for a full 32-byte step.  The zero run of a
 * sparse cryo block is ~1 MB: bytewise steps of 32 made it one dependent L2 round trip per
 * 32 bytes, with the rest of the CTA waiting at the next barrier.  Stops at the first
 * 128-byte group that holds a mismatch or reaches within 8 bytes of `len` (the unaligned
 * 4-byte loads read up to the next aligned word); the caller's bytewise loop finishes.
 */
CRYO_DEV uint32_t zse_extend_wide(const uint8_t *in, uint32_t len, uint32_t pos, uint32_t off, uint32_t ml,
                                  uint32_t lane)
{
    for (;;)
    {
        uint32_t x[4];
        bool     stop = false;

#pragma unroll
        for (uint32_t u = 0; u < 4; u++)
        {
            const uint32_t idx = pos + ml + 128u * u + 4u * lane;

            x[u] = idx + 8u <= len ? (zse_ld4(in + idx) ^ zse_ld4(in + idx - off)) : 1u;
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
        if (stop)
            return ml;
    }
}

/* warp-uniform forward extension of a match at (pos, pos - off): bytes beyond `have` */
CRYO_DEV uint32_t zse_extend(const uint8_t *in, uint32_t len, uint32_t pos, uint32_t off, uint32_t have,
                             uint32_t lane)
{
    uint32_t ml = have;

    for (;;)
    {
        uint32_t idx = pos + ml + lane;
        bool     eq = idx < len && in[idx] == in[idx - off];
        uint32_t ne = ~__ballot_sync(CRYO_FULL, eq);

        if (ne == 0)
        {
            ml += 32;
            ml = zse_extend_wide(in, len, pos, off, ml, lane);
            continue;
        }
        return ml + (uint32_t) __ffs((int) ne) - 1u;
    }
}

/*
 * One warp parses in[0, len) greedily.  Sequences go to seq[] (x = ll | (ml-3) << 16,
 * y = offset), their literals are appended to lit[].  Returns the sequence count; *nlit_out
 * is the total literal count including the run after the last match.
 *
 * Probe schedule (libzstd's ZSTD_fast, 16 pairs at a time): positions p + k*S and p + k*S + 1,
 * S = P.step growing by one for every 128 bytes scanned without a match.  Every probe also
 * tests the last used offset (a repeat-offset match costs almost nothing to code) and a
 * repeat hit wins over a hash hit that starts at most one byte earlier, like libzstd's
 * check of ip+1.
 */
CRYO_DEV uint32_t zse_find_matches(const uint8_t *in, uint32_t len, const ZseParams &P, uint4 *seq,
                                   uint8_t *lit, uint16_t *table, uint32_t lane, uint32_t *nlit_out)
{
    uint32_t anchor = 0, p = 0, nseq = 0, nlit = 0, missed = 0;
    uint32_t rep1 = 0, rep2 = 0;
    const uint32_t mm = P.mm;
    const uint32_t tailmask = mm >= 8 ? 0xFFFFFFFFu : (mm <= 4 ? 0u : ((1u << (8u * (mm - 4u))) - 1u));

    for (uint32_t i = lane; i < (1u << ZSE_HASHLOG) / 8; i += 32)
        reinterpret_cast<uint4 *>(table)[i] = make_uint4(0, 0, 0, 0);
    __syncwarp();

    if (len >= 32)
    {
        const uint32_t plimit = len - 12;       /* last probe position (8 readable bytes + slack) */

        while (p <= plimit && nseq < ZSE_MAXSEQ)
        {
            const uint32_t S = P.step + (missed >> 7);
            const uint32_t pos = p + (lane >> 1) * S + (lane & 1u);
            const bool     valid = pos <= plimit;
            uint32_t v = 0, v2 = 0, h = 0, cand = 0;
            bool     hit = false, rhit = false;

            if (valid)
            {
                v = zse_ld4(in + pos);
                v2 = zse_ld4(in + pos + 4) & tailmask;
                h = ((v * 2654435761u) ^ (v2 * 2246822519u)) >> (32 - ZSE_HASHLOG);
                cand = table[h];
                hit = cand < pos && zse_ld4(in + cand) == v &&
                      (zse_ld4(in + cand + 4) & tailmask) == v2;
                rhit = rep1 != 0 && pos >= rep1 && zse_ld4(in + pos - rep1) == v;
            }
            /* probes of one group cannot see each other through the table: a probe whose
             * bytes repeat the previous probe's (runs, short periods) matches it directly */
            {
                uint32_t pv = __shfl_up_sync(CRYO_FULL, v, 1), pv2 = __shfl_up_sync(CRYO_FULL, v2, 1);
                uint32_t pp = __shfl_up_sync(CRYO_FULL, pos, 1);

                if (valid && !hit && lane > 0 && pv == v && pv2 == v2)
                {
                    hit = true;
                    cand = pp;
                }
            }
            const uint32_t mh = __ballot_sync(CRYO_FULL, hit), mr = __ballot_sync(CRYO_FULL, rhit);
            const int      kh = mh ? __ffs((int) mh) - 1 : 64, kr = mr ? __ffs((int) mr) - 1 : 64;
            const bool     use_rep = mr != 0 && kr <= kh + 1;
            const int      k = use_rep ? kr : kh;

            {
                /* one store per slot, the highest lane's (see lz4e_insert: the winner of stores to one address
                 * is unspecified, and the stream must not depend on scheduling) */
                const bool     ins = valid && (int) lane <= (k > 31 ? 31 : k);
                const uint32_t peers = __match_any_sync(CRYO_FULL, ins ? h : ~0u);

                if (ins && lane == 31u - (uint32_t) __clz((int) peers))
                    table[h] = (uint16_t) pos;
            }
            __syncwarp();
            if (k > 31)
            {
                p += 16 * S;
                missed += 16 * S;
                continue;
            }
            uint32_t  mpos = p + ((uint32_t) k >> 1) * S + ((uint32_t) k & 1u);
            uint32_t  mcand = use_rep ? mpos - rep1 : __shfl_sync(CRYO_FULL, cand, k);
            const uint32_t off = mpos - mcand;
            const uint32_t mpos0 = mpos;

            /* extend backwards over bytes still in the literal run, 32 bytes per step */
            for (;;)
            {
                bool eq = mpos >= anchor + 1 + lane && mcand >= 1 + lane &&
                          in[mpos - 1 - lane] == in[mcand - 1 - lane];
                uint32_t ne = ~__ballot_sync(CRYO_FULL, eq);
                uint32_t back = ne ? (uint32_t) __ffs((int) ne) - 1u : 32u;

                mpos -= back;
                mcand -= back;
                if (back < 32)
                    break;
            }
            uint32_t ml = zse_extend(in, len, mpos, off, (use_rep || mm < 4 ? 4u : mm) + (mpos0 - mpos), lane);
            const uint32_t ll = mpos - anchor;

            if (lane == 0)
                seq[nseq] = make_uint4(ll | ((ml - 3u) << 16), off, 0u, 0u);
            nseq++;
            if (ll)
                team_copy(lit + nlit, in + anchor, ll, lane, 32);
            nlit += ll;
            if (off != rep1)
            {
                rep2 = rep1;
                rep1 = off;
            }
            p = anchor = mpos + ml;
            missed = 0;
            {
                /* like libzstd: remember match start + 2 and then match end - 2 (the later one where both hash
                 * to one slot) */
                const uint32_t q = lane == 0 ? mpos + 2 : p - 2;
                const bool     ins = lane < 2 && q <= plimit;
                uint32_t       hq = ~0u;

                if (ins)
                {
                    uint32_t a = zse_ld4(in + q), b = zse_ld4(in + q + 4) & tailmask;

                    hq = ((a * 2654435761u) ^ (b * 2246822519u)) >> (32 - ZSE_HASHLOG);
                }
                const uint32_t h1 = __shfl_sync(CRYO_FULL, hq, 1);

                if (ins && !(lane == 0 && h1 == hq))
                    table[hq] = (uint16_t) q;
            }
            __syncwarp();
            /* immediate matches at the second repeat offset (no literals in between) */
            while (rep2 != 0 && p <= plimit && nseq < ZSE_MAXSEQ && p >= rep2 &&
                   zse_ld4(in + p) == zse_ld4(in + p - rep2))
            {
                const uint32_t ml2 = zse_extend(in, len, p, rep2, 4u, lane);
                const uint32_t t = rep2;

                if (lane == 0)
                    seq[nseq] = make_uint4(0u | ((ml2 - 3u) << 16), rep2, 0u, 0u);
                nseq++;
                rep2 = rep1;
                rep1 = t;
                p = anchor = p + ml2;
            }
        }
    }
    if (len > anchor)
        team_copy(lit + nlit, in + anchor, len - anchor, lane, 32);
    nlit += len - anchor;
    *nlit_out = nlit;
    __syncwarp();
    return nseq;
}

/* ---- literals ---------------------------------------------------------------- */

/*
 * Length-limited (11 bits) Huffman code lengths from hist[256] (warp).  Needs >= 2 present
 * symbols.  Writes hlen[256] (0 = absent) and returns the longest length used.
 */
CRYO_DEV uint32_t zse_huf_lengths(const uint32_t *hist, uint8_t *hlen, uint16_t *sorted,
                                  uint32_t *nodew, uint16_t *parent, uint32_t lane)
{
    /* rank sort: present symbols by ascending (count, symbol); absent symbols are dropped */
    uint32_t present = 0;

    for (uint32_t s = lane; s < 256; s += 32)
    {
        hlen[s] = 0;
        present += hist[s] ? 1u : 0u;
    }
    present = __reduce_add_sync(CRYO_FULL, present);
    __syncwarp();
    for (uint32_t s = lane; s < 256; s += 32)
    {
        const uint32_t c = hist[s];

        if (c == 0)
            continue;
        uint32_t r = 0;

        for (uint32_t t = 0; t < 256; t++)
        {
            const uint32_t d = hist[t];

            r += (d != 0 && (d < c || (d == c && t < s))) ? 1u : 0u;
        }
        sorted[r] = (uint16_t) s;
    }
    __syncwarp();
    const uint32_t m = present;
    uint32_t maxlen = 0;

    if (lane == 0)
    {
        /* two-queue merge: leaves 0..m-1 (ascending), internal nodes m..2m-2 */
        for (uint32_t i = 0; i < m; i++)
            nodew[i] = hist[sorted[i]];
        uint32_t li = 0, ni = m, nn = m;

        while (nn < 2 * m - 1)
        {
            uint32_t a, b;

            if (li < m && (ni >= nn || nodew[li] <= nodew[ni]))
                a = li++;
            else
                a = ni++;
            if (li < m && (ni >= nn || nodew[li] <= nodew[ni]))
                b = li++;
            else
                b = ni++;
            nodew[nn] = nodew[a] + nodew[b];
            parent[a] = (uint16_t) nn;
            parent[b] = (uint16_t) nn;
            nn++;
        }
        /* depths, root = 2m-2; reuse nodew[] for the depth of internal nodes */
        uint32_t count[40];

        for (int i = 0; i < 40; i++)
            count[i] = 0;
        nodew[2 * m - 2] = 0;
        for (int i = (int) (2 * m - 3); i >= 0; i--)
        {
            uint32_t d = nodew[parent[i]] + 1u;

            nodew[i] = d;
            if ((uint32_t) i < m)
                count[d > 39 ? 39 : d]++;
        }
        /* enforce the 11-bit limit on the count-per-length vector (Kraft sum stays exact) */
        const int L = 11;

        for (int i = L + 1; i < 40; i++)
            count[L] += count[i];
        uint32_t total = 0;

        for (int i = L; i >= 1; i--)
            total += count[i] << (L - i);
        while (total != (1u << L))
        {
            count[L]--;
            for (int i = L - 1; i >= 1; i--)
                if (count[i])
                {
                    count[i]--;
                    count[i + 1] += 2;
                    break;
                }
            total--;
        }
        /* shortest codes to the most frequent symbols */
        uint32_t idx = m;

        for (int l = 1; l <= L; l++)
            for (uint32_t c = 0; c < count[l]; c++)
            {
                hlen[sorted[--idx]] = (uint8_t) l;
                maxlen = (uint32_t) l;
            }
    }
    maxlen = __shfl_sync(CRYO_FULL, maxlen, 0);
    __syncwarp();
    return maxlen;
}

/*
 * Tree description (RFC 8878 4.2.1) of hlen[] into desc[]; also turns hlen[] lengths into the
 * canonical codes hcode[s] = code << 4 | len.  Returns the description size, 0 when the tree
 * cannot be described (then the literals go out raw).  Warp; the serial parts run on lane 0.
 */
CRYO_DEV uint32_t zse_huf_describe(uint8_t *hlen, uint32_t maxbits, uint16_t *hcode, uint8_t *desc,
                                   uint8_t *smem, uint32_t lane)
{
    int16_t  *wnorm = reinterpret_cast<int16_t *>(smem + ZE_WNORM);
    uint32_t *wcell = reinterpret_cast<uint32_t *>(smem + ZE_WCELL);
    uint16_t *wenc = reinterpret_cast<uint16_t *>(smem + ZE_WENC);
    uint16_t *wmisc = reinterpret_cast<uint16_t *>(smem + ZE_WMISC);
    uint32_t  dsize = 0;

    /* canonical codes: cells by ascending weight (longest codes first), symbols ascending */
    if (lane == 0)
    {
        uint32_t rank_count[13], rank_start[14];

        for (int r = 0; r < 13; r++)
            rank_count[r] = 0;
        for (uint32_t s = 0; s < 256; s++)
            if (hlen[s])
                rank_count[maxbits + 1 - hlen[s]]++;
        rank_start[1] = 0;
        for (uint32_t r = 1; r <= maxbits; r++)
            rank_start[r + 1] = rank_start[r] + (rank_count[r] << (r - 1));
        for (uint32_t s = 0; s < 256; s++)
        {
            uint32_t l = hlen[s];

            if (l)
            {
                uint32_t w = maxbits + 1 - l;

                hcode[s] = (uint16_t) (((rank_start[w] >> (w - 1)) << 4) | l);
                rank_start[w] += 1u << (w - 1);
            }
            else
                hcode[s] = 0;
        }
    }
    __syncwarp();
    /* weights; the last present symbol's weight is implied */
    int last = -1;

    for (int s = 255 - (int) lane; s >= 0; s -= 32)
        if (hlen[s] && last < 0)
            last = s;
    last = (int) __reduce_max_sync(CRYO_FULL, (uint32_t) (last + 1)) - 1;
    const uint32_t nw = (uint32_t) last;        /* weights written: symbols 0 .. last-1 */

    for (uint32_t s = lane; s < 256; s += 32)
        hlen[s] = hlen[s] ? (uint8_t) (maxbits + 1 - hlen[s]) : 0;     /* now weights */
    __syncwarp();
    if (nw == 0)
        return 0;                   /* a single symbol: the caller emits RLE literals instead */

    /* FSE-compressed weights (two interleaved states), when possible and smaller */
    uint32_t fse_size = 0;

    if (nw >= 2)
    {
        uint32_t *whist = reinterpret_cast<uint32_t *>(wcell);      /* u32[16], before the cells */
        uint32_t  distinct = 0, maxc = 0;

        if (lane == 0)
        {
            for (int i = 0; i < 16; i++)
                whist[i] = 0;
            for (uint32_t s = 0; s < nw; s++)
                whist[hlen[s]]++;
            for (int i = 0; i < 13; i++)
            {
                distinct += whist[i] ? 1u : 0u;
                maxc = whist[i] > maxc ? whist[i] : maxc;
            }
        }
        distinct = __shfl_sync(CRYO_FULL, distinct, 0);
        maxc = __shfl_sync(CRYO_FULL, maxc, 0);
        if (distinct >= 2 && maxc > 1)
        {
            /* table log: FSE_optimalTableLog(6, nw, 12) */
            int log = 6;
            int srcbits = zs_highbit(nw - 1) - 2;
            int minbits = zs_highbit(nw) + 1;
            int symbits = zs_highbit(maxbits) + 2;

            if (symbits < minbits)
                minbits = symbits;
            if (srcbits < log)
                log = srcbits;
            if (minbits > log)
                log = minbits;
            if (log < 5)
                log = 5;
            if (log > 6)
                log = 6;
            uint32_t hdr = 0;

            if (lane == 0)
            {
                zse_fse_normalize(whist, (int) maxbits + 1, nw, log, wnorm);
                hdr = zse_fse_write_ncount(wnorm, (int) maxbits + 1, log, desc + 1);
            }
            hdr = __shfl_sync(CRYO_FULL, hdr, 0);
            __syncwarp();
            zse_fse_build_enc(wnorm, (int) maxbits + 1, log, wenc, wmisc, wcell, wmisc + 16, wmisc + 32, lane);
            if (lane == 0)
            {
                /* symbols alternate state 1 (even index), state 2 (odd); encoded backwards */
                uint64_t acc = 0;
                uint32_t nacc = 0, out = 1 + hdr;
                uint32_t X[2];
                int      i = (int) nw - 1;

                X[i & 1] = wenc[wmisc[hlen[i]]];
                i--;
                X[i & 1] = wenc[wmisc[hlen[i]]];
                i--;
                for (; i >= 0; i--)
                {
                    uint32_t u = zse_fse_step(X[i & 1], hlen[i], wenc, wmisc, wnorm, log);

                    acc |= (uint64_t) (u & 0xFFFu) << nacc;
                    nacc += u >> 12;
                    while (nacc >= 8)
                    {
                        desc[out++] = (uint8_t) acc;
                        acc >>= 8;
                        nacc -= 8;
                    }
                }
                acc |= (uint64_t) X[1] << nacc;
                nacc += (uint32_t) log;
                acc |= (uint64_t) X[0] << nacc;
                nacc += (uint32_t) log;
                acc |= (uint64_t) 1 << nacc;
                nacc += 1;
                while (nacc > 0)
                {
                    desc[out++] = (uint8_t) acc;
                    acc >>= 8;
                    nacc = nacc >= 8 ? nacc - 8 : 0;
                }
                fse_size = out - 1;
            }
            fse_size = __shfl_sync(CRYO_FULL, fse_size, 0);
            __syncwarp();
        }
    }
    const uint32_t direct_size = nw <= 128 ? (nw + 1) / 2 : 0xFFFFu;

    if (fse_size && fse_size < 128 && fse_size < direct_size)
    {
        if (lane == 0)
            desc[0] = (uint8_t) fse_size;
        dsize = 1 + fse_size;
    }
    else if (nw <= 128)
    {
        if (lane == 0)
        {
            desc[0] = (uint8_t) (127 + nw);
            for (uint32_t i = 0; i < nw; i += 2)
                desc[1 + i / 2] = (uint8_t) ((hlen[i] << 4) | (i + 1 < nw ? hlen[i + 1] : 0));
        }
        dsize = 1 + direct_size;
    }
    __syncwarp();
    return dsize;
}

/* total code bits of lit[0, n) under hcode (warp); lit is 16-byte aligned */
CRYO_DEV uint32_t zse_huf_stream_bits(const uint8_t *lit, uint32_t lo, uint32_t n, const uint16_t *hcode,
                                      uint32_t lane)
{
    uint32_t bits = 0;

    for (uint32_t i = lane; i < n; i += 32)
        bits += hcode[lit[lo + i]] & 15u;
    return __reduce_add_sync(CRYO_FULL, bits);
}

/*
 * Pack lit[lo, lo+n) as one backward-read Huffman stream at byte position `at` of the zeroed
 * word array w: the LAST symbol sits at the lowest bit position, the end mark above the first.
 */
CRYO_DEV void zse_huf_pack(const uint8_t *lit, uint32_t lo, uint32_t n, const uint16_t *hcode,
                           uint32_t *w, uint32_t at, uint32_t total_bits, uint32_t lane)
{
    uint32_t base = at * 8u;           /* bit position of the next (later-in-text = lower) symbol */
    const uint32_t rounds = (n + 255) / 256;

    /* 8 symbols per lane per round, walking from the end of the text to its start */
    for (uint32_t r = 0; r < rounds; r++)
    {
        /* lane 0 takes the 8 symbols nearest the end of what is left */
        const uint32_t hi = n - r * 256u;                  /* symbols [0, hi) are not packed yet */
        const uint32_t my_hi = hi > lane * 8u ? hi - lane * 8u : 0u;
        const uint32_t my_n = my_hi < 8u ? my_hi : 8u;
        /* 8 codes of up to 11 bits can exceed 64 bits: pack in two halves instead */
        uint32_t n1 = 0, n2 = 0;
        uint64_t a1 = 0, a2 = 0;

        for (uint32_t k = 0; k < my_n; k++)
        {
            uint32_t c = hcode[lit[lo + my_hi - 1 - k]];

            if (k < 4)
            {
                a1 |= (uint64_t) (c >> 4) << n1;
                n1 += c & 15u;
            }
            else
            {
                a2 |= (uint64_t) (c >> 4) << n2;
                n2 += c & 15u;
            }
        }
        const uint32_t mine = n1 + n2;
        const uint32_t incl = zse_scan_incl(mine, lane);
        const uint32_t pos = base + incl - mine;

        zse_put(w, pos, (uint32_t) a1, n1 > 32 ? 32 : n1);
        if (n1 > 32)
            zse_put(w, pos + 32, (uint32_t) (a1 >> 32), n1 - 32);
        zse_put(w, pos + n1, (uint32_t) a2, n2 > 32 ? 32 : n2);
        if (n2 > 32)
            zse_put(w, pos + n1 + 32, (uint32_t) (a2 >> 32), n2 - 32);
        base += __shfl_sync(CRYO_FULL, incl, 31);
    }
    if (lane == 0)
        zse_put(w, at * 8u + total_bits, 1u, 1u);
}

/* ---- one zstd block ------------------------------------------------------------ */

struct ZseBlockOut
{
    uint32_t    type;           /* 0 raw (copy from src), 1 RLE, 2 compressed (body in scratch) */
    uint32_t    size;           /* body bytes for type 2; regenerated size otherwise */
    uint32_t    byte;           /* RLE byte */
};

/*
 * Compress in[0, len) (len <= ZSE_BLOCK) into the warp's scratch.  smem: this warp's
 * ZSE_PER_WARP bytes.  scr: this warp's ZSE_SCR_PER_WARP bytes of global memory.
 */
CRYO_DEV ZseBlockOut zse_block(const uint8_t *in, uint32_t len, const ZseParams &P, uint8_t *smem,
                               uint8_t *scr, uint32_t lane)
{
    ZseBlockOut R;

    R.type = 0;
    R.size = len;
    R.byte = 0;
    if (len == 0)
        return R;
    /* RLE block: every byte equals the first */
    {
        const uint8_t b0 = in[0];
        bool          same = true;

        if (((uintptr_t) in & 15u) == 0 && len >= 64)
        {
            const uint32_t w = b0 * 0x01010101u;
            const uint32_t nv = len >> 4;

            for (uint32_t v0 = 0; v0 < nv && same; v0 += 128)
            {
                bool ok = true;

#pragma unroll
                for (uint32_t k = 0; k < 4; k++)
                {
                    uint32_t v = v0 + k * 32 + lane;

                    if (v < nv)
                    {
                        uint4 q = ld16(in + 16 * (size_t) v);

                        ok = ok && q.x == w && q.y == w && q.z == w && q.w == w;
                    }
                }
                same = __all_sync(CRYO_FULL, ok);
            }
            if (same)
            {
                bool ok = true;

                for (uint32_t i = (nv << 4) + lane; i < len; i += 32)
                    ok = ok && in[i] == b0;
                same = __all_sync(CRYO_FULL, ok);
            }
        }
        else
        {
            bool ok = true;

            for (uint32_t i = lane; i < len; i += 32)
                ok = ok && in[i] == b0;
            same = __all_sync(CRYO_FULL, ok);
        }
        if (same)
        {
            R.type = 1;
            R.byte = b0;
            return R;
        }
    }
    if (len < 64)
        return R;               /* tiny tail: raw */

    uint4    *seq = reinterpret_cast<uint4 *>(scr + ZSE_SCR_SEQ);
    uint8_t  *lit = scr + ZSE_SCR_LIT;
    uint32_t *ow = reinterpret_cast<uint32_t *>(scr + ZSE_SCR_OUT);
    uint32_t  nlit = 0;
    const uint32_t nseq = zse_find_matches(in, len, P, seq, lit, reinterpret_cast<uint16_t *>(smem),
                                           lane, &nlit);

    __threadfence_block();
    __syncwarp();

    /* ================= literals section: plan ================= */
    uint32_t *hist = reinterpret_cast<uint32_t *>(smem + ZE_HIST);
    uint16_t *hcode = reinterpret_cast<uint16_t *>(smem + ZE_HCODE);
    uint8_t  *hlen = smem + ZE_HLEN;
    uint8_t  *hdesc = smem + ZE_HDESC;
    uint32_t  lit_mode = 0;             /* 0 raw, 1 RLE, 2 Huffman */
    uint32_t  lit_streams = 1, lit_hdr, lit_csize = 0, desc_size = 0;
    uint32_t  sbits[4] = {0, 0, 0, 0}, sbytes[4] = {0, 0, 0, 0};
    const uint32_t seg = (nlit + 3) / 4;

    if (P.huffman && nlit >= 64)
    {
        for (uint32_t s = lane; s < 256; s += 32)
            hist[s] = 0;
        __syncwarp();
        for (uint32_t i = lane; i < nlit; i += 32)
            atomicAdd(hist + lit[i], 1u);
        __syncwarp();
        uint32_t maxc = 0, present = 0;

        for (uint32_t s = lane; s < 256; s += 32)
        {
            maxc = hist[s] > maxc ? hist[s] : maxc;
            present += hist[s] ? 1u : 0u;
        }
        maxc = __reduce_max_sync(CRYO_FULL, maxc);
        present = __reduce_add_sync(CRYO_FULL, present);
        if (present == 1)
            lit_mode = 1;
        else
        {
            const uint32_t maxbits = zse_huf_lengths(hist, hlen, reinterpret_cast<uint16_t *>(smem + ZE_SORTED),
                                                     reinterpret_cast<uint32_t *>(smem + ZE_NODEW),
                                                     reinterpret_cast<uint16_t *>(smem + ZE_PARENT), lane);

            desc_size = zse_huf_describe(hlen, maxbits, hcode, hdesc, smem, lane);
            if (desc_size)
            {
                lit_streams = nlit < 256 ? 1u : 4u;
                uint32_t total = desc_size + (lit_streams == 4 ? 6u : 0u);

                for (uint32_t k = 0; k < lit_streams; k++)
                {
                    uint32_t lo = lit_streams == 4 ? k * seg : 0u;
                    uint32_t cnt = lit_streams == 4 ? (k < 3 ? seg : nlit - 3 * seg) : nlit;

                    sbits[k] = zse_huf_stream_bits(lit, lo, cnt, hcode, lane);
                    sbytes[k] = sbits[k] / 8u + 1u;
                    total += sbytes[k];
                }
                /* libzstd keeps Huffman only when it gains at least (n >> 6) + 2 bytes */
                if (total + (nlit >> 6) + 2 < nlit && (lit_streams == 1 ? total < 1024 : true) &&
                    sbytes[0] < 65536 && sbytes[1] < 65536 && sbytes[2] < 65536)
                {
                    lit_mode = 2;
                    lit_csize = total;
                }
            }
        }
    }
    if (lit_mode == 2)
        lit_hdr = lit_streams == 1 ? 3u : (nlit < 1024 && lit_csize < 1024 ? 3u : nlit < 16384 && lit_csize < 16384 ? 4u : 5u);
    else
        lit_hdr = nlit < 32 ? 1u : nlit < 4096 ? 2u : 3u;
    const uint32_t lit_total = lit_hdr + (lit_mode == 2 ? lit_csize : lit_mode == 1 ? 1u : nlit);

    /* Huffman streams are packed now (the shared-memory tables are reused by the sequence
     * phase); the body is zeroed up to a safe bound first */
    uint32_t body_cap = lit_total + 16u;    /* grows once the sequence section is planned */

    if (lit_total + 3 >= len && nseq == 0)
        return R;                           /* no gain possible: raw block */
    /* zero [0, lit_total + 8) of the body */
    for (uint32_t i = lane; i < (lit_total + 8u + 3u) / 4u; i += 32)
        ow[i] = 0;
    __threadfence_block();
    __syncwarp();
    if (lit_mode == 2)
    {
        /* header: type 2 | size_format << 2 | regen << 4 | csize << (4 + nbits) */
        if (lane == 0)
        {
            uint64_t h;

            if (lit_streams == 1)
                h = 2u | (0u << 2) | ((uint64_t) nlit << 4) | ((uint64_t) lit_csize << 14);
            else if (lit_hdr == 3)
                h = 2u | (1u << 2) | ((uint64_t) nlit << 4) | ((uint64_t) lit_csize << 14);
            else if (lit_hdr == 4)
                h = 2u | (2u << 2) | ((uint64_t) nlit << 4) | ((uint64_t) lit_csize << 18);
            else
                h = 2u | (3u << 2) | ((uint64_t) nlit << 4) | ((uint64_t) lit_csize << 22);
            for (uint32_t i = 0; i < lit_hdr; i++)
                zse_put_byte(ow, i, (uint32_t) (h >> (8 * i)));
            for (uint32_t i = 0; i < desc_size; i++)
                zse_put_byte(ow, lit_hdr + i, hdesc[i]);
            if (lit_streams == 4)
                for (uint32_t k = 0; k < 3; k++)
                {
                    zse_put_byte(ow, lit_hdr + desc_size + 2 * k, sbytes[k]);
                    zse_put_byte(ow, lit_hdr + desc_size + 2 * k + 1, sbytes[k] >> 8);
                }
        }
        uint32_t at = lit_hdr + desc_size + (lit_streams == 4 ? 6u : 0u);

        for (uint32_t k = 0; k < lit_streams; k++)
        {
            uint32_t lo = lit_streams == 4 ? k * seg : 0u;
            uint32_t cnt = lit_streams == 4 ? (k < 3 ? seg : nlit - 3 * seg) : nlit;

            zse_huf_pack(lit, lo, cnt, hcode, ow, at, sbits[k], lane);
            at += sbytes[k];
        }
    }
    else
    {
        if (lane == 0)
        {
            uint32_t t = lit_mode;          /* 0 raw, 1 RLE */
            uint32_t h = lit_hdr == 1 ? (t | (nlit << 3)) : lit_hdr == 2 ? (t | (1u << 2) | (nlit << 4))
                                                                       : (t | (3u << 2) | (nlit << 4));

            for (uint32_t i = 0; i < lit_hdr; i++)
                zse_put_byte(ow, i, h >> (8 * i));
            if (lit_mode == 1)
                zse_put_byte(ow, lit_hdr, lit[0]);
        }
        /* raw literal bytes are copied at the very end (plain stores) */
    }
    __syncwarp();

    /* ================= sequences section ================= */
    uint32_t *qhist = reinterpret_cast<uint32_t *>(smem + ZQ_HIST);
    int16_t  *qnorm = reinterpret_cast<int16_t *>(smem + ZQ_NORM);
    uint16_t *qcum = reinterpret_cast<uint16_t *>(smem + ZQ_CUM);
    uint16_t *qenc[3] = {reinterpret_cast<uint16_t *>(smem + ZQ_ENC_LL),
                         reinterpret_cast<uint16_t *>(smem + ZQ_ENC_OF),
                         reinterpret_cast<uint16_t *>(smem + ZQ_ENC_ML)};
    uint8_t  *qdesc = smem + ZQ_DESC;
    uint32_t  seq_hdr = nseq < 128 ? 1u : nseq < 0x7F00u ? 2u : 3u;
    uint32_t  mode[3] = {0, 0, 0}, dsz[3] = {0, 0, 0};
    int       qlog[3] = {0, 0, 0};
    uint32_t  init_state[3] = {0, 0, 0};
    uint32_t  seq_bits = 0;

    if (nseq)
    {
        /* repeat offsets: history starts unknown (0 never matches a real offset) */
        uint32_t r0 = 0, r1 = 0, r2 = 0;

        for (uint32_t i = lane; i < 3 * 64; i += 32)
            qhist[i] = 0;
        __syncwarp();
        for (uint32_t c0 = 0; c0 < nseq; c0 += 32)
        {
            const uint32_t i = c0 + lane;
            uint4    q = make_uint4(0, 1, 0, 0);

            if (i < nseq)
                q = seq[i];
            const uint32_t my_ll = q.x & 0xFFFFu, my_off = q.y;
            uint32_t my_ofv = 0;
            const uint32_t cnt = nseq - c0 < 32 ? nseq - c0 : 32u;

            for (uint32_t k = 0; k < cnt; k++)
            {
                const uint32_t o = __shfl_sync(CRYO_FULL, my_off, (int) k);
                const uint32_t l = __shfl_sync(CRYO_FULL, my_ll, (int) k);
                uint32_t v;

                if (l)
                {
                    if (o == r0)
                        v = 1;
                    else if (o == r1)
                    {
                        v = 2;
                        r1 = r0;
                        r0 = o;
                    }
                    else if (o == r2)
                    {
                        v = 3;
                        r2 = r1;
                        r1 = r0;
                        r0 = o;
                    }
                    else
                    {
                        v = o + 3;
                        r2 = r1;
                        r1 = r0;
                        r0 = o;
                    }
                }
                else
                {
                    if (o == r1)
                    {
                        v = 1;
                        r1 = r0;
                        r0 = o;
                    }
                    else if (o == r2)
                    {
                        v = 2;
                        r2 = r1;
                        r1 = r0;
                        r0 = o;
                    }
                    else if (r0 > 1 && o == r0 - 1)
                    {
                        v = 3;
                        r2 = r1;
                        r1 = r0;
                        r0 = o;
                    }
                    else
                    {
                        v = o + 3;
                        r2 = r1;
                        r1 = r0;
                        r0 = o;
                    }
                }
                if (k == lane)
                    my_ofv = v;
            }
            if (i < nseq)
            {
                const uint32_t llc = zse_ll_code(my_ll), mlc = zse_ml_code((q.x >> 16) + 3u);
                const uint32_t ofc = (uint32_t) zs_highbit(my_ofv);

                q.y = my_ofv | (ofc << 24);
                q.z = llc | (mlc << 8);
                q.w = 0;
                seq[i] = q;
                atomicAdd(qhist + llc, 1u);
                atomicAdd(qhist + 64 + ofc, 1u);
                atomicAdd(qhist + 128 + mlc, 1u);
            }
        }
        __threadfence_block();
        __syncwarp();

        /* per table (lane t = table t): mode, normalised counts, description */
        uint32_t my_mode = 0, my_dsz = 0, my_cost = 0;
        int      my_log = 0;

        if (lane < 3)
        {
            const int       t = (int) lane;
            const uint32_t *h = qhist + 64 * t;
            int16_t        *nm = qnorm + 64 * t;
            const int       nsym_max = t == 0 ? 36 : t == 1 ? 32 : 53;
            const int       maxlog = t == 1 ? 8 : 9;
            const int16_t  *def = t == 0 ? ZS_LL_DEFAULT : t == 1 ? ZS_OF_DEFAULT : ZS_ML_DEFAULT;
            const int       deflog = t == 1 ? 5 : 6, defn = t == 0 ? 36 : t == 1 ? 29 : 53;
            int             top = -1, distinct = 0;

            for (int s = 0; s < nsym_max; s++)
                if (h[s])
                {
                    top = s;
                    distinct++;
                }
            if (distinct == 1)
            {
                my_mode = 1;                /* RLE: one byte, no state bits */
                qdesc[96 * t] = (uint8_t) top;
                my_dsz = 1;
                my_log = 0;
                for (int s = 0; s < 64; s++)
                    nm[s] = 0;
                nm[top] = 1;
            }
            else
            {
                /* predefined, if every used symbol exists in the default distribution */
                uint32_t cost_def = 0xFFFFFFFFu;

                if (top < defn)
                {
                    uint64_t c = 0;

                    for (int s = 0; s <= top; s++)
                        if (h[s])
                            c += (uint64_t) h[s] * (((uint32_t) deflog << 8) -
                                                    zse_log2_fp(def[s] < 0 ? 1u : (uint32_t) def[s]));
                    cost_def = (uint32_t) ((c + 255) >> 8);
                }
                /* FSE_optimalTableLog */
                int log = maxlog;
                int srcbits = zs_highbit(nseq - 1) - 2;
                int minbits = zs_highbit(nseq) + 1;
                int symbits = zs_highbit((uint32_t) top) + 2;

                if (symbits < minbits)
                    minbits = symbits;
                if (srcbits < log)
                    log = srcbits;
                if (minbits > log)
                    log = minbits;
                if (log < 5)
                    log = 5;
                if (log > maxlog)
                    log = maxlog;
                zse_fse_normalize(h, top + 1, nseq, log, nm);
                for (int s = top + 1; s < 64; s++)
                    nm[s] = 0;
                uint32_t nb = zse_fse_write_ncount(nm, top + 1, log, qdesc + 96 * t);
                uint32_t cost_fse = nb * 8u + zse_fse_cost_bits(h, nm, top + 1, log);

                if (cost_def <= cost_fse)
                {
                    my_mode = 0;
                    my_dsz = 0;
                    my_log = deflog;
                    for (int s = 0; s < 64; s++)
                        nm[s] = s < defn ? def[s] : (int16_t) 0;
                    my_cost = cost_def;
                }
                else
                {
                    my_mode = 2;
                    my_dsz = nb;
                    my_log = log;
                    my_cost = cost_fse;
                }
            }
        }
        (void) my_cost;
        for (int t = 0; t < 3; t++)
        {
            mode[t] = __shfl_sync(CRYO_FULL, my_mode, t);
            dsz[t] = __shfl_sync(CRYO_FULL, my_dsz, t);
            qlog[t] = __shfl_sync(CRYO_FULL, my_log, t);
        }
        __syncwarp();
        for (int t = 0; t < 3; t++)
        {
            if (mode[t] == 1)
                continue;
            const int nsym = t == 0 ? 36 : t == 1 ? 32 : 53;

            zse_fse_build_enc(qnorm + 64 * t, nsym, qlog[t], qenc[t], qcum + 64 * t,
                              reinterpret_cast<uint32_t *>(smem + ZQ_CELL),
                              reinterpret_cast<uint16_t *>(smem + ZQ_NEXT),
                              reinterpret_cast<uint16_t *>(smem + ZQ_CUMW), lane);
        }
        /* the three FSE state chains, backwards, one lane per table */
        uint32_t my_init = 0;

        if (lane < 3 && my_mode != 1)
        {
            const int       t = (int) lane;
            const uint16_t *enc = reinterpret_cast<const uint16_t *>(
                smem + (t == 0 ? ZQ_ENC_LL : t == 1 ? ZQ_ENC_OF : ZQ_ENC_ML));
            const uint16_t *cum = qcum + 64 * t;
            const int16_t  *nm = qnorm + 64 * t;
            const int       log = my_log;
            uint16_t       *upd = reinterpret_cast<uint16_t *>(seq);   /* 8 u16 per sequence */
            const uint32_t  slot = t == 0 ? 6u : t == 1 ? 5u : 7u;      /* z.hi, w.lo, w.hi */
            uint32_t        zc = seq[nseq - 1].z;
            uint32_t        s = t == 0 ? (zc & 0xFFu) : t == 2 ? ((zc >> 8) & 0xFFu) : (seq[nseq - 1].y >> 24);
            uint32_t        X = enc[cum[s]];

            for (int i = (int) nseq - 2; i >= 0; i--)
            {
                zc = seq[i].z;
                s = t == 0 ? (zc & 0xFFu) : t == 2 ? ((zc >> 8) & 0xFFu) : (seq[i].y >> 24);
                upd[8 * (size_t) i + slot] = (uint16_t) zse_fse_step(X, s, enc, cum, nm, log);
            }
            my_init = X;
        }
        for (int t = 0; t < 3; t++)
            init_state[t] = __shfl_sync(CRYO_FULL, my_init, t);
        __threadfence_block();
        __syncwarp();
        /* bit count of the interleaved stream */
        uint32_t bits = 0;

        for (uint32_t i = lane; i < nseq; i += 32)
        {
            const uint4 q = seq[i];
            const uint32_t llc = q.z & 0xFFu, mlc = (q.z >> 8) & 0xFFu, ofc = q.y >> 24;

            bits += ZS_LL_BITS[llc] + ZS_ML_BITS[mlc] + ofc;
            if (i + 1 < nseq)
                bits += ((q.z >> 28) & 15u) + ((q.w >> 12) & 15u) + (q.w >> 28);
        }
        seq_bits = __reduce_add_sync(CRYO_FULL, bits) + (uint32_t) (qlog[0] + qlog[1] + qlog[2]) + 1u;
    }
    const uint32_t seq_total = seq_hdr + (nseq ? 1u + dsz[0] + dsz[1] + dsz[2] + (seq_bits + 7u) / 8u : 0u);
    const uint32_t body = lit_total + seq_total;

    (void) body_cap;
    if (body + 3u >= len || body > ZSE_BLOCK)
        return R;                           /* does not shrink: raw block */

    /* ================= write the sequences section ================= */
    for (uint32_t i = (lit_total + 8u + 3u) / 4u + lane; i < (body + 8u + 3u) / 4u; i += 32)
        ow[i] = 0;
    __threadfence_block();
    __syncwarp();
    if (lit_mode == 0)
    {
        /* raw literals: plain stores; the words they share with their neighbours are only
         * touched by byte-granular stores and atomics on other bytes */
        for (uint32_t i = lane; i < nlit; i += 32)
            reinterpret_cast<uint8_t *>(ow)[lit_hdr + i] = lit[i];
    }
    uint32_t at = lit_total;

    if (lane == 0)
    {
        if (nseq < 128)
            zse_put_byte(ow, at, nseq);
        else if (nseq < 0x7F00u)
        {
            zse_put_byte(ow, at, (nseq >> 8) + 128u);
            zse_put_byte(ow, at + 1, nseq);
        }
        else
        {
            zse_put_byte(ow, at, 255u);
            zse_put_byte(ow, at + 1, nseq - 0x7F00u);
            zse_put_byte(ow, at + 2, (nseq - 0x7F00u) >> 8);
        }
    }
    at += seq_hdr;
    if (nseq)
    {
        if (lane == 0)
        {
            zse_put_byte(ow, at, (mode[0] << 6) | (mode[1] << 4) | (mode[2] << 2));
            uint32_t a = at + 1;

            for (int t = 0; t < 3; t++)
                for (uint32_t i = 0; i < dsz[t]; i++)
                    zse_put_byte(ow, a++, qdesc[96 * t + i]);
        }
        at += 1 + dsz[0] + dsz[1] + dsz[2];
        /* bitstream: sequence nseq-1 lowest, then nseq-2 ... 0, then ML/OF/LL initial states */
        uint32_t base = at * 8u;

        for (uint32_t c0 = 0; c0 < nseq; c0 += 32)
        {
            const uint32_t j = c0 + lane;               /* j-th sequence from the end */
            uint32_t mine = 0;
            uint4    q = make_uint4(0, 0, 0, 0);
            uint32_t llc = 0, mlc = 0, ofc = 0;
            bool     has_upd = false;

            if (j < nseq)
            {
                const uint32_t i = nseq - 1 - j;

                q = seq[i];
                llc = q.z & 0xFFu;
                mlc = (q.z >> 8) & 0xFFu;
                ofc = q.y >> 24;
                has_upd = i + 1 < nseq;
                mine = ZS_LL_BITS[llc] + ZS_ML_BITS[mlc] + ofc;
                if (has_upd)
                    mine += ((q.z >> 28) & 15u) + ((q.w >> 12) & 15u) + (q.w >> 28);
            }
            const uint32_t incl = zse_scan_incl(mine, lane);
            uint32_t pos = base + incl - mine;

            if (j < nseq)
            {
                if (has_upd)
                {
                    const uint32_t uo = q.z >> 16, ul = q.w & 0xFFFFu, um = q.w >> 16;

                    zse_put(ow, pos, uo & 0xFFFu, uo >> 12);
                    pos += uo >> 12;
                    zse_put(ow, pos, um & 0xFFFu, um >> 12);
                    pos += um >> 12;
                    zse_put(ow, pos, ul & 0xFFFu, ul >> 12);
                    pos += ul >> 12;
                }
                const uint32_t ll = q.x & 0xFFFFu, ml = (q.x >> 16) + 3u, ofv = q.y & 0xFFFFFFu;

                zse_put(ow, pos, ll - ZS_LL_BASE[llc], ZS_LL_BITS[llc]);
                pos += ZS_LL_BITS[llc];
                zse_put(ow, pos, ml - ZS_ML_BASE[mlc], ZS_ML_BITS[mlc]);
                pos += ZS_ML_BITS[mlc];
                zse_put(ow, pos, ofv - (1u << ofc), ofc);
            }
            base += __shfl_sync(CRYO_FULL, incl, 31);
        }
        if (lane == 0)
        {
            zse_put(ow, base, init_state[2], (uint32_t) qlog[2]);
            base += (uint32_t) qlog[2];
            zse_put(ow, base, init_state[1], (uint32_t) qlog[1]);
            base += (uint32_t) qlog[1];
            zse_put(ow, base, init_state[0], (uint32_t) qlog[0]);
            base += (uint32_t) qlog[0];
            zse_put(ow, base, 1u, 1u);
        }
    }
    __threadfence_block();
    __syncwarp();
    R.type = 2;
    R.size = body;
    return R;
}

/* ---- frames ------------------------------------------------------------------------ */

/* bytes of the frame header for a content size of n (single segment, content size field of 1 / 2 / 4 bytes) */
CRYO_DEV uint32_t zse_frame_header_size(uint32_t n)
{
    return n < 256u ? 6u : n < 65536u + 256u ? 7u : 9u;
}

/* overlap-safe move of n bytes to a LOWER address by one warp: 512 bytes per step, read before written */
CRYO_DEV void zse_move_down(uint8_t *dst, const uint8_t *src, uint32_t n, uint32_t lane)
{
    if (dst == src)
        return;
    for (uint32_t i0 = 0; i0 < n; i0 += 512u)
    {
        uint8_t v[16];

#pragma unroll
        for (uint32_t q = 0; q < 16; q++)
            v[q] = i0 + 32u * q + lane < n ? src[i0 + 32u * q + lane] : (uint8_t) 0;
        __syncwarp();
#pragma unroll
        for (uint32_t q = 0; q < 16; q++)
            if (i0 + 32u * q + lane < n)
                dst[i0 + 32u * q + lane] = v[q];
        __syncwarp();
    }
}

/*
 * The encoder's work loop, one warp.  Work items are (frame, 64 KiB block) pairs handed out in order from a
 * queue in global memory.  A block is written where it would start if every block before it were stored Raw
 * (frame header + b x (64 KiB + 3): inside cryogpu_compress_bound); the warp that finishes the last block of
 * a frame writes the frame header and closes the gaps, moving the blocks down in order.  With one CTA per
 * frame (round 1) fourteen warps waited at a barrier for the two whose blocks hold the tuples of a sparse
 * cryo block (84 % of the stall samples, profiles/r01g_other_kernels_ncu_summary.txt); here they take blocks
 * of the next frames instead.
 *   queue[0]: next item; done[f]: finished blocks of frame f (zeroed by the caller); bmeta[f * ZSE_MAXBLK + b]:
 *   bytes of block b with its header; scr: this warp's ZSE_SCR_PER_WARP bytes of global scratch; smem: this
 *   warp's ZSE_PER_WARP bytes.
 */
#define ZSE_MAXBLK 2048u                /* block_size <= 128 MiB */

CRYO_DEV void zstd_encode_worker(const uint8_t *src, uint64_t src_stride, uint32_t n, uint8_t *dst, uint64_t dst_stride,
                                 uint32_t dst_cap, int level, uint32_t *dst_size, int32_t *status, uint8_t *scr,
                                 uint32_t nframes, uint32_t *queue, uint32_t *done, uint32_t *bmeta, uint8_t *smem,
                                 uint32_t lane)
{
    const ZseParams P = zse_params(level);
    const uint32_t nblk = n ? (n + ZSE_BLOCK - 1) / ZSE_BLOCK : 1u, hdr = zse_frame_header_size(n);
    const uint64_t items = (uint64_t) nframes * nblk;
    const bool     fits = dst_cap >= 16u && (uint64_t) hdr + (uint64_t) n + 3ull * nblk <= dst_cap;

    for (;;)
    {
        uint32_t w = 0;

        if (lane == 0)
            w = atomicAdd(queue, 1u);
        w = __shfl_sync(CRYO_FULL, w, 0);
        if (w >= items)
            return;
        const uint32_t f = w / nblk, b = w % nblk;
        const uint8_t *fsrc = src + f * src_stride;
        uint8_t       *fdst = dst + f * dst_stride;
        const uint32_t lo = b * ZSE_BLOCK, len = n - lo < ZSE_BLOCK ? n - lo : ZSE_BLOCK;

        if (fits)
        {
            const ZseBlockOut R = zse_block(fsrc + lo, len, P, smem, scr, lane);
            uint8_t       *d = fdst + hdr + (size_t) b * (ZSE_BLOCK + 3u);
            const uint32_t last = b + 1 == nblk ? 1u : 0u;
            const uint32_t hsize = R.type == 2 ? R.size : len;
            const uint32_t h = last | (R.type << 1) | (hsize << 3);
            const uint32_t bytes = 3u + (R.type == 1 ? 1u : R.type == 0 ? len : R.size);

            if (lane < 3)
                d[lane] = (uint8_t) (h >> (8 * lane));
            if (R.type == 0)
                team_copy(d + 3, fsrc + lo, len, lane, 32);
            else if (R.type == 1)
            {
                if (lane == 0)
                    d[3] = (uint8_t) R.byte;
            }
            else
                team_copy(d + 3, scr + ZSE_SCR_OUT, R.size, lane, 32);
            if (lane == 0)
                bmeta[(size_t) f * ZSE_MAXBLK + b] = bytes;
        }
        __syncwarp();
        __threadfence();                /* the block and its size before the count */
        uint32_t fin = 0;

        if (lane == 0)
            fin = atomicAdd(done + f, 1u);
        fin = __shfl_sync(CRYO_FULL, fin, 0);
        if (fin != nblk - 1u)
            continue;
        __threadfence();                /* ... and the other warps' after it */
        if (!fits)
        {
            if (lane == 0)
            {
                dst_size[f] = 0;
                status[f] = ST_OUTPUT;
            }
            continue;
        }
        /* frame header: magic, descriptor (single segment, content size), content size */
        if (lane == 0)
        {
            uint32_t o = 0;

            fdst[o++] = 0x28;
            fdst[o++] = 0xB5;
            fdst[o++] = 0x2F;
            fdst[o++] = 0xFD;
            if (n < 256)
            {
                fdst[o++] = 0x20;
                fdst[o++] = (uint8_t) n;
            }
            else if (n < 65536 + 256)
            {
                fdst[o++] = 0x60;
                fdst[o++] = (uint8_t) (n - 256);
                fdst[o++] = (uint8_t) ((n - 256) >> 8);
            }
            else
            {
                fdst[o++] = 0xA0;
                fdst[o++] = (uint8_t) n;
                fdst[o++] = (uint8_t) (n >> 8);
                fdst[o++] = (uint8_t) (n >> 16);
                fdst[o++] = (uint8_t) (n >> 24);
            }
        }
        uint32_t pos = hdr;

        for (uint32_t k = 0; k < nblk; k++)
        {
            const uint32_t bytes = bmeta[(size_t) f * ZSE_MAXBLK + k];

            zse_move_down(fdst + pos, fdst + hdr + (size_t) k * (ZSE_BLOCK + 3u), bytes, lane);
            pos += bytes;
        }
        if (lane == 0)
        {
            dst_size[f] = pos;
            status[f] = ST_OK;
        }
    }
}
