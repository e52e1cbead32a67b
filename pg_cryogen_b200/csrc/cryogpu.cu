/*
 * cryogpu.cu -- C ABI of libcryogpu.so (include/cryogpu.h) and the sm_100a kernel
 * entry points.  Host side: lazy per-device context, pinned staging, chunked
 * H2D / kernel / D2H pipelines for the *_host calls, block-range sharding over
 * several GPUs.  No CPU codec lives here: every byte of LZ4 / zstd work is done
 * by the kernels in lz4_decode_w/c.cuh, zstd_decode_w/p/c.cuh, lz4_encode.cuh and
 * zstd_encode.cuh.
 */
#include "../../include/cryogpu.h"

#include "lz4_decode_w.cuh"
#include "lz4_decode_c.cuh"
#include "zstd_decode_w.cuh"
#include "zstd_decode_p.cuh"
#include "zstd_decode_c.cuh"
#include "lz4_encode.cuh"
#include "zstd_encode.cuh"
#include "cryo_pages.cuh"
#include "cryo_tuples.cuh"

#include <cuda_runtime.h>

#if defined(__x86_64__) || defined(_M_X64)
#include <emmintrin.h>
#define CRYO_HAVE_SSE2 1
#endif

#include <sys/mman.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <functional>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

/* ------------------------------------------------------------------ errors */

static thread_local char g_err[512] = "";

static int
fail(int code, const char *fmt, ...)
{
    va_list ap;

    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CU(call)                                                                         \
    do {                                                                                 \
        cudaError_t e_ = (call);                                                         \
        if (e_ != cudaSuccess)                                                           \
            return fail(CRYOGPU_E_CUDA, "%s: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                        __FILE__, __LINE__);                                             \
    } while (0)

/* ----------------------------------------------------------------- kernels */

/* development aid (-DZP_TIMELINE): every pipeline kernel records the first CTA start and the last CTA
 * end on the GPU's global timer, printed by cryogpu_decompress_device when CRYOGPU_ZP_TIMELINE is set */
#ifdef ZP_TIMELINE
__device__ unsigned long long zp_tl[32];
#define ZP_TL_BEGIN(k)                                                                  \
    if (threadIdx.x == 0)                                                               \
    {                                                                                   \
        unsigned long long t_;                                                          \
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));                          \
        atomicMin(&zp_tl[2 * (k)], t_);                                                 \
    }
#define ZP_TL_END(k)                                                                    \
    __syncthreads();                                                                    \
    if (threadIdx.x == 0)                                                               \
    {                                                                                   \
        unsigned long long t_;                                                          \
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));                          \
        atomicMax(&zp_tl[2 * (k) + 1], t_);                                             \
    }
#else
#define ZP_TL_BEGIN(k)
#define ZP_TL_END(k)
#endif

/* sequences after which the one-warp-per-block LZ4 decoder hands a block to the CTA decoder (lz4_decode_w.cuh) */
#define LZ4W_BUDGET 3072u

/* latency path and match-rich blocks: one CTA per block, persistent CTAs take the routed blocks in order */
__global__ void __launch_bounds__(CX_THREADS, 1)
k_lz4_decode_c(const int32_t *methods, const uint8_t *src, const uint64_t *src_off,
               const uint32_t *src_size, uint8_t *dst, uint64_t dst_stride, uint32_t cap,
               uint32_t *out_size, int32_t *status, uint32_t n, const uint32_t *list,
               uint32_t *counter, unsigned long long *gseq)
{
    __shared__ uint32_t next_b;

    ZP_TL_BEGIN(10)
    for (;;)
    {
        __syncthreads();
        if (threadIdx.x == 0)
            next_b = atomicAdd(counter, 1u);
        __syncthreads();
        /* list: the blocks the warp decoder gave up (counter[1] of them); without it every LZ4 block of the batch */
        if (next_b >= (list ? counter[1] : n))
        {
            ZP_TL_END(10)
            return;
        }
        const uint32_t b = list ? list[next_b] : next_b;

        if (methods[b] != CRYOGPU_LZ4)
            continue;
        lz4c_decode_block(src + src_off[b], src_size[b], dst + b * dst_stride, cap, out_size + b, status + b,
                          CRYO_SMEM_BASE(), gseq + (size_t) blockIdx.x * LZ4C_SEQCAP, threadIdx.x);
    }
}

/* throughput path: one warp per block, LZ4W_WARPS blocks per CTA */
__global__ void __launch_bounds__(LZ4W_THREADS)
k_lz4_decode_w(const int32_t *methods, const uint8_t *src, const uint64_t *src_off,
               const uint32_t *src_size, uint8_t *dst, uint64_t dst_stride, uint32_t cap,
               uint32_t *out_size, int32_t *status, uint32_t n, uint32_t *list, uint32_t *count)
{
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t b = blockIdx.x * LZ4W_WARPS + warp;

    ZP_TL_BEGIN(9)
    if (b >= n || methods[b] != CRYOGPU_LZ4)
        return;
    /* list: where the blocks with too many sequences for one warp are queued for k_lz4_decode_c */
    if (lz4w_decode_block(src + src_off[b], src_size[b], dst + b * dst_stride, cap, out_size + b,
                          status + b, CRYO_SMEM_BASE() + warp * LZ4W_PER_WARP, lane,
                          list && cap <= LZ4C_MAXCAP ? LZ4W_BUDGET : 0u) && lane == 0)
        list[atomicAdd(count, 1u)] = b;
}

/* throughput path (default): one warp per frame, ZSW_WARPS frames per CTA */
__global__ void __launch_bounds__(ZSW_THREADS, ZSW_CTAS_PER_SM)
k_zstd_decode_w(const int32_t *methods, const uint8_t *src, const uint64_t *src_off,
                const uint32_t *src_size, uint8_t *dst, uint64_t dst_stride, uint32_t cap,
                uint32_t *out_size, int32_t *status, uint8_t *scratch, uint64_t scratch_stride,
                const uint32_t *predef, uint32_t n, const uint32_t *only)
{
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t b = blockIdx.x * ZSW_WARPS + warp;

    ZP_TL_BEGIN(12)
    if (b >= n || methods[b] != CRYOGPU_ZSTD || (only && only[b] == 0))
        return;
    zstdw_decode_frame(src + src_off[b], src_size[b], dst + b * dst_stride, cap, out_size + b,
                       status + b, scratch + b * scratch_stride, predef,
                       CRYO_SMEM_BASE() + warp * ZSW_PER_WARP, lane);
}

/* defaults of the pipeline's knobs (each has an environment override, see launch_zstd_decode) */
#ifndef ZP_L2HINT_DEFAULT
#define ZP_L2HINT_DEFAULT 1
#endif
#ifndef ZP_EXEC_PREFETCH_DEFAULT
#define ZP_EXEC_PREFETCH_DEFAULT 0
#endif
#ifndef ZP_PF_INFLIGHT_DEFAULT
#define ZP_PF_INFLIGHT_DEFAULT 2        /* bulk groups (one per raw / RLE block) a CTA of the raw / RLE stage keeps in flight */
#endif
#ifndef ZP_EARLY_CTAS_DEFAULT
#define ZP_EARLY_CTAS_DEFAULT (-1)      /* CTAs of the early pass of the raw / RLE stage (-1: one per SM, 0: no early pass) */
#endif
#ifndef ZP_EARLY_PCT_DEFAULT
#define ZP_EARLY_PCT_DEFAULT 55         /* share of the batch's frames it takes, from the end */
#endif

/* phase-split pipeline (default zstd path): zstd_decode_p.cuh */
__global__ void __launch_bounds__(32)
k_zp_parse(const ZpArgs a)
{
    ZP_TL_BEGIN(0)
    const uint32_t f = blockIdx.x * 32u + threadIdx.x;

    /*
     * The warp's frames are asked into L2 first (the first 32 KiB of each: a sparse or medium frame whole), line by
     * line across the lanes.  Everything after this reads them piecemeal -- the walk from block header to block
     * header below, the table descriptions, the 256-byte window refills of the lane-serial stages -- and each piece
     * that has to come from HBM stalls a chain (pf_hint bit 4; CRYOGPU_ZP_SRC_PREFETCH=0: off).
     */
    if (a.pf_hint & 16u)
    {
        const bool     mine = f < a.n && a.methods[f] == ZP_METHOD_ZSTD;
        const uint64_t my_off = mine ? a.src_off[f] : 0;
        const uint32_t my_size = mine ? a.src_size[f] : 0;

        for (uint32_t t = 0; t < 32u; t++)
        {
            const uint64_t off = __shfl_sync(CRYO_FULL, my_off, (int) t);
            const uint32_t size = min(__shfl_sync(CRYO_FULL, my_size, (int) t), 32768u);

            for (uint32_t o = 128u * threadIdx.x; o < size; o += 4096u)
                asm volatile("prefetch.global.L2 [%0];" ::"l"(a.src + off + o));
        }
    }
    if (f < a.n)
        zp_stage1(a, f);
    ZP_TL_END(0)
}

/* bulk-copy engine (TMA) helpers for the raw / RLE stage: shared -> global, completion by bulk groups */
#define ZP0_CHUNK 16384u

__device__ __forceinline__ void
zp0_bulk_store(uint8_t *dst, const uint8_t *smem_src, uint32_t bytes)
{
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                 ::"l"(dst), "r"((uint32_t) __cvta_generic_to_shared(smem_src)), "r"(bytes) : "memory");
}

/* the same with an L2 policy: the zero runs stream through, the literals and sequences the
 * executor is reading at the same time should stay */
__device__ __forceinline__ void
zp0_bulk_store_hint(uint8_t *dst, const uint8_t *smem_src, uint32_t bytes, uint64_t policy)
{
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;"
                 ::"l"(dst), "r"((uint32_t) __cvta_generic_to_shared(smem_src)), "r"(bytes), "l"(policy) : "memory");
}

#define ZP0_THREADS 128u                /* few registers beside the executor's three CTAs per SM */

/* wait until at most k of the thread's bulk groups are pending (the instruction takes an immediate) */
__device__ __forceinline__ void
zp0_wait_pending(uint32_t k)
{
    switch (k)
    {
        case 0: asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); break;
        case 1: asm volatile("cp.async.bulk.wait_group 1;" ::: "memory"); break;
        case 2: asm volatile("cp.async.bulk.wait_group 2;" ::: "memory"); break;
        case 3: asm volatile("cp.async.bulk.wait_group 3;" ::: "memory"); break;
        case 4: asm volatile("cp.async.bulk.wait_group 4;" ::: "memory"); break;
        case 5: asm volatile("cp.async.bulk.wait_group 5;" ::: "memory"); break;
        case 6: asm volatile("cp.async.bulk.wait_group 6;" ::: "memory"); break;
        case 7: asm volatile("cp.async.bulk.wait_group 7;" ::: "memory"); break;
        default: asm volatile("cp.async.bulk.wait_group 8;" ::: "memory"); break;
    }
}

/*
 * The raw / RLE stage.  Persistent, one CTA per SM.  Its unit of work is a run of one byte -- an RLE block (the zero
 * runs of sparse cryo blocks: 73 % of the headline table's bytes), or a long run stage 4 hands over (ZP_JOBS: another
 * 24 %) -- written by the bulk-copy engine: a 16 KiB pattern in shared memory, one elected thread issuing cp.async.bulk
 * stores of it, no LSU or register traffic on an SM that is executing sequences at the same time.  One bulk group per
 * unit, a.pf_inflight of them in flight; a unit is published (pf_done of its frame) when its group has completed.
 * Raw blocks and unaligned edges go through ordinary stores.
 */
struct Zp0
{
    uint8_t  *pat;              /* shared: ZP0_CHUNK bytes of the current byte */
    int       cur;              /* that byte, -1: none yet */
    uint32_t  window;           /* groups in flight */
    uint32_t  issued, published;        /* units committed / published (thread 0) */
    uint32_t  ticket;           /* number of the job this lane of warp 0 is waiting for, ~0u: none taken */
    uint32_t  ring[8];          /* the units not yet published: a block's frame, or 1 << 31 | a job's slot (thread 0) */
};

/* n bytes of `byte` at dst (every thread of the CTA calls this with the same arguments); the unit belongs to frame f */
__device__ __forceinline__ void
zp0_unit_fill(const ZpArgs &a, Zp0 &z, uint8_t *dst, uint32_t n, int byte)
{
    if (byte != z.cur)
    {
        /* new pattern: the engine must have read the old one out first (every store so far is in a committed group) */
        if (threadIdx.x == 0)
            asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        __syncthreads();
        const uint32_t w = (uint32_t) byte * 0x01010101u;

        for (uint32_t k = threadIdx.x; k < ZP0_CHUNK / 16u; k += ZP0_THREADS)
            reinterpret_cast<uint4 *>(z.pat)[k] = make_uint4(w, w, w, w);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        z.cur = byte;
    }
    /* edges by hand, the 16-byte aligned body by the engine */
    const uint32_t head = (16u - (uint32_t) ((uintptr_t) dst & 15u)) & 15u;
    const uint32_t h = head < n ? head : n, body = (n - h) & ~15u, tail = n - h - body;

    if (threadIdx.x < h)
        dst[threadIdx.x] = (uint8_t) byte;
    if (threadIdx.x < tail)
        dst[h + body + threadIdx.x] = (uint8_t) byte;
    if (threadIdx.x < h || threadIdx.x < tail)
        __threadfence();                /* ordinary stores: fenced before the barrier in front of the unit's publication */
    if (threadIdx.x == 0)
    {
        if (a.pf_hint & 1u)
        {
            uint64_t policy;

            asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
            for (uint32_t o = 0; o < body; o += ZP0_CHUNK)
                zp0_bulk_store_hint(dst + h + o, z.pat, body - o < ZP0_CHUNK ? body - o : ZP0_CHUNK, policy);
        }
        else
            for (uint32_t o = 0; o < body; o += ZP0_CHUNK)
                zp0_bulk_store(dst + h + o, z.pat, body - o < ZP0_CHUNK ? body - o : ZP0_CHUNK);
    }
}

/* the unit just written (bulk stores issued by thread 0, ordinary stores fenced) is committed; units whose groups have
 * completed are published.  publish = false: the early pass (nobody waits for its blocks: the kernel's end says it all) */
__device__ __forceinline__ void
zp0_unit_done(const ZpArgs &a, Zp0 &z, uint32_t f, bool publish, bool drain)
{
    __syncthreads();                    /* every thread's ordinary stores of the unit, fenced, before its publication */
    if (threadIdx.x != 0)
        return;
    if (!drain)
    {
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        z.ring[z.issued & 7u] = f;
        z.issued++;
    }
    zp0_wait_pending(drain ? 0u : z.window - 1u);
    const uint32_t complete = drain ? z.issued : (z.issued >= z.window - 1u ? z.issued - (z.window - 1u) : 0u);

    if (z.published < complete)
    {
        asm volatile("fence.proxy.async;" ::: "memory");
        for (; z.published < complete; z.published++)
        {
            const uint32_t unit = z.ring[z.published & 7u];

            if (!publish)
                continue;
            if (unit & 0x80000000u)
            {
                /* a job: done in its own slot (pf_done counts a frame's blocks, in block order) */
                __threadfence();
                atomicOr(a.jobs + 4u * (size_t) (unit & 0x7FFFFFFFu) + 3, ZP_JOB_DONE);
            }
            else
                zp_stage0_done(a, unit << 8, 1u);
        }
    }
}

/*
 * Jobs of stage 4's, if the CTA's tickets have come up.  Jobs are numbered as they are queued; a ticket is a fetch-and-add
 * on the head (no two CTAs ever contend for a job -- claiming with compare-and-swap, 148 CTAs took 3.3 ms over the
 * step's 6 898 jobs).  A CTA holds ZP0_TAKE tickets, one per lane of warp 0, and looks at their slots side by side
 * whenever it passes here: a job is 120 KB, 2.6 us of the engine's time, and ticket + flag + fields are three dependent
 * round trips of 1-2 us each -- taken one job at a time they left the engine idle half the time.
 * Returns the number served; ~0u: none ever will be (stage 4 has finished and queued fewer).
 */
#define ZP0_TAKE 4u

__device__ __forceinline__ uint32_t
zp0_serve_jobs(const ZpArgs &a, Zp0 &z, uint32_t (*s_job)[5], uint32_t *s_over)
{
    uint32_t *ctl = reinterpret_cast<uint32_t *>(a.seq_alloc);

    __syncthreads();
    if (threadIdx.x < 32u)
    {
        bool over = true;

        if (threadIdx.x < ZP0_TAKE)
        {
            uint32_t w3 = 0;

            over = false;
            if (z.ticket == ~0u)
                z.ticket = atomicAdd(ctl + ZPC_JOB_HEAD, 1u);
            if (z.ticket < a.n * ZP_JOBS)
                w3 = zp_ld_acquire(a.jobs + 4u * (size_t) z.ticket + 3);
            if (!(w3 & ZP_JOB_READY) && zp_ld_acquire(ctl + ZPC_EXEC_DONE) >= a.exec_warps)
            {
                /* no more jobs will be queued: either ours is among them (its fields follow the slot's allocation at once) or not */
                if (z.ticket < zp_ld_acquire(ctl + ZPC_JOB_TAIL))
                    for (uint32_t spin = 0; spin < 200000u && !(w3 & ZP_JOB_READY); spin++)
                        w3 = zp_ld_acquire(a.jobs + 4u * (size_t) z.ticket + 3);
                else
                    over = true;
            }
            if (w3 & ZP_JOB_READY)
            {
                const uint32_t *job = a.jobs + 4u * (size_t) z.ticket;

                s_job[threadIdx.x][0] = job[0];
                s_job[threadIdx.x][1] = job[1];
                s_job[threadIdx.x][2] = job[2];
                s_job[threadIdx.x][4] = z.ticket;
                z.ticket = ~0u;
            }
            s_job[threadIdx.x][3] = w3;
        }
        over = __all_sync(CRYO_FULL, over);
        if (threadIdx.x == 0)
            *s_over = over ? 1u : 0u;
    }
    __syncthreads();
    uint32_t served = 0;

    for (uint32_t t = 0; t < ZP0_TAKE; t++)
    {
        if (!(s_job[t][3] & ZP_JOB_READY))
            continue;
        const uint32_t f = s_job[t][0];

        zp0_unit_fill(a, z, a.dst + (size_t) f * a.dst_stride + s_job[t][1], s_job[t][2], (int) (s_job[t][3] & 0xFFu));
        zp0_unit_done(a, z, 0x80000000u | s_job[t][4], true, false);
        served++;
    }
    return served ? served : (*s_over ? ~0u : 0u);
}

template <bool EARLY>
__device__ __forceinline__ void zp_prefill_body(const ZpArgs &a)
{
    __shared__ __align__(128) uint8_t pat[ZP0_CHUNK];
    __shared__ uint32_t spec[ZP_MAXB], s_len[ZP_MAXB], s_what[ZP_MAXB], s_off[ZP_MAXB];
    __shared__ uint32_t next_f, s_job[ZP0_TAKE][5], s_over;
    uint32_t *counter = reinterpret_cast<uint32_t *>(a.seq_alloc) + (EARLY ? 5 : 4);    /* zeroed with seq_alloc */
    Zp0       z;

    z.pat = pat;
    z.cur = -1;
    z.window = a.pf_inflight > 8u ? 8u : a.pf_inflight < 1u ? 1u : a.pf_inflight;
    z.issued = z.published = 0;
    z.ticket = ~0u;
    if (!EARLY && a.jobs && threadIdx.x == 0)
        atomicAdd(reinterpret_cast<uint32_t *>(a.seq_alloc) + ZPC_SERVERS, 1u);     /* stage 4 may queue jobs: somebody will take them */
    /*
     * Frames are handed out by a counter, not by blockIdx: the CTAs of this kernel do not all become resident at
     * once beside the executor's (in some states of the process a third of them start a millisecond late, and
     * with a fixed share of the frames each the stage then took 1.76 ms instead of 0.75, profiles/README.md); the
     * ones that are running take whatever is next.
     */
    for (;;)
    {
        __syncthreads();
        if (threadIdx.x == 0)
            next_f = atomicAdd(counter, 1u);
        __syncthreads();
        if (next_f >= (EARLY ? a.early_frames : a.n))
            break;
        /* the early pass works from the end of the batch, whose frames stage 4 reaches last */
        const uint32_t f = EARLY ? a.n - 1u - next_f : next_f;
        const uint32_t nb = a.fr[(size_t) f * ZP_FF];
        const uint8_t *in = a.src + a.src_off[f];
        uint8_t *out = a.dst + (size_t) f * a.dst_stride;

        if (threadIdx.x < 32u)
        {
            /* EARLY: guessed by stage 1; otherwise exact: stage 3b has measured the Compressed blocks */
            const uint32_t at = zp_frame_positions_warp<EARLY>(a, f, threadIdx.x);

            /* what the blocks are, side by side with their positions: read in the loop below, block after block, the
             * descriptor and then the frame's byte were two dependent round trips per block, 10 us of a sparse frame's 25 */
            if (threadIdx.x < ZP_MAXB)
            {
                const uint32_t *b = a.blk + ((size_t) f * ZP_MAXB + threadIdx.x) * ZP_BF;

                spec[threadIdx.x] = at;
                if (at != ~0u)
                {
                    s_len[threadIdx.x] = b[ZPB_BSIZE];
                    s_off[threadIdx.x] = b[ZPB_OFF];
                    s_what[threadIdx.x] = (b[ZPB_KIND] & 3u) == 0 ? ~0u : b[ZPB_RLEBYTE];   /* Raw, or the byte of the run */
                }
            }
        }
        __syncthreads();
        for (uint32_t j = 0; j < nb; j++)
        {
            if (spec[j] == ~0u)
                continue;
            if (s_what[j] == ~0u)
            {
                team_copy(out + spec[j], in + s_off[j], s_len[j], threadIdx.x, ZP0_THREADS);
                __threadfence();
            }
            else
                zp0_unit_fill(a, z, out + spec[j], s_len[j], (int) s_what[j]);
            zp0_unit_done(a, z, f, !EARLY, false);
        }
        /* (CRYOGPU_ZP_JOBS=2, pf_hint bit 5: a run stage 4 has handed over meanwhile after every frame, so that they do not
         * pile up behind the frames.  Measured no better, and less even from run to run: off) */
        if (!EARLY && a.jobs && (a.pf_hint & 32u))
            zp0_serve_jobs(a, z, s_job, &s_over);
    }
    if (!EARLY && a.jobs)
    {
        /* the frames are done: serve stage 4's runs until its warps have all finished and the queue is empty.  The wait is
         * bounded (about 50 ms); a run nobody served is noticed afterwards (zp_stage5_check) */
        /* (the bound: ~20 ms without a job.  Under a tool that runs kernels one after the other -- ncu, the sanitizer --
         * stage 4 has not even started: this stage then waits the bound out and the check sends the frames to the fallback) */
        uint32_t *ctl = reinterpret_cast<uint32_t *>(a.seq_alloc);
        __shared__ uint32_t s_up;

        if (z.window < ZP0_TAKE)
            z.window = ZP0_TAKE;        /* a round's jobs in flight together */
        /* stage 4 runs beside this kernel, or (under a profiler, a sanitizer) only after it: then nothing is to come */
        if (threadIdx.x == 0)
        {
            uint32_t up = 0;

            for (uint32_t spin = 0; spin < 400u && !up; spin++)
            {
                up = zp_ld_acquire(ctl + ZPC_EXEC_UP);
                if (!up)
                    __nanosleep(256);
            }
            s_up = up;
        }
        __syncthreads();
        for (uint32_t idle = s_up ? 0u : 20000u; idle < 20000u;)
        {
            const uint32_t r = zp0_serve_jobs(a, z, s_job, &s_over);

            if (r == ~0u)
                break;
            if (r)
            {
                idle = 0;
                continue;
            }
            __nanosleep(256);
            idle++;
        }
    }
    zp0_unit_done(a, z, 0, !EARLY, true);
    if (!EARLY && a.jobs && threadIdx.x == 0)
        atomicSub(reinterpret_cast<uint32_t *>(a.seq_alloc) + ZPC_SERVERS, 1u);
}

__global__ void __launch_bounds__(ZP0_THREADS)
k_zp_prefill(const ZpArgs a)
{
    ZP_TL_BEGIN(1)
#ifndef ZP_ABLATE_PREFILL       /* timing experiment only: the raw / RLE blocks are left to the executor's time-out */
    zp_prefill_body<false>(a);
#endif
    ZP_TL_END(1)
}

__global__ void __launch_bounds__(256)
k_zp_check(const ZpArgs a)
{
    zp_stage5_check(a, blockIdx.x * 256u + threadIdx.x);
}

/*
 * The same stage BEFORE the entropy stages have measured anything, beside them (they are bound by the latency of
 * their serial chains and leave HBM idle): every raw / RLE block at the position stage 1 guessed for it.  A guess
 * that turns out wrong costs nothing but the bytes: the late pass writes that block again where it belongs, and
 * every other byte of the frame's declared size is written by stage 4 after this kernel has ended.
 */
__global__ void __launch_bounds__(ZP0_THREADS)
k_zp_prefill_early(const ZpArgs a)
{
    ZP_TL_BEGIN(13)
    zp_prefill_body<true>(a);
    ZP_TL_END(13)
}


__global__ void __launch_bounds__(32 * ZP2A_WARPS)
k_zp_huftab(const ZpArgs a, uint32_t split)
{
    ZP_TL_BEGIN(2)
    ZP_FOR_GROUP_BLOCKS_CTA(a, blockIdx.x, split, ZPF_HUFMASK, threadIdx.x, zp_stage2a(a, g, j, CRYO_SMEM_BASE(), threadIdx.x));
    ZP_TL_END(2)
}

__global__ void __launch_bounds__(32)
k_zp_literals(const ZpArgs a, uint32_t split)
{
    ZP_TL_BEGIN(3)
    ZP_FOR_GROUP_BLOCKS(a, blockIdx.x, split, ZPF_HUFMASK, threadIdx.x, zp_stage2b(a, g, j, CRYO_SMEM_BASE(), threadIdx.x));
    ZP_TL_END(3)
}

__global__ void __launch_bounds__(32 * ZP3A_WARPS)
k_zp_fsetab(const ZpArgs a, uint32_t split)
{
    ZP_TL_BEGIN(4)
    ZP_FOR_GROUP_BLOCKS_CTA(a, blockIdx.x, split, ZPF_SEQMASK, threadIdx.x, zp_stage3a(a, g, j, CRYO_SMEM_BASE(), threadIdx.x));
    ZP_TL_END(4)
}

__global__ void __launch_bounds__(32)
k_zp_sequences_small(const ZpArgs a, uint32_t split)
{
    ZP_TL_BEGIN(5)
    ZP_FOR_GROUP_BLOCKS(a, blockIdx.x, split, ZPF_SEQMASK, threadIdx.x,
                        (zp_stage3b<ZP3B_SMALL, 0, ZP3B_SMALL_LANES>(a, g, j, CRYO_SMEM_BASE(), threadIdx.x)));
    ZP_TL_END(5)
}

__global__ void __launch_bounds__(32)
k_zp_sequences_large(const ZpArgs a, uint32_t split)
{
    ZP_TL_BEGIN(6)
    ZP_FOR_GROUP_BLOCKS(a, blockIdx.x, split, ZPF_SEQMASK, threadIdx.x,
                        (zp_stage3b<ZP3B_LARGE, ZP3B_SMALL, ZP_G>(a, g, j, CRYO_SMEM_BASE(), threadIdx.x)));
    ZP_TL_END(6)
}

#ifndef ZP4_MAXNREG
#define ZP4_MAXNREG 72
#endif
__global__ void __maxnreg__(ZP4_MAXNREG)
k_zp_execute(const ZpArgs a)
{
    ZP_TL_BEGIN(7)
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (a.jobs && threadIdx.x == 0)
        zp_st_release(reinterpret_cast<uint32_t *>(a.seq_alloc) + ZPC_EXEC_UP, 1u);
    zp_stage4(a, blockIdx.x * ZP4_WARPS + warp, CRYO_SMEM_BASE() + warp * ZP4_PER_WARP, lane);
    /* stage 0 serves the runs this kernel hands over until every warp of it has said it is done */
    if (a.jobs && lane == 0)
    {
        __threadfence();
        atomicAdd(reinterpret_cast<uint32_t *>(a.seq_alloc) + ZPC_EXEC_DONE, 1u);
    }
    ZP_TL_END(7)
}

/* stage 4 with one CTA per frame (zstd_decode_c.cuh): persistent CTAs take the frames stage 1 routed to them */
__global__ void __launch_bounds__(CX_THREADS, 1)
k_zp_execute_c(const ZpArgs a, uint32_t *counter)
{
    __shared__ uint32_t next_f;

    ZP_TL_BEGIN(11)
    for (;;)
    {
        __syncthreads();
        if (threadIdx.x == 0)
            next_f = atomicAdd(counter, 1u);
        __syncthreads();
        if (next_f >= *a.cxcount)
        {
            ZP_TL_END(11)
            return;
        }
        const uint32_t f = a.cxlist[next_f];

        if (a.flag[f] != 0 || a.fr[(size_t) f * ZP_FF] == 0)
            continue;                   /* a later stage declined the frame */
        zp_stage4_cx(a, f, CRYO_SMEM_BASE(), threadIdx.x);
    }
}

/* the three predefined FSE tables of RFC 8878 3.1.1.3.2.2, built once per context */
__global__ void
k_zstd_build_predef(uint32_t *predef)
{
    __shared__ __align__(16) uint8_t sm[2048];

    zsw_build_predef(predef, sm, threadIdx.x);
}

__global__ void
k_flag_unknown_methods(const int32_t *methods, size_t n, uint32_t *out_size, int32_t *status)
{
    size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x;

    if (i < n && methods[i] != CRYOGPU_LZ4 && methods[i] != CRYOGPU_ZSTD)
    {
        status[i] = CRYOGPU_ST_METHOD;      /* compression.c:157 "unknown compression method" */
        out_size[i] = 0;
    }
}

/* persistent: the warps of one CTA per SM take (block, segment) items from a queue (lz4_encode.cuh) */
__global__ void __launch_bounds__(LZ4E_THREADS)
k_lz4_encode(const uint8_t *src, uint64_t src_stride, uint32_t block_size, uint8_t *dst,
             uint64_t dst_stride, uint32_t dst_cap, int accel, uint32_t *dst_size,
             int32_t *status, uint8_t *scratch, uint64_t scratch_stride, uint32_t n, uint32_t *queue, uint32_t *done)
{
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    lz4_encode_worker(src, src_stride, block_size, dst, dst_stride, dst_cap, accel, dst_size, status, scratch,
                      scratch_stride, n, queue, done,
                      reinterpret_cast<uint16_t *>(CRYO_SMEM_BASE() + warp * LZ4E_HASH_BYTES), lane);
}

/* persistent: the warps of one CTA per SM take (frame, 64 KiB block) items from a queue (zstd_encode.cuh) */
__global__ void __launch_bounds__(ZSTDE_THREADS)
k_zstd_encode(const uint8_t *src, uint64_t src_stride, uint32_t block_size, uint8_t *dst,
              uint64_t dst_stride, uint32_t dst_cap, int level, uint32_t *dst_size,
              int32_t *status, uint8_t *scratch, uint64_t scratch_stride, uint32_t n, uint32_t *queue, uint32_t *done,
              uint32_t *bmeta)
{
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    zstd_encode_worker(src, src_stride, block_size, dst, dst_stride, dst_cap, level, dst_size, status,
                       scratch + blockIdx.x * scratch_stride + (size_t) warp * ZSE_SCR_PER_WARP, n, queue, done, bmeta,
                       CRYO_SMEM_BASE() + warp * ZSE_PER_WARP, lane);
}


/*
 * Sparse return for the host-pointer decompress call: a 1 MiB cryo block of narrow rows is
 * ~98 % zeros (SURVEY.md 0.1), and shipping zeros over PCIe is what bounds the host call.
 * One CTA per block marks which 4 KiB pages of the decoded block hold a non-zero byte and
 * packs those pages into a staging buffer; the host copies only them and zero-fills the rest
 * of the caller's block itself.  The chunk was just written, so this scan reads L2.
 */
#define SP_PAGE      4096u
#define SP_MAXPAGES  2048u          /* blocks up to 8 MiB */
#define SP_WORDS     (SP_MAXPAGES / 32u)

__global__ void __launch_bounds__(256)
k_page_compact(const uint8_t *out, uint64_t stride, uint32_t block_size, uint32_t *bitmap,
               uint32_t *page_off, uint32_t *counter, uint8_t *staging)
{
    __shared__ uint32_t flags[SP_WORDS];
    __shared__ uint32_t base_sh;
    const uint32_t b = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint8_t *blk = out + b * stride;
    const uint32_t pages = (block_size + SP_PAGE - 1) / SP_PAGE, words = (pages + 31) / 32;

    for (uint32_t i = tid; i < SP_WORDS; i += 256)
        flags[i] = 0;
    __syncthreads();
    for (uint32_t p = warp; p < pages; p += 8)
    {
        const uint32_t len = block_size - p * SP_PAGE < SP_PAGE ? block_size - p * SP_PAGE : SP_PAGE;
        bool nz = (len & 15u) != 0;         /* a ragged tail page is always shipped */

        if (!nz)
        {
            const uint4 *q = reinterpret_cast<const uint4 *>(blk + (size_t) p * SP_PAGE);
            uint32_t acc = 0;

            for (uint32_t v = lane; v < len / 16; v += 32)
            {
                uint4 x = q[v];

                acc |= x.x | x.y | x.z | x.w;
            }
            nz = __any_sync(0xffffffffu, acc != 0);
        }
        if (nz && lane == 0)
            atomicOr(&flags[p >> 5], 1u << (p & 31));
    }
    __syncthreads();
    if (tid == 0)
    {
        uint32_t c = 0;

        for (uint32_t w = 0; w < words; w++)
            c += (uint32_t) __popc(flags[w]);
        base_sh = atomicAdd(counter, c);
        page_off[b] = base_sh;
    }
    for (uint32_t w = tid; w < SP_WORDS; w += 256)
        bitmap[b * SP_WORDS + w] = w < words ? flags[w] : 0u;
    __syncthreads();
    const uint32_t base = base_sh;

    for (uint32_t p = warp; p < pages; p += 8)
    {
        if (!(flags[p >> 5] & (1u << (p & 31))))
            continue;
        uint32_t rank = (uint32_t) __popc(flags[p >> 5] & ((1u << (p & 31)) - 1u));

        for (uint32_t w = 0; w < (p >> 5); w++)
            rank += (uint32_t) __popc(flags[w]);
        const uint32_t len = block_size - p * SP_PAGE < SP_PAGE ? block_size - p * SP_PAGE : SP_PAGE;
        const uint8_t *src = blk + (size_t) p * SP_PAGE;
        uint8_t *dst = staging + (size_t) (base + rank) * SP_PAGE;

        if ((len & 15u) == 0)
            for (uint32_t v = lane; v < len / 16; v += 32)
                reinterpret_cast<uint4 *>(dst)[v] = reinterpret_cast<const uint4 *>(src)[v];
        else
            for (uint32_t i = lane; i < len; i += 32)
                dst[i] = src[i];
    }
}

/* CTAs worth launching for the LZ4 encoder: one per LZ4E_WARPS work items */
static size_t
lz4e_items(uint32_t block_size, size_t n)
{
    uint32_t seg;

    return (n * lz4e_seg_count(block_size, &seg) + LZ4E_WARPS - 1) / LZ4E_WARPS;
}

/* ---- page chains (cryo_pages.cuh): one CTA per cryo block ---- */

__global__ void __launch_bounds__(256)
k_pages_gather(const uint8_t *pages, const uint32_t *slot, const uint32_t *blkno, const uint32_t *chain_off,
               uint8_t *comp, uint64_t *src_off, uint32_t *src_size, int32_t *dec_method, int32_t *hdr_method,
               int32_t *chain_status, uint32_t max_csize)
{
    const uint32_t b = blockIdx.x;

    pg_gather_block(pages, slot, blkno, chain_off[b], chain_off[b + 1], comp, src_off + b, src_size + b, dec_method + b,
                    hdr_method + b, chain_status + b, max_csize, threadIdx.x, 256);
}

/* after the decoders: a block whose chain failed reports that, not the decoders' "unknown method" */
__global__ void
k_pages_status(const int32_t *chain_status, const uint32_t *src_size, int32_t *status, uint32_t *out_size,
               uint32_t *comp_size, uint32_t n)
{
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;

    if (b >= n)
        return;
    if (chain_status[b] != PG_ST_OK)
    {
        status[b] = chain_status[b];
        out_size[b] = 0;
    }
    if (comp_size)
        comp_size[b] = src_size[b];
}

__global__ void __launch_bounds__(256)
k_pages_split(const uint8_t *comp, uint64_t comp_stride, const uint32_t *comp_size, const int32_t *comp_status,
              uint32_t method, uint32_t xid, const uint32_t *blkno, uint32_t cap_pages, uint8_t *pages,
              uint64_t pages_stride, uint32_t *npages, int32_t *status)
{
    const uint32_t b = blockIdx.x;
    uint32_t np = 0;

    if (comp_status[b] == ST_OK)
        np = pg_split_block(comp + b * comp_stride, comp_size[b], method, xid, blkno + (size_t) b * cap_pages, cap_pages,
                            pages + b * pages_stride, threadIdx.x, 256);
    if (threadIdx.x == 0)
    {
        npages[b] = np;
        status[b] = comp_status[b] != ST_OK ? comp_status[b] : np ? ST_OK : ST_OUTPUT;
    }
}

/* tuple-level walk of decoded blocks (cryo_pages.cuh): one warp per block, 8 blocks per CTA */
__global__ void __launch_bounds__(256)
k_tuple_stats(const uint8_t *blocks, uint64_t stride, uint32_t block_size, const int32_t *status, uint32_t *ntuples,
              unsigned long long *tuple_bytes, int32_t *valid, uint32_t n)
{
    const uint32_t b = blockIdx.x * 8u + (threadIdx.x >> 5), lane = threadIdx.x & 31u;

    if (b >= n)
        return;
    if (status && status[b] != ST_OK)
    {
        if (lane == 0)
        {
            ntuples[b] = 0;
            tuple_bytes[b] = 0;
            valid[b] = 0;
        }
        return;
    }
    pg_tuple_stats(blocks + b * stride, block_size, ntuples + b, tuple_bytes + b, valid + b, lane);
}

/* batched tuple fetch (cryo_tuples.cuh): select and gather one warp per block, 8 blocks per CTA; the scan one CTA */
__global__ void __launch_bounds__(256)
k_tuple_select(const uint8_t *blocks, uint64_t stride, uint32_t block_size, const int32_t *block_status,
               const tup_u64 *sel_off, const uint32_t *sel_pos, tup_u64 *cnt, tup_u64 *bytes, int32_t *status, uint32_t n)
{
    const uint32_t b = blockIdx.x * 8u + (threadIdx.x >> 5), lane = threadIdx.x & 31u;

    if (b < n)
        tup_select_block(blocks + b * stride, block_size, block_status ? block_status[b] : ST_OK, sel_off, sel_pos, b,
                         cnt + b, bytes + b, status + b, lane);
}

__global__ void __launch_bounds__(TUP_SCAN_THREADS)
k_tuple_scan(uint32_t n, const tup_u64 *cnt, const tup_u64 *bytes, int32_t *status, tup_u64 ent0, tup_u64 byte0,
             tup_u64 tup_cap, tup_u64 data_cap, tup_u64 *block_first, tup_u64 *byte_first, tup_u64 *need)
{
    tup_scan(n, cnt, bytes, status, ent0, byte0, tup_cap, data_cap, block_first, byte_first, need,
             (tup_u64 *) CRYO_SMEM_BASE(), threadIdx.x, TUP_SCAN_THREADS);
}

__global__ void __launch_bounds__(256, 4)      /* 4 CTAs per SM: 62 registers, no spills (a bare 256 spilled) */
k_tuple_gather(const uint8_t *blocks, uint64_t stride, uint32_t block_size, const int32_t *status, const tup_u64 *sel_off,
               const uint32_t *sel_pos, const tup_u64 *block_first, const tup_u64 *byte_first, TupOut o, uint32_t n)
{
    const uint32_t b = blockIdx.x * 8u + (threadIdx.x >> 5), lane = threadIdx.x & 31u;

    if (b < n && status[b] == ST_OK)
        tup_gather_block(blocks + b * stride, block_size, sel_off, sel_pos, b, block_first[b], byte_first[b], o, lane);
}

/* cryo blocks from packed tuples (cryo_tuples.cuh): one CTA per block */
__global__ void __launch_bounds__(BLK_THREADS)
k_block_build(const uint8_t *data, tup_u64 data_lo, tup_u64 data_size, const tup_u64 *tup_off, const uint32_t *tup_len,
              const tup_u64 *block_first, uint32_t block_size, uint8_t *dst, uint64_t dst_stride, int32_t *status)
{
    const uint32_t b = blockIdx.x;

    blk_build_block(data, data_lo, data_size, tup_off, tup_len, block_first, b, block_size, dst + b * dst_stride, status + b,
                    (uint32_t *) CRYO_SMEM_BASE(), threadIdx.x);
}

/* CRYOGPU_LZ4_KERNEL = warp | cx forces one LZ4 decoder for every block; default: routed per block */
static int
lz4_kernel_choice()
{
    static int v = -1;

    if (v < 0)
    {
        const char *e = getenv("CRYOGPU_LZ4_KERNEL");

        v = (e && strcmp(e, "warp") == 0) ? 1 : (e && strcmp(e, "cx") == 0) ? 2 : 0;
    }
    return v;
}

/* device memory behind the CTA-per-block LZ4 decoder for a batch of n blocks: the work counter and the
 * length of the list, the list of blocks the warp decoder gave up, the sequence records of one parse round per CTA */
static size_t
lz4c_grid(size_t n, int sm_count)
{
    return std::min<size_t>(n, (size_t) sm_count);
}

static size_t
lz4c_bytes(size_t n, int sm_count)
{
    return 256 + ((n * 4 + 255) & ~(size_t) 255) + lz4c_grid(n, sm_count) * LZ4C_SCRATCH_BYTES;
}

/*
 * LZ4 blocks of a batch.  Small batches (every block can have an SM of its own) go to the CTA-per-block
 * kernel whole; in larger ones the warp decoder hands over the blocks with too many sequences.  work: lz4c_bytes(n) bytes, or nullptr
 * (allocation failed, block size beyond the record format): one warp per block.
 */
static void
launch_lz4_decode(cudaStream_t st, size_t n, const int32_t *methods, const uint8_t *src,
                  const uint64_t *src_off, const uint32_t *src_size, uint8_t *dst,
                  uint64_t dst_stride, uint32_t cap, uint32_t *out_size, int32_t *status, void *work,
                  int sm_count)
{
    const int choice = lz4_kernel_choice();

    if (!work || cap > LZ4C_MAXCAP || choice == 1)
    {
        k_lz4_decode_w<<<(unsigned) ((n + LZ4W_WARPS - 1) / LZ4W_WARPS), LZ4W_THREADS, LZ4W_SMEM, st>>>(
            methods, src, src_off, src_size, dst, dst_stride, cap, out_size, status, (uint32_t) n, nullptr, nullptr);
        return;
    }
    uint32_t *counter = (uint32_t *) work;
    const size_t na = (n * 4 + 255) & ~(size_t) 255;
    uint32_t *list = (uint32_t *) ((uint8_t *) work + 256);
    unsigned long long *gseq = (unsigned long long *) ((uint8_t *) work + 256 + na);
    const bool all_cx = choice == 2 || n <= (size_t) 2 * sm_count;

    cudaMemsetAsync(counter, 0, 8, st);         /* work counter, length of the list */
    if (!all_cx)
        k_lz4_decode_w<<<(unsigned) ((n + LZ4W_WARPS - 1) / LZ4W_WARPS), LZ4W_THREADS, LZ4W_SMEM, st>>>(
            methods, src, src_off, src_size, dst, dst_stride, cap, out_size, status, (uint32_t) n, list, counter + 1);
    k_lz4_decode_c<<<(unsigned) lz4c_grid(n, sm_count), CX_THREADS, LZ4C_SMEM, st>>>(
        methods, src, src_off, src_size, dst, dst_stride, cap, out_size, status, (uint32_t) n,
        all_cx ? nullptr : list, counter, gseq);
}

/* CRYOGPU_ZSTD_KERNEL = warp selects the one-warp-per-frame decoder for every frame (2); default: the
 * phase-split pipeline (3, zstd_decode_p.cuh), which hands the frames it declines to that decoder */
static int
zstd_kernel_variant()
{
    static int v = -1;

    if (v < 0)
    {
        const char *e = getenv("CRYOGPU_ZSTD_KERNEL");

        v = (e && strcmp(e, "warp") == 0) ? 2 : 3;
    }
    return v;
}

/* device memory behind the pipeline for n frames of capacity cap, and its carving */
static size_t
zp_al(size_t v)
{
    return (v + 255) & ~(size_t) 255;
}

static size_t
zp_bytes(size_t n, uint32_t cap)
{
    return zp_al(n * ZP_FF * 4) + 3 * zp_al(n * 4) + zp_al(n * 8) + 256 + zp_al(n * ZP_MAXB * ZP_BF * 4) +
           zp_al(n * zp_lit_stride(cap)) + zp_al(zp_seq_cap(n, cap) * 8) + zp_al(n * ZP_MAXB * 4096) +
           zp_al(n * ZP_MAXB * ZP3_CELLS * 4) + zp_al(n * ZP_JOBS * 16) + zp_al(n * 4);
}

static void
zp_carve(ZpArgs &a, void *base, size_t n, uint32_t cap)
{
    uint8_t *p = (uint8_t *) base;

    a.fr = (uint32_t *) p;
    p += zp_al(n * ZP_FF * 4);
    a.flag = (uint32_t *) p;
    p += zp_al(n * 4);
    a.pf_done = (uint32_t *) p;
    p += zp_al(n * 4);
    a.cxlist = (uint32_t *) p;
    p += zp_al(n * 4);
    a.seqbase = (uint64_t *) p;
    p += zp_al(n * 8);
    a.seq_alloc = (unsigned long long *) p;         /* + 8: work counter of k_zp_execute_c, + 12: cxcount, + 16: work counter of k_zp_prefill */
    a.cxcount = (uint32_t *) p + 3;
    p += 256;
    a.blk = (uint32_t *) p;
    p += zp_al(n * ZP_MAXB * ZP_BF * 4);
    a.lit = p;
    a.lit_stride = zp_lit_stride(cap);
    p += zp_al(n * a.lit_stride);
    a.seq = (uint64_t *) p;
    a.seq_cap = zp_seq_cap(n, cap);
    p += zp_al(a.seq_cap * 8);
    a.huftab = (uint16_t *) p;
    p += zp_al(n * ZP_MAXB * 4096);
    a.fsetab = (uint32_t *) p;
    p += zp_al(n * ZP_MAXB * ZP3_CELLS * 4);
    a.jobs = (uint32_t *) p;
    p += zp_al(n * ZP_JOBS * 16);
    a.pf_expect = (uint32_t *) p;
}

static void
launch_zstd_decode(cudaStream_t st, size_t n, const int32_t *methods, const uint8_t *src,
                   const uint64_t *src_off, const uint32_t *src_size, uint8_t *dst,
                   uint64_t dst_stride, uint32_t cap, uint32_t *out_size, int32_t *status,
                   uint8_t *scratch, const uint32_t *predef, void *zpbuf, cudaStream_t *aux,
                   cudaEvent_t *ev, int sm_count)
{
    /* no work area (allocation failed, or more frames than the pipeline indexes): one warp per frame */
    const int variant = zstd_kernel_variant() == 3 && !zpbuf ? 2 : zstd_kernel_variant();

    if (variant == 2)
        k_zstd_decode_w<<<(unsigned) ((n + ZSW_WARPS - 1) / ZSW_WARPS), ZSW_THREADS, ZSW_SMEM, st>>>(
            methods, src, src_off, src_size, dst, dst_stride, cap, out_size, status, scratch,
            ZSTDD_SCRATCH_BYTES, predef, (uint32_t) n, nullptr);
    else
    {
        ZpArgs a = {};
        const unsigned ngroups = (unsigned) ((n + ZP_G - 1) / ZP_G);

        a.methods = methods;
        a.src = src;
        a.src_off = src_off;
        a.src_size = src_size;
        a.dst = dst;
        a.dst_stride = dst_stride;
        a.cap = cap;
        a.n = (uint32_t) n;
        a.out_size = out_size;
        a.status = status;
        a.predef = predef;
        zp_carve(a, zpbuf, n, cap);
        {
            static int hint = -1;

            if (hint < 0)
            {
                const char *e = getenv("CRYOGPU_ZP_PREFILL_L2HINT"), *x = getenv("CRYOGPU_ZP_EXEC_PREFETCH"),
                           *s = getenv("CRYOGPU_ZP_SRC_PREFETCH");

                hint = (e ? atoi(e) != 0 : ZP_L2HINT_DEFAULT) | ((x ? atoi(x) != 0 : ZP_EXEC_PREFETCH_DEFAULT) << 1) |
                       ((s ? atoi(s) != 0 : 1) << 4);

            }
            a.pf_hint = (uint32_t) hint;
        }
        /*
         * Who runs stage 4.  A batch small enough that every frame can have an SM of its own goes to the
         * CTA-per-frame executor whole (bit 2): the warp executor and the raw / RLE stage are not launched.
         * In a larger batch stage 1 routes every frame by its number of sequences.  CRYOGPU_ZSTD_EXEC =
         * warp | cx forces one of them.
         */
        static int exec_choice = -1;

        if (exec_choice < 0)
        {
            const char *e = getenv("CRYOGPU_ZSTD_EXEC");

            exec_choice = (e && strcmp(e, "warp") == 0) ? 1 : (e && strcmp(e, "cx") == 0) ? 2 : 0;
        }
        const bool all_cx = exec_choice == 2 || (exec_choice == 0 && n <= (size_t) 2 * sm_count);
        uint32_t  *cx_counter = (uint32_t *) (a.seq_alloc + 1);

        if (all_cx)
            a.pf_hint |= 4u;
        else if (exec_choice == 1)
            a.pf_hint |= 8u;
        cudaMemsetAsync(a.seq_alloc, 0, 64, st);       /* + the work counters of k_zp_execute_c and k_zp_prefill, the job queue's */
        {
            /* long runs of stage 4 handed to stage 0 (ZP_JOBS); CRYOGPU_ZP_JOBS=0: stage 4 writes them itself */
            static int use_jobs = -1;

            if (use_jobs < 0)
            {
                const char *e = getenv("CRYOGPU_ZP_JOBS");

                use_jobs = e ? atoi(e) : 1;
            }
            if (use_jobs == 2)
                a.pf_hint |= 32u;
            if (!use_jobs || all_cx)
            {
                a.jobs = nullptr;
                a.pf_expect = nullptr;
            }
            else
                cudaMemsetAsync(a.jobs, 0, n * ZP_JOBS * 16, st);
            a.exec_warps = (uint32_t) ((n + ZP4_WARPS - 1) / ZP4_WARPS) * ZP4_WARPS;
        }
        k_zp_parse<<<(unsigned) ((n + 31) / 32), 32, 0, st>>>(a);
        /*
         * literals (st) and sequences (aux 0) are independent of each other and bound by latency.
         * Once the sequences are walked the positions of the raw / RLE blocks are known (zp_frame_positions);
         * those blocks (aux 1, one persistent CTA per SM, bound by HBM) are then written beside the
         * executor (st, bound by instruction issue), which synchronises with them per frame through
         * pf_done.  Running them beside the entropy stages instead was measured slower (a stage that
         * saturates HBM stretches the memory latency the lockstep stages depend on;
         * profiles/r01e_arrangements.txt).
         */
        static int pf_ctas = -1;                /* CTAs per SM of the raw / RLE stage (tuning knob) */

        if (pf_ctas < 0)
        {
            const char *e = getenv("CRYOGPU_ZP_PREFILL_CTAS");

            pf_ctas = e && atoi(e) > 0 ? atoi(e) : 1;
        }
        const unsigned pf_grid = (unsigned) std::min<size_t>(n, (size_t) pf_ctas * sm_count);

        /*
         * The lane-serial stages: warps per group of ZP_G frames (see ZP_FOR_GROUP_BLOCKS).  As many as one wave
         * of the device holds, so that a batch whose warps all fit runs as ONE wave (a second, nearly empty wave
         * doubles the stage: its length is that of the longest chain), and at most one per block index.
         */
        static int wave[5] = {0, 0, 0, 0, 0};   /* warps of stage 2b / 3b small / 3b large, CTAs of 2a / 3a resident on the device */

        if (wave[0] == 0)
        {
            int per_sm[5] = {1, 1, 1, 1, 1};

            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm[3], k_zp_huftab, 32 * ZP2A_WARPS, ZP2A_SMEM);
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm[4], k_zp_fsetab, 32 * ZP3A_WARPS, ZP3A_SMEM);
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm[0], k_zp_literals, 32, ZP2B_SMEM);
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm[1], k_zp_sequences_small, 32,
                                                          ZP3B_SMEM(ZP3B_SMALL, ZP3B_SMALL_LANES));
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm[2], k_zp_sequences_large, 32, ZP3B_SMEM(ZP3B_LARGE, ZP_G));
            for (int k = 0; k < 5; k++)
                wave[k] = std::max(1, per_sm[k]) * sm_count;
        }
        unsigned split[5];

        for (int k = 0; k < 5; k++)
            split[k] = std::min<unsigned>(ZP_MAXB, std::max<unsigned>(1u, (unsigned) wave[k] / ngroups));
        /*
         * The early pass of the raw / RLE stage (aux 1; CRYOGPU_ZP_EARLY_CTAS, CRYOGPU_ZP_EARLY_PCT): beside the entropy
         * stages, which leave HBM idle for a third of the step, the raw / RLE blocks of the last PCT % of the frames are
         * written at the positions stage 1 guessed.  Alone it gained nothing (its stores stretch the literal stage, and the
         * executor took its 480 us with or without the raw / RLE stage beside it: 1.04-1.36 ms per step against 1.02);
         * with the executor's long runs handed to stage 0 as well (ZP_JOBS) the executor is down to its sequence work and
         * the step follows the bytes: 0.90 ms at 50-60 %, 1.0-1.15 at 70-100 % (profiles/r02_early_pass.txt).
         */
        static int early_ctas = -1, early_pct = -1;

        if (early_ctas < 0)
        {
            const char *e = getenv("CRYOGPU_ZP_EARLY_CTAS"), *q = getenv("CRYOGPU_ZP_EARLY_PCT");

            early_ctas = e ? atoi(e) : ZP_EARLY_CTAS_DEFAULT;
            if (early_ctas < 0)
                early_ctas = sm_count;
            early_pct = q ? std::min(100, std::max(0, atoi(q))) : ZP_EARLY_PCT_DEFAULT;
        }
        a.early_frames = (early_ctas > 0 && !all_cx) ? (uint32_t) (n * (size_t) early_pct / 100) : 0u;
        {
            static int inflight = -1;           /* 128 KiB groups of the raw / RLE stage in flight per CTA */

            if (inflight < 0)
            {
                const char *e = getenv("CRYOGPU_ZP_PF_INFLIGHT");

                inflight = e && atoi(e) > 0 ? atoi(e) : ZP_PF_INFLIGHT_DEFAULT;
            }
            a.pf_inflight = (uint32_t) inflight;
        }
        cudaEventRecord(ev[0], st);
        cudaStreamWaitEvent(aux[0], ev[0], 0);
        if (a.early_frames)
        {
            cudaStreamWaitEvent(aux[1], ev[0], 0);
            k_zp_prefill_early<<<(unsigned) std::min<size_t>(a.early_frames, (size_t) early_ctas), ZP0_THREADS, 0, aux[1]>>>(a);
            cudaEventRecord(ev[3], aux[1]);
        }
        k_zp_fsetab<<<ngroups * split[4], 32 * ZP3A_WARPS, ZP3A_SMEM, aux[0]>>>(a, split[4]);
        k_zp_sequences_small<<<ngroups * split[1], 32, ZP3B_SMEM(ZP3B_SMALL, ZP3B_SMALL_LANES), aux[0]>>>(a, split[1]);
        k_zp_sequences_large<<<ngroups * split[2], 32, ZP3B_SMEM(ZP3B_LARGE, ZP_G), aux[0]>>>(a, split[2]);
        cudaEventRecord(ev[1], aux[0]);
        k_zp_huftab<<<ngroups * split[3], 32 * ZP2A_WARPS, ZP2A_SMEM, st>>>(a, split[3]);
        k_zp_literals<<<ngroups * split[0], 32, ZP2B_SMEM, st>>>(a, split[0]);
        cudaStreamWaitEvent(st, ev[1], 0);
        if (all_cx)
            k_zp_execute_c<<<(unsigned) std::min<size_t>(n, (size_t) sm_count), CX_THREADS, ZC_SMEM, st>>>(a, cx_counter);
        else
        {
            cudaEventRecord(ev[0], st);
            cudaStreamWaitEvent(aux[1], ev[0], 0);
            k_zp_prefill<<<pf_grid, ZP0_THREADS, 0, aux[1]>>>(a);
            cudaEventRecord(ev[2], aux[1]);
            if (a.early_frames)
                cudaStreamWaitEvent(st, ev[3], 0);      /* stage 4 writes over wrong guesses: the early pass must have ended */
            k_zp_execute<<<(unsigned) ((n + ZP4_WARPS - 1) / ZP4_WARPS), ZP4_THREADS, ZP4_SMEM, st>>>(a);
            /*
             * The frames with many sequences, after the warp executor in the same stream.  A CTA of this
             * kernel takes a whole SM (1 024 threads x 64 registers): launched beside the others it makes
             * the SMs drain first and then races the raw / RLE stage and the warp executor for them, and
             * that stage must have its CTAs resident before the executor's (profiles/r01e_arrangements.txt;
             * measured again in round 2: 4.0 ms per headline step instead of 1.1).  With nothing routed the
             * CTAs find an empty list and leave.
             */
            if (exec_choice != 1)
                k_zp_execute_c<<<(unsigned) std::min<size_t>(n, (size_t) sm_count), CX_THREADS, ZC_SMEM, st>>>(a, cx_counter);
            cudaStreamWaitEvent(st, ev[2], 0);
            if (a.jobs)
                k_zp_check<<<(unsigned) ((n * ZP_JOBS + 255) / 256), 256, 0, st>>>(a);
        }
        /* frames the pipeline declined (flag set): decoded from scratch, one warp per frame */
        k_zstd_decode_w<<<(unsigned) ((n + ZSW_WARPS - 1) / ZSW_WARPS), ZSW_THREADS, ZSW_SMEM, st>>>(
            methods, src, src_off, src_size, dst, dst_stride, cap, out_size, status, scratch,
            ZSTDD_SCRATCH_BYTES, predef, (uint32_t) n, a.flag);
    }
}


/* ------------------------------------------------------- host worker pool */

/* A few host threads that place sparse results into the caller's blocks (copy the non-zero
 * pages, zero-fill the rest).  This is data placement for the host-pointer API, not a codec. */
struct HostPool
{
    std::vector<std::thread> th;
    std::mutex              m;
    std::condition_variable cv, done;
    std::function<void(size_t)> job;
    std::atomic<size_t>     next{0};
    size_t                  total = 0, active = 0;
    uint64_t                gen = 0;
    bool                    stop = false;

    void start(int n)
    {
        for (int i = 0; i < n; i++)
            th.emplace_back([this]() {
                uint64_t seen = 0;

                for (;;)
                {
                    {
                        std::unique_lock<std::mutex> lk(m);

                        cv.wait(lk, [&]() { return stop || gen != seen; });
                        if (stop)
                            return;
                        seen = gen;
                    }
                    work();
                    {
                        std::lock_guard<std::mutex> lk(m);

                        if (--active == 0)
                            done.notify_all();
                    }
                }
            });
    }
    void work()
    {
        for (;;)
        {
            size_t i = next.fetch_add(1);

            if (i >= total)
                return;
            job(i);
        }
    }
    /* run f(0..items-1) on the pool and the calling thread; returns when all are done */
    void run(size_t items, std::function<void(size_t)> f)
    {
        {
            std::lock_guard<std::mutex> lk(m);

            job = std::move(f);
            total = items;
            next = 0;
            active = th.size();
            gen++;
        }
        cv.notify_all();
        work();
        std::unique_lock<std::mutex> lk(m);

        done.wait(lk, [&]() { return active == 0; });
    }
    ~HostPool()
    {
        {
            std::lock_guard<std::mutex> lk(m);

            stop = true;
        }
        cv.notify_all();
        for (auto &t : th)
            t.join();
    }
};

/* ----------------------------------------------------------------- context */

struct DevBuf
{
    void   *p = nullptr;
    size_t  cap = 0;
};

struct cryogpu_ctx
{
    int          device = -1;
    cudaStream_t stream = nullptr;      /* compute + copies of the *_host calls */
    cudaStream_t stream2 = nullptr;     /* second lane for double buffering */
    cudaEvent_t  ev[2] = {nullptr, nullptr};
    DevBuf       scratch;               /* per-block kernel scratch */
    DevBuf       zp[2];                 /* zstd pipeline work areas (zstd_decode_p.cuh), per lane */
    DevBuf       lzw[2];                /* CTA-per-block LZ4 decoder work areas (lz4c_bytes), per lane */
    DevBuf       pgw;                   /* page-chain calls: gathered streams / compressed blocks before the split */
    DevBuf       tpw, tpo;              /* tuple fetch: per-block counts and offsets, selection; packed output (host calls) */
    DevBuf       h_tpw, h_tpo;          /* tuple fetch, host calls: pinned selection / results, packed output */
    cudaEvent_t  busy = nullptr;        /* end of the last device-resident call: the work areas are shared */
    cudaStream_t zaux[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};   /* side streams of the pipeline's concurrent stages */
    cudaEvent_t  zev[2][4] = {{nullptr, nullptr, nullptr, nullptr}, {nullptr, nullptr, nullptr, nullptr}};
    uint32_t    *predef = nullptr;      /* predefined zstd FSE tables (device) */
    /* *_host staging (device + pinned host), two lanes */
    DevBuf       d_in[2], d_out[2], d_meta[2];
    DevBuf       h_in[2], h_meta[2], h_out[2];
    std::recursive_mutex mu;            /* recursive: the page-chain host calls hold it around the device calls they make */
    bool         attrs_set = false;
    int          sm_count = 148;
    /* sparse return of the host decompress call */
    DevBuf       d_stage[2], d_sp[2];   /* packed non-zero pages; bitmap + page_off + counter */
    DevBuf       h_stage[2], h_sp[2];
    HostPool    *pool = nullptr;
    int          sparse = -1;           /* -1 unset, 0 off, 1 on (CRYOGPU_SPARSE_D2H) */
    int          zero_unmap = -1;       /* -1 unset (CRYOGPU_ZERO_UNMAP, default off), 0 off, 1 on (cryogpu_set_zero_by_unmap) */
    uint64_t     last_h2d = 0, last_d2h = 0;
    size_t       last_zp_n = 0;         /* frames of the last decompress_device call that took the pipeline */
    size_t       last_lz_n = 0;         /* blocks of the last decompress_device call that were routed per block (0: not routed) */
    uint32_t     last_zp_cap = 0;
};

static int
dev_reserve(DevBuf &b, size_t bytes)
{
    if (bytes <= b.cap)
        return CRYOGPU_OK;
    if (b.p)
        CU(cudaFree(b.p));
    b.p = nullptr;
    b.cap = 0;
    bytes = (bytes + (1u << 20) - 1) & ~(size_t) ((1u << 20) - 1);
    CU(cudaMalloc(&b.p, bytes));
    b.cap = bytes;
    return CRYOGPU_OK;
}

static int
host_reserve(DevBuf &b, size_t bytes)
{
    if (bytes <= b.cap)
        return CRYOGPU_OK;
    if (b.p)
        CU(cudaFreeHost(b.p));
    b.p = nullptr;
    b.cap = 0;
    bytes = (bytes + (1u << 20) - 1) & ~(size_t) ((1u << 20) - 1);
    CU(cudaMallocHost(&b.p, bytes));
    b.cap = bytes;
    return CRYOGPU_OK;
}

/*
 * The side streams of lane l of the pipeline (and, for lane 1, the second stream of the host calls).  Lane 1 is
 * made when a host call first needs a second chunk in flight: every stream alive takes a share of the hardware
 * work queues (see cryogpu_init).  zaux[l][1] carries the raw / RLE stage, whose CTAs must become resident
 * before the executor's (profiles/r01e_arrangements.txt): highest priority, so they win whenever an SM has room.
 */
static int
make_lane_streams(cryogpu_ctx *ctx, int l)
{
    int lo_pri = 0, hi_pri = 0;

    if (ctx->zaux[l][0])
        return CRYOGPU_OK;
    CU(cudaDeviceGetStreamPriorityRange(&lo_pri, &hi_pri));
    if (l == 1 && !ctx->stream2)
        CU(cudaStreamCreateWithFlags(&ctx->stream2, cudaStreamNonBlocking));
    for (int k = 0; k < 2; k++)
        CU(cudaStreamCreateWithPriority(&ctx->zaux[l][k], cudaStreamNonBlocking, k == 1 ? hi_pri : lo_pri));
    return CRYOGPU_OK;
}

static int
set_kernel_attrs(cryogpu_ctx *ctx)
{
    if (ctx->attrs_set)
        return CRYOGPU_OK;
    CU(cudaFuncSetAttribute(k_lz4_decode_c, cudaFuncAttributeMaxDynamicSharedMemorySize, LZ4C_SMEM));
    CU(cudaFuncSetAttribute(k_zp_execute_c, cudaFuncAttributeMaxDynamicSharedMemorySize, ZC_SMEM));
    CU(cudaFuncSetAttribute(k_lz4_decode_w, cudaFuncAttributeMaxDynamicSharedMemorySize, LZ4W_SMEM));
    CU(cudaFuncSetAttribute(k_zstd_decode_w, cudaFuncAttributeMaxDynamicSharedMemorySize, ZSW_SMEM));
    CU(cudaFuncSetAttribute(k_zp_sequences_large, cudaFuncAttributeMaxDynamicSharedMemorySize, ZP3B_SMEM(ZP3B_LARGE, ZP_G)));
    CU(cudaFuncSetAttribute(k_zp_sequences_small, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            ZP3B_SMEM(ZP3B_SMALL, ZP3B_SMALL_LANES)));
    /* the pipeline's kernels run side by side on one SM (zstd_decode_p.cuh): give them all the same
     * shared-memory carve-out, because an SM has to drain before it can change its L1 / shared split */
    {
        const void *zp_kernels[] = {(const void *) k_zp_parse, (const void *) k_zp_prefill, (const void *) k_zp_huftab,
                                    (const void *) k_zp_literals, (const void *) k_zp_fsetab,
                                    (const void *) k_zp_sequences_small, (const void *) k_zp_sequences_large,
                                    (const void *) k_zp_execute, (const void *) k_zstd_decode_w,
                                    (const void *) k_zp_execute_c, (const void *) k_lz4_decode_c,
                                    (const void *) k_lz4_decode_w,
                                    (const void *) k_flag_unknown_methods};

        for (const void *k : zp_kernels)
            CU(cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    }
    CU(cudaMalloc(&ctx->predef, ZSW_PREDEF_CELLS * sizeof(uint32_t)));
    k_zstd_build_predef<<<1, 32, 0, ctx->stream>>>(ctx->predef);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(ctx->stream));
    CU(cudaFuncSetAttribute(k_lz4_encode, cudaFuncAttributeMaxDynamicSharedMemorySize, LZ4E_SMEM));
    CU(cudaFuncSetAttribute(k_zstd_encode, cudaFuncAttributeMaxDynamicSharedMemorySize, ZSTDE_SMEM));
    ctx->attrs_set = true;
    return CRYOGPU_OK;
}

extern "C" int
cryogpu_version(void)
{
    return CRYOGPU_VERSION;
}

extern "C" const char *
cryogpu_last_error(void)
{
    return g_err;
}

extern "C" const char *
cryogpu_status_string(int s)
{
    switch (s)
    {
        case CRYOGPU_ST_OK: return "ok";
        case CRYOGPU_ST_INPUT: return "truncated or over-long input";
        case CRYOGPU_ST_OUTPUT: return "output exceeds block capacity";
        case CRYOGPU_ST_OFFSET: return "match offset outside the output";
        case CRYOGPU_ST_FORMAT: return "malformed stream";
        case CRYOGPU_ST_SIZE: return "frame content size mismatch";
        case CRYOGPU_ST_METHOD: return "unknown compression method";
        case CRYOGPU_ST_UNSUPPORTED: return "unsupported stream feature";
        case CRYOGPU_ST_EMPTY_BLOCK: return "first page of the chain is new (empty block)";
        case CRYOGPU_ST_WRONG_START: return "page is not the first page of its cryo block";
        case CRYOGPU_ST_CHAIN: return "page chain does not hold the compressed block";
        default: return "unknown status";
    }
}

extern "C" int
cryogpu_device_count(void)
{
    int n = 0;

    if (cudaGetDeviceCount(&n) != cudaSuccess)
    {
        cudaGetLastError();
        return 0;
    }
    return n;
}

extern "C" int
cryogpu_init(int device, cryogpu_ctx **out)
{
    if (!out)
        return fail(CRYOGPU_E_ARG, "cryogpu_init: ctx is NULL");
    *out = nullptr;
    /*
     * Streams are mapped onto hardware work queues, 8 by default; streams that share a queue serialise, and the
     * pipeline wants its three streams (caller's, sequence chain, raw / RLE stage) on different queues.  Only
     * effective before the process's CUDA context exists (a PostgreSQL backend's first codec call); a host
     * application that initialises CUDA earlier sets the variable itself (bench.py does).
     */
    setenv("CUDA_DEVICE_MAX_CONNECTIONS", "32", 0);
    int n = cryogpu_device_count();

    if (n <= 0)
        return fail(CRYOGPU_E_CUDA, "no CUDA device: libcryogpu has no CPU fallback");
    if (device < 0 || device >= n)
        return fail(CRYOGPU_E_ARG, "device %d out of range (0..%d)", device, n - 1);
    cudaDeviceProp prop;

    CU(cudaSetDevice(device));
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(CRYOGPU_E_CUDA, "device %d is sm_%d%d; libcryogpu is built for sm_100a only",
                    device, prop.major, prop.minor);
    cryogpu_ctx *ctx = new cryogpu_ctx();

    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount > 0 ? prop.multiProcessorCount : 148;
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev[0], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev[1], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->busy, cudaEventDisableTiming) != cudaSuccess)
    {
        delete ctx;
        return fail(CRYOGPU_E_CUDA, "stream/event creation failed: %s",
                    cudaGetErrorString(cudaGetLastError()));
    }
    if (make_lane_streams(ctx, 0) != CRYOGPU_OK)
    {
        delete ctx;
        return CRYOGPU_E_CUDA;
    }
    for (int l = 0; l < 2; l++)
    {
        for (int k = 0; k < 4; k++)
            if (cudaEventCreateWithFlags(&ctx->zev[l][k], cudaEventDisableTiming) != cudaSuccess)
            {
                delete ctx;
                return fail(CRYOGPU_E_CUDA, "event creation failed: %s", cudaGetErrorString(cudaGetLastError()));
            }
    }
    int rc = set_kernel_attrs(ctx);

    if (rc != CRYOGPU_OK)
    {
        delete ctx;
        return rc;
    }
    *out = ctx;
    return CRYOGPU_OK;
}

extern "C" void
cryogpu_shutdown(cryogpu_ctx *ctx)
{
    if (!ctx)
        return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->stream2)
        cudaStreamSynchronize(ctx->stream2);
    cudaFree(ctx->scratch.p);
    cudaFree(ctx->zp[0].p);
    cudaFree(ctx->zp[1].p);
    cudaFree(ctx->lzw[0].p);
    cudaFree(ctx->lzw[1].p);
    cudaFree(ctx->pgw.p);
    cudaFree(ctx->tpw.p);
    cudaFree(ctx->tpo.p);
    cudaFreeHost(ctx->h_tpw.p);
    cudaFreeHost(ctx->h_tpo.p);
    if (ctx->busy)
        cudaEventDestroy(ctx->busy);
    cudaFree(ctx->predef);
    for (int i = 0; i < 2; i++)
    {
        cudaFree(ctx->d_in[i].p);
        cudaFree(ctx->d_out[i].p);
        cudaFree(ctx->d_meta[i].p);
        cudaFreeHost(ctx->h_in[i].p);
        cudaFreeHost(ctx->h_meta[i].p);
        cudaFreeHost(ctx->h_out[i].p);
        cudaFree(ctx->d_stage[i].p);
        cudaFree(ctx->d_sp[i].p);
        cudaFreeHost(ctx->h_stage[i].p);
        cudaFreeHost(ctx->h_sp[i].p);
        cudaEventDestroy(ctx->ev[i]);
    }
    cudaStreamDestroy(ctx->stream);
    if (ctx->stream2)
        cudaStreamDestroy(ctx->stream2);
    for (int l = 0; l < 2; l++)
    {
        for (int k = 0; k < 2; k++)
            if (ctx->zaux[l][k])
                cudaStreamDestroy(ctx->zaux[l][k]);
        for (int k = 0; k < 4; k++)
            cudaEventDestroy(ctx->zev[l][k]);
    }
    delete ctx->pool;
    delete ctx;
}

extern "C" int
cryogpu_device(const cryogpu_ctx *ctx)
{
    return ctx ? ctx->device : -1;
}

extern "C" int
cryogpu_zstd_pipeline_stats(cryogpu_ctx *ctx, uint64_t *frames, uint64_t *fallback_frames)
{
    if (!ctx)
        return fail(CRYOGPU_E_ARG, "ctx is NULL");
    std::lock_guard<std::recursive_mutex> g(ctx->mu);       /* last_zp_n / last_zp_cap and the work area are the context's */
    uint64_t total = 0, fb = 0;

    CU(cudaSetDevice(ctx->device));
    CU(cudaDeviceSynchronize());
    if (ctx->last_zp_n)
    {
        ZpArgs a = {};
        std::vector<uint32_t> fr(ctx->last_zp_n * ZP_FF), flag(ctx->last_zp_n);

        zp_carve(a, ctx->zp[0].p, ctx->last_zp_n, ctx->last_zp_cap);
        CU(cudaMemcpy(fr.data(), a.fr, fr.size() * 4, cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(flag.data(), a.flag, flag.size() * 4, cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < ctx->last_zp_n; i++)
        {
            /* a frame the pipeline kept has its block count in fr[0]; one it declined has the flag */
            total += fr[i * ZP_FF] != 0 || flag[i] != 0;
            fb += flag[i] != 0;
        }
    }
    if (frames)
        *frames = total;
    if (fallback_frames)
        *fallback_frames = fb;
    return CRYOGPU_OK;
}

extern "C" int
cryogpu_lz4_route_stats(cryogpu_ctx *ctx, uint64_t *blocks, uint64_t *cta_blocks)
{
    if (!ctx)
        return fail(CRYOGPU_E_ARG, "ctx is NULL");
    uint64_t total = 0, cx = 0;

    CU(cudaSetDevice(ctx->device));
    CU(cudaDeviceSynchronize());
    if (ctx->last_lz_n)
    {
        uint32_t cnt[2] = {0, 0};       /* work counter, length of the list of blocks handed to the CTA decoder */

        CU(cudaMemcpy(cnt, ctx->lzw[0].p, sizeof(cnt), cudaMemcpyDeviceToHost));
        total = ctx->last_lz_n;
        cx = cnt[1];
    }
    if (blocks)
        *blocks = total;
    if (cta_blocks)
        *cta_blocks = cx;
    return CRYOGPU_OK;
}

extern "C" void
cryogpu_last_transfer_bytes(const cryogpu_ctx *ctx, uint64_t *h2d, uint64_t *d2h)
{
    if (h2d)
        *h2d = ctx ? ctx->last_h2d : 0;
    if (d2h)
        *d2h = ctx ? ctx->last_d2h : 0;
}

extern "C" uint64_t
cryogpu_compress_bound(int method, uint64_t n)
{
    if (method == CRYOGPU_LZ4)
        return n + n / 255 + 16;                            /* LZ4_compressBound */
    if (method == CRYOGPU_ZSTD)                             /* ZSTD_compressBound */
        return n + (n >> 8) + (n < (128u << 10) ? (((128u << 10) - n) >> 11) : 0);
    return 0;
}

extern "C" void *
cryogpu_host_alloc(size_t bytes)
{
    void *p = nullptr;

    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess)
    {
        fail(CRYOGPU_E_NOMEM, "cudaMallocHost(%zu): %s", bytes,
             cudaGetErrorString(cudaGetLastError()));
        return nullptr;
    }
    return p;
}

extern "C" void
cryogpu_host_free(void *p)
{
    if (p)
        cudaFreeHost(p);
}

/* ------------------------------------------------------- device-resident API */

/* argument checks of the device-resident decompress calls */
static int
check_decompress_args(const cryogpu_ctx *ctx, size_t n, const void *d_dst, uint64_t dst_stride, uint32_t block_size)
{
    if (!ctx)
        return fail(CRYOGPU_E_ARG, "ctx is NULL");
    if (((uintptr_t) d_dst & 15) || (dst_stride & 15) || dst_stride < block_size)
        return fail(CRYOGPU_E_ARG, "d_dst and dst_stride must be multiples of 16, stride >= block_size");
    if (block_size == 0 || block_size > (1u << 27) || n > 0x7fffffffu)
        return fail(CRYOGPU_E_ARG, "block_size or n out of range");
    return CRYOGPU_OK;
}

/* the launches of one batched decompression on st; ctx->mu is held and st already waits for ctx->busy */
static int
decompress_device_locked(cryogpu_ctx *ctx, cudaStream_t st, size_t n, const int32_t *d_methods,
                         const uint8_t *d_src, const uint64_t *d_src_off,
                         const uint32_t *d_src_size, uint8_t *d_dst, uint64_t dst_stride,
                         uint32_t block_size, uint32_t *d_out_size, int32_t *d_status)
{
    bool  use_zp = false;
    void *lzw = nullptr;

    {
        int rc = dev_reserve(ctx->scratch, n * (size_t) ZSTDD_SCRATCH_BYTES);

        if (rc != CRYOGPU_OK)
            return rc;
        /* the CTA-per-block LZ4 decoder's area; without it every LZ4 block takes the warp kernel */
        if (block_size <= LZ4C_MAXCAP)
        {
            if (dev_reserve(ctx->lzw[0], lz4c_bytes(n, ctx->sm_count)) == CRYOGPU_OK)
                lzw = ctx->lzw[0].p;
            else
                cudaGetLastError();
        }
        /* the pipeline's work area (about 2.3 x the batch's output); without it the batch still
         * decodes, one warp per frame */
        use_zp = zstd_kernel_variant() == 3 && n <= 0xFFFFFFu;
        if (use_zp)
        {
            DevBuf &zb = ctx->zp[0];
            const size_t need = zp_bytes(n, block_size);

            if (need > zb.cap)
            {
                if (zb.p)
                    cudaFree(zb.p);
                zb.p = nullptr;
                zb.cap = 0;
                if (cudaMalloc(&zb.p, need) == cudaSuccess)
                    zb.cap = need;
                else
                {
                    cudaGetLastError();         /* not an error of this call */
                    zb.p = nullptr;
                    use_zp = false;
                }
            }
        }
    }
    k_flag_unknown_methods<<<(unsigned) ((n + 255) / 256), 256, 0, st>>>(d_methods, n, d_out_size,
                                                                         d_status);
    launch_lz4_decode(st, n, d_methods, d_src, d_src_off, d_src_size, d_dst, dst_stride, block_size,
                      d_out_size, d_status, lzw, ctx->sm_count);
    ctx->last_zp_n = use_zp ? n : 0;
    ctx->last_zp_cap = block_size;
    ctx->last_lz_n = lzw && lz4_kernel_choice() == 0 && n > (size_t) 2 * ctx->sm_count ? n : 0;
    launch_zstd_decode(st, n, d_methods, d_src, d_src_off, d_src_size, d_dst, dst_stride, block_size,
                       d_out_size, d_status, (uint8_t *) ctx->scratch.p, ctx->predef, use_zp ? ctx->zp[0].p : nullptr, ctx->zaux[0],
                       ctx->zev[0], ctx->sm_count);
    CU(cudaGetLastError());
    return CRYOGPU_OK;
}

extern "C" int
cryogpu_decompress_device(cryogpu_ctx *ctx, size_t n, const int32_t *d_methods,
                          const uint8_t *d_src, const uint64_t *d_src_off,
                          const uint32_t *d_src_size, uint8_t *d_dst, uint64_t dst_stride,
                          uint32_t block_size, uint32_t *d_out_size, int32_t *d_status,
                          void *stream)
{
    if (ctx && n == 0)
        return CRYOGPU_OK;
    int rc = check_decompress_args(ctx, n, d_dst, dst_stride, block_size);

    if (rc != CRYOGPU_OK)
        return rc;
    if (!d_methods || !d_src || !d_src_off || !d_src_size || !d_dst || !d_out_size || !d_status)
        return fail(CRYOGPU_E_ARG, "NULL device pointer");
    cudaStream_t st = stream ? (cudaStream_t) stream : ctx->stream;

    CU(cudaSetDevice(ctx->device));
    /*
     * The work areas belong to the context, so calls on one context run one after the other on the
     * device whatever streams they were given: this call's stream first waits for the end of the
     * previous device-resident call (cryogpu.h).  Work areas only grow; growing one frees and
     * allocates, which waits for the device: a steady-state call only enqueues.
     */
    std::lock_guard<std::recursive_mutex> g(ctx->mu);

    CU(cudaStreamWaitEvent(st, ctx->busy, 0));
    rc = decompress_device_locked(ctx, st, n, d_methods, d_src, d_src_off, d_src_size, d_dst, dst_stride, block_size,
                                  d_out_size, d_status);
    if (rc != CRYOGPU_OK)
        return rc;
    CU(cudaEventRecord(ctx->busy, st));
    return CRYOGPU_OK;
}

/* 64 KiB zstd blocks per frame, and CTAs worth launching for the zstd encoder (one per ZSE_WARPS work items) */
static size_t
zstde_blocks(uint32_t block_size)
{
    return ZSE_MAXBLK;                  /* bmeta rows are ZSE_MAXBLK wide whatever the block size */
}

static size_t
zstde_grid(uint32_t block_size, size_t n, int sm_count)
{
    const size_t nblk = block_size ? ((size_t) block_size + ZSE_BLOCK - 1) / ZSE_BLOCK : 1;

    return std::max<size_t>(1, std::min<size_t>((n * nblk + ZSE_WARPS - 1) / ZSE_WARPS, (size_t) sm_count));
}

/* scratch behind one batched compression of n blocks: LZ4 per block (+ the work queue and the per-block counts),
 * zstd per CTA of the persistent grid */
static size_t
compress_scratch_bytes(int method, uint32_t block_size, size_t n, int sm_count)
{
    if (method == CRYOGPU_LZ4)
        return n * lz4e_scratch_bytes(block_size) + ((n * 4 + 256 + 255) & ~(size_t) 255);
    return zstde_grid(block_size, n, sm_count) * zstde_scratch_bytes(block_size) + ((n * 4 + 256 + 255) & ~(size_t) 255) +
           n * (size_t) zstde_blocks(block_size) * 4;
}

/* the launches of one batched compression on st; scr: compress_scratch_bytes() of device memory, 256-byte aligned */
static int
launch_compress(cudaStream_t st, size_t n, int method, int level_or_accel, const uint8_t *d_src, uint64_t src_stride,
                uint32_t block_size, uint8_t *d_dst, uint64_t dst_stride, uint32_t dst_cap, uint32_t *d_dst_size,
                int32_t *d_status, uint8_t *scr, int sm_count)
{
    if (method == CRYOGPU_LZ4)
    {
        const size_t per = lz4e_scratch_bytes(block_size), qbytes = (n * 4 + 256 + 255) & ~(size_t) 255;
        uint32_t    *queue = (uint32_t *) (scr + n * per);      /* [0]: next work item; [64 + b]: finished segments of block b */

        CU(cudaMemsetAsync(queue, 0, qbytes, st));
        k_lz4_encode<<<(unsigned) std::min<size_t>(lz4e_items(block_size, n), (size_t) sm_count), LZ4E_THREADS, LZ4E_SMEM, st>>>(
            d_src, src_stride, block_size, d_dst, dst_stride, dst_cap, level_or_accel, d_dst_size, d_status, scr, per,
            (uint32_t) n, queue, queue + 64);
    }
    else
    {
        /* per CTA scratch | queue [0], finished blocks per frame [64 + f] | bytes of every block [f * ZSE_MAXBLK + b] */
        const size_t grid = zstde_grid(block_size, n, sm_count), qbytes = (n * 4 + 256 + 255) & ~(size_t) 255;
        uint32_t    *queue = (uint32_t *) (scr + grid * zstde_scratch_bytes(block_size));
        uint32_t    *bmeta = (uint32_t *) ((uint8_t *) queue + qbytes);

        if (block_size > ZSE_MAXBLK * (uint64_t) ZSE_BLOCK)
            return fail(CRYOGPU_E_ARG, "block_size above 128 MiB");
        CU(cudaMemsetAsync(queue, 0, qbytes, st));
        k_zstd_encode<<<(unsigned) grid, ZSTDE_THREADS, ZSTDE_SMEM, st>>>(
            d_src, src_stride, block_size, d_dst, dst_stride, dst_cap, level_or_accel, d_dst_size, d_status, scr,
            zstde_scratch_bytes(block_size), (uint32_t) n, queue, queue + 64, bmeta);
    }
    CU(cudaGetLastError());
    return CRYOGPU_OK;
}

/* one batched compression on st with the context's scratch; ctx->mu is held and st already waits for ctx->busy */
static int
compress_device_locked(cryogpu_ctx *ctx, cudaStream_t st, size_t n, int method, int level_or_accel,
                       const uint8_t *d_src, uint64_t src_stride, uint32_t block_size,
                       uint8_t *d_dst, uint64_t dst_stride, uint32_t dst_cap,
                       uint32_t *d_dst_size, int32_t *d_status)
{
    int rc = dev_reserve(ctx->scratch, compress_scratch_bytes(method, block_size, n, ctx->sm_count));

    if (rc != CRYOGPU_OK)
        return rc;
    return launch_compress(st, n, method, level_or_accel, d_src, src_stride, block_size, d_dst, dst_stride, dst_cap,
                           d_dst_size, d_status, (uint8_t *) ctx->scratch.p, ctx->sm_count);
}

extern "C" int
cryogpu_compress_device(cryogpu_ctx *ctx, size_t n, int method, int level_or_accel,
                        const uint8_t *d_src, uint64_t src_stride, uint32_t block_size,
                        uint8_t *d_dst, uint64_t dst_stride, uint32_t dst_cap,
                        uint32_t *d_dst_size, int32_t *d_status, void *stream)
{
    if (!ctx)
        return fail(CRYOGPU_E_ARG, "ctx is NULL");
    if (method != CRYOGPU_LZ4 && method != CRYOGPU_ZSTD)
        return fail(CRYOGPU_E_METHOD, "unknown compression method %d", method);
    if (n == 0)
        return CRYOGPU_OK;
    if (!d_src || !d_dst || !d_dst_size || !d_status)
        return fail(CRYOGPU_E_ARG, "NULL device pointer");
    if (((uintptr_t) d_src & 15) || (src_stride & 15) || ((uintptr_t) d_dst & 15) || (dst_stride & 15))
        return fail(CRYOGPU_E_ARG, "device pointers and strides must be multiples of 16");
    if (block_size == 0 || block_size > (1u << 27) || src_stride < block_size || dst_stride < dst_cap ||
        n > 0x7fffffffu)
        return fail(CRYOGPU_E_ARG, "size out of range");
    if (dst_cap < cryogpu_compress_bound(method, block_size))
        return fail(CRYOGPU_E_ARG, "dst_cap %u below cryogpu_compress_bound", dst_cap);
    cudaStream_t st = stream ? (cudaStream_t) stream : ctx->stream;

    CU(cudaSetDevice(ctx->device));
    std::lock_guard<std::recursive_mutex> g(ctx->mu);

    CU(cudaStreamWaitEvent(st, ctx->busy, 0));      /* the scratch area is the context's: see cryogpu_decompress_device */
    int rc = compress_device_locked(ctx, st, n, method, level_or_accel, d_src, src_stride, block_size, d_dst, dst_stride,
                                    dst_cap, d_dst_size, d_status);

    if (rc != CRYOGPU_OK)
        return rc;
    CU(cudaEventRecord(ctx->busy, st));
    return CRYOGPU_OK;
}

/* ------------------------------------------------------------ page chains */

static HostPool *host_pool(cryogpu_ctx *ctx);
static bool is_pinned(const void *p);
static size_t tp_al(size_t v);

extern "C" uint32_t
cryogpu_pages_needed(uint64_t compressed_size)
{
    return pg_pages_needed(compressed_size);
}

extern "C" int
cryogpu_decompress_pages_device(cryogpu_ctx *ctx, size_t n, const uint8_t *d_pages, const uint32_t *d_page_slot,
                                const uint32_t *d_page_blkno, const uint32_t *d_chain_off, size_t total_entries,
                                uint8_t *d_dst, uint64_t dst_stride, uint32_t block_size, uint32_t *d_out_size,
                                int32_t *d_status, int32_t *d_methods, uint32_t *d_comp_size, void *stream)
{
    if (ctx && n == 0)
        return CRYOGPU_OK;
    int rc = check_decompress_args(ctx, n, d_dst, dst_stride, block_size);

    if (rc != CRYOGPU_OK)
        return rc;
    if (!d_pages || !d_page_slot || !d_page_blkno || !d_chain_off || !d_dst || !d_out_size || !d_status || !d_methods)
        return fail(CRYOGPU_E_ARG, "NULL device pointer");
    if (((uintptr_t) d_pages & 15) || total_entries == 0 || total_entries > 0x7fffffffu)
        return fail(CRYOGPU_E_ARG, "d_pages must be 16-byte aligned, total_entries in range");
    cudaStream_t st = stream ? (cudaStream_t) stream : ctx->stream;

    CU(cudaSetDevice(ctx->device));
    std::lock_guard<std::recursive_mutex> g(ctx->mu);

    CU(cudaStreamWaitEvent(st, ctx->busy, 0));
    /* work area: the gathered streams (one page of room per chain entry), then per block: offset, size, the
     * method for the decoders, the outcome of the gather */
    const size_t comp_bytes = total_entries * (size_t) PG_PAGE, na = (n * 8 + 255) & ~(size_t) 255;

    rc = dev_reserve(ctx->pgw, comp_bytes + 4 * na);
    if (rc != CRYOGPU_OK)
        return rc;
    uint8_t  *comp = (uint8_t *) ctx->pgw.p;
    uint64_t *src_off = (uint64_t *) (comp + comp_bytes);
    uint32_t *src_size = (uint32_t *) (comp + comp_bytes + na);
    int32_t  *dec_method = (int32_t *) (comp + comp_bytes + 2 * na);
    int32_t  *chain_status = (int32_t *) (comp + comp_bytes + 3 * na);
    /* the largest stream either library writes for a block of this size */
    const uint32_t max_csize = (uint32_t) std::max(cryogpu_compress_bound(CRYOGPU_LZ4, block_size),
                                                   cryogpu_compress_bound(CRYOGPU_ZSTD, block_size));

    k_pages_gather<<<(unsigned) n, 256, 0, st>>>(d_pages, d_page_slot, d_page_blkno, d_chain_off, comp, src_off, src_size,
                                                 dec_method, d_methods, chain_status, max_csize);
    rc = decompress_device_locked(ctx, st, n, dec_method, comp, src_off, src_size, d_dst, dst_stride, block_size,
                                  d_out_size, d_status);
    if (rc != CRYOGPU_OK)
        return rc;
    k_pages_status<<<(unsigned) ((n + 255) / 256), 256, 0, st>>>(chain_status, src_size, d_status, d_out_size, d_comp_size,
                                                                  (uint32_t) n);
    CU(cudaGetLastError());
    CU(cudaEventRecord(ctx->busy, st));
    return CRYOGPU_OK;
}

extern "C" int
cryogpu_compress_pages_device(cryogpu_ctx *ctx, size_t n, int method, int level_or_accel, const uint8_t *d_src,
                              uint64_t src_stride, uint32_t block_size, const uint32_t *d_page_blkno, uint32_t cap_pages,
                              uint32_t created_xid, uint8_t *d_pages, uint32_t *d_npages, uint32_t *d_comp_size,
                              int32_t *d_status, void *stream)
{
    if (!ctx)
        return fail(CRYOGPU_E_ARG, "ctx is NULL");
    if (method != CRYOGPU_LZ4 && method != CRYOGPU_ZSTD)
        return fail(CRYOGPU_E_METHOD, "unknown compression method %d", method);
    if (n == 0)
        return CRYOGPU_OK;
    if (!d_src || !d_page_blkno || !d_pages || !d_npages || !d_comp_size || !d_status)
        return fail(CRYOGPU_E_ARG, "NULL device pointer");
    if (((uintptr_t) d_src & 15) || (src_stride & 15) || ((uintptr_t) d_pages & 15))
        return fail(CRYOGPU_E_ARG, "device pointers and strides must be multiples of 16");
    if (block_size == 0 || block_size > (1u << 27) || src_stride < block_size || n > 0x7fffffffu)
        return fail(CRYOGPU_E_ARG, "size out of range");
    const uint64_t bound = cryogpu_compress_bound(method, block_size);

    if (cap_pages < pg_pages_needed(bound) || cap_pages > 0xFFFFu)
        return fail(CRYOGPU_E_ARG, "cap_pages %u below cryogpu_pages_needed(cryogpu_compress_bound)", cap_pages);
    cudaStream_t st = stream ? (cudaStream_t) stream : ctx->stream;

    CU(cudaSetDevice(ctx->device));
    std::lock_guard<std::recursive_mutex> g(ctx->mu);

    CU(cudaStreamWaitEvent(st, ctx->busy, 0));
    const uint64_t cstride = (bound + 15) & ~(uint64_t) 15;
    const size_t   na = (n * 4 + 255) & ~(size_t) 255;
    int            rc = dev_reserve(ctx->pgw, n * cstride + na);

    if (rc != CRYOGPU_OK)
        return rc;
    uint8_t *comp = (uint8_t *) ctx->pgw.p;
    int32_t *cst = (int32_t *) (comp + n * cstride);

    rc = compress_device_locked(ctx, st, n, method, level_or_accel, d_src, src_stride, block_size, comp, cstride,
                                (uint32_t) cstride, d_comp_size, cst);
    if (rc != CRYOGPU_OK)
        return rc;
    k_pages_split<<<(unsigned) n, 256, 0, st>>>(comp, cstride, d_comp_size, cst, (uint32_t) method, created_xid, d_page_blkno,
                                                cap_pages, d_pages, (uint64_t) cap_pages * PG_PAGE, d_npages, d_status);
    CU(cudaGetLastError());
    CU(cudaEventRecord(ctx->busy, st));
    return CRYOGPU_OK;
}

/*
 * Host-pointer variants: the pages as they lie in the buffer pool (one pointer per page), staged through
 * pinned memory in chunks, the device calls above, results back.  Sized for the cache-fill and flush calls
 * (tens of blocks), not pipelined like cryogpu_decompress_host.
 */
#define PG_HOST_CHUNK 128u

extern "C" int
cryogpu_decompress_pages_host(cryogpu_ctx *ctx, size_t n, const void *const *pages, const uint32_t *page_blkno,
                              const uint32_t *chain_off, void *const *dst, uint32_t block_size, uint32_t *out_size,
                              int32_t *status, int32_t *methods, uint32_t *comp_size)
{
    if (!ctx)
        return fail(CRYOGPU_E_ARG, "ctx is NULL");
    if (n == 0)
        return CRYOGPU_OK;
    if (!pages || !page_blkno || !chain_off || !dst || !out_size || !status || !methods)
        return fail(CRYOGPU_E_ARG, "NULL argument");
    if (block_size == 0 || block_size > (1u << 27))
        return fail(CRYOGPU_E_ARG, "block_size out of range");
    const uint64_t stride = ((uint64_t) block_size + 15) & ~(uint64_t) 15;
    uint64_t       h2d = 0, d2h = 0;
    std::lock_guard<std::recursive_mutex> hold(ctx->mu);     /* the staging areas are the context's */

    CU(cudaSetDevice(ctx->device));
    for (size_t lo = 0; lo < n; lo += PG_HOST_CHUNK)
    {
        const size_t   cnt = std::min<size_t>(PG_HOST_CHUNK, n - lo);
        const uint32_t e0 = chain_off[lo], e1 = chain_off[lo + cnt], ne = e1 - e0;

        if (e1 < e0)
            return fail(CRYOGPU_E_ARG, "chain_off must not decrease");
        if (ne == 0)
        {
            for (size_t i = 0; i < cnt; i++)
            {
                status[lo + i] = CRYOGPU_ST_EMPTY_BLOCK;
                out_size[lo + i] = 0;
                methods[lo + i] = 0;
                if (comp_size)
                    comp_size[lo + i] = 0;
            }
            continue;
        }
        /* layout of the staging areas: pages | slot | blkno | chain_off (cnt + 1) ; results: out_size | status | methods | comp_size */
        const size_t pg_bytes = (size_t) ne * PG_PAGE, meta_in = ((size_t) ne * 8 + (cnt + 1) * 4 + 255) & ~(size_t) 255;
        const size_t meta_out = (cnt * 16 + 255) & ~(size_t) 255;
        int          rc;

        if ((rc = host_reserve(ctx->h_in[0], pg_bytes + meta_in)) != CRYOGPU_OK ||
            (rc = dev_reserve(ctx->d_in[0], pg_bytes + meta_in)) != CRYOGPU_OK ||
            (rc = host_reserve(ctx->h_out[0], cnt * stride + meta_out)) != CRYOGPU_OK ||
            (rc = dev_reserve(ctx->d_out[0], cnt * stride + meta_out)) != CRYOGPU_OK)
            return rc;
        uint8_t  *hi = (uint8_t *) ctx->h_in[0].p, *di = (uint8_t *) ctx->d_in[0].p;
        uint8_t  *ho = (uint8_t *) ctx->h_out[0].p, *dout = (uint8_t *) ctx->d_out[0].p;
        uint32_t *h_slot = (uint32_t *) (hi + pg_bytes), *h_blk = h_slot + ne, *h_coff = h_blk + ne;

        host_pool(ctx)->run((ne + 255) / 256, [&](size_t part) {
            for (uint32_t e = (uint32_t) part * 256u; e < ne && e < (uint32_t) (part + 1) * 256u; e++)
            {
                memcpy(hi + (size_t) e * PG_PAGE, pages[e0 + e], PG_PAGE);
                h_slot[e] = e;
                h_blk[e] = page_blkno[e0 + e];
            }
        });
        for (size_t i = 0; i <= cnt; i++)
            h_coff[i] = chain_off[lo + i] - e0;
        CU(cudaMemcpyAsync(di, hi, pg_bytes + meta_in, cudaMemcpyHostToDevice, ctx->stream));
        h2d += pg_bytes + meta_in;
        uint8_t *dm = dout + cnt * stride;

        rc = cryogpu_decompress_pages_device(ctx, cnt, di, (uint32_t *) (di + pg_bytes), (uint32_t *) (di + pg_bytes) + ne,
                                             (uint32_t *) (di + pg_bytes) + 2 * (size_t) ne, ne, dout, stride, block_size,
                                             (uint32_t *) dm, (int32_t *) (dm + cnt * 4), (int32_t *) (dm + cnt * 8),
                                             (uint32_t *) (dm + cnt * 12), ctx->stream);
        if (rc != CRYOGPU_OK)
            return rc;
        const bool dst_pinned = is_pinned(dst[lo]);     /* the batched cache's slots are: straight into them */

        if (dst_pinned)
        {
            CU(cudaMemcpyAsync(ho + cnt * stride, dout + cnt * stride, meta_out, cudaMemcpyDeviceToHost, ctx->stream));
            for (size_t i = 0; i < cnt; i++)
                CU(cudaMemcpyAsync(dst[lo + i], dout + i * stride, block_size, cudaMemcpyDeviceToHost, ctx->stream));
        }
        else
            CU(cudaMemcpyAsync(ho, dout, cnt * stride + meta_out, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        d2h += cnt * stride + meta_out;
        const uint8_t *hm = ho + cnt * stride;

        memcpy(out_size + lo, hm, cnt * 4);
        memcpy(status + lo, hm + cnt * 4, cnt * 4);
        memcpy(methods + lo, hm + cnt * 8, cnt * 4);
        if (comp_size)
            memcpy(comp_size + lo, hm + cnt * 12, cnt * 4);
        /* into the caller's blocks with the context's host threads (one thread moves ~6 GB/s) */
        if (!dst_pinned)
            host_pool(ctx)->run(cnt, [&](size_t i) {
                if (status[lo + i] == CRYOGPU_ST_OK)
                    memcpy(dst[lo + i], ho + i * stride, out_size[lo + i]);
            });
    }
    ctx->last_h2d = h2d;
    ctx->last_d2h = d2h;
    return CRYOGPU_OK;
}

extern "C" int
cryogpu_compress_pages_host(cryogpu_ctx *ctx, size_t n, int method, int level_or_accel, const void *const *src,
                            uint32_t block_size, const uint32_t *page_blkno, uint32_t cap_pages, uint32_t created_xid,
                            void *const *pages_out, uint32_t *npages, uint32_t *comp_size, int32_t *status)
{
    if (!ctx)
        return fail(CRYOGPU_E_ARG, "ctx is NULL");
    if (method != CRYOGPU_LZ4 && method != CRYOGPU_ZSTD)
        return fail(CRYOGPU_E_METHOD, "unknown compression method %d", method);
    if (n == 0)
        return CRYOGPU_OK;
    if (!src || !page_blkno || !pages_out || !npages || !comp_size || !status)
        return fail(CRYOGPU_E_ARG, "NULL argument");
    if (block_size == 0 || block_size > (1u << 27))
        return fail(CRYOGPU_E_ARG, "block_size out of range");
    const uint64_t stride = ((uint64_t) block_size + 15) & ~(uint64_t) 15;
    const size_t   pstride = (size_t) cap_pages * PG_PAGE;
    uint64_t       h2d = 0, d2h = 0;
    std::lock_guard<std::recursive_mutex> hold(ctx->mu);     /* the staging areas are the context's */

    CU(cudaSetDevice(ctx->device));
    for (size_t lo = 0; lo < n; lo += PG_HOST_CHUNK)
    {
        const size_t cnt = std::min<size_t>(PG_HOST_CHUNK, n - lo);
        const size_t meta_in = (cnt * cap_pages * 4 + 255) & ~(size_t) 255, meta_out = (cnt * 12 + 255) & ~(size_t) 255;
        int          rc;

        if ((rc = host_reserve(ctx->h_in[0], cnt * stride + meta_in)) != CRYOGPU_OK ||
            (rc = dev_reserve(ctx->d_in[0], cnt * stride + meta_in)) != CRYOGPU_OK ||
            (rc = host_reserve(ctx->h_out[0], cnt * pstride + meta_out)) != CRYOGPU_OK ||
            (rc = dev_reserve(ctx->d_out[0], cnt * pstride + meta_out)) != CRYOGPU_OK)
            return rc;
        uint8_t *hi = (uint8_t *) ctx->h_in[0].p, *di = (uint8_t *) ctx->d_in[0].p;
        uint8_t *ho = (uint8_t *) ctx->h_out[0].p, *dout = (uint8_t *) ctx->d_out[0].p;

        for (size_t i = 0; i < cnt; i++)
            memcpy(hi + i * stride, src[lo + i], block_size);
        memcpy(hi + cnt * stride, page_blkno + lo * cap_pages, cnt * cap_pages * 4);
        CU(cudaMemcpyAsync(di, hi, cnt * stride + meta_in, cudaMemcpyHostToDevice, ctx->stream));
        h2d += cnt * stride + meta_in;
        uint8_t *dm = dout + cnt * pstride;

        rc = cryogpu_compress_pages_device(ctx, cnt, method, level_or_accel, di, stride, block_size,
                                           (uint32_t *) (di + cnt * stride), cap_pages, created_xid, dout, (uint32_t *) dm,
                                           (uint32_t *) (dm + cnt * 4), (int32_t *) (dm + cnt * 8), ctx->stream);
        if (rc != CRYOGPU_OK)
            return rc;
        /* the counts first: only the pages each block needs come back */
        CU(cudaMemcpyAsync(ho + cnt * pstride, dm, meta_out, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        const uint8_t *hm = ho + cnt * pstride;

        memcpy(npages + lo, hm, cnt * 4);
        memcpy(comp_size + lo, hm + cnt * 4, cnt * 4);
        memcpy(status + lo, hm + cnt * 8, cnt * 4);
        d2h += meta_out;
        for (size_t i = 0; i < cnt; i++)
            if (status[lo + i] == CRYOGPU_ST_OK)
            {
                CU(cudaMemcpyAsync(ho + i * pstride, dout + i * pstride, (size_t) npages[lo + i] * PG_PAGE,
                                   cudaMemcpyDeviceToHost, ctx->stream));
                d2h += (size_t) npages[lo + i] * PG_PAGE;
            }
        CU(cudaStreamSynchronize(ctx->stream));
        for (size_t i = 0; i < cnt; i++)
            if (status[lo + i] == CRYOGPU_ST_OK)
                for (uint32_t k = 0; k < npages[lo + i]; k++)
                    memcpy(pages_out[(lo + i) * cap_pages + k], ho + i * pstride + (size_t) k * PG_PAGE, PG_PAGE);
    }
    ctx->last_h2d = h2d;
    ctx->last_d2h = d2h;
    return CRYOGPU_OK;
}

/*
 * Flush path of a batch of blocks (f-3): compress, THEN ask the caller for the block numbers -- how many
 * pages a block needs is only known after compression, and cryo_preserve (pg_cryogen.c:737-759) allocates
 * them then too: the first page was reserved when the block was started (cryo_reserve_blockno,
 * pg_cryogen.c:588-601), the others come from ReadBuffer(P_NEW) -- then cut the page images on the device
 * and place them where the caller says each page lives.
 *
 * One chunk of it, blocks [lo, lo + cnt) already in HBM at d_blocks (work enqueued on ctx->stream, ctx->mu held).
 * d_pre_status (may be NULL): a status per block from before the encoders (the block build); a block that failed
 * there keeps it, asks alloc for no page and writes nothing.  d_blk / h_blk: cnt * cap_pages block numbers of
 * device / pinned staging for the page rows.
 */
static int
flush_chunk(cryogpu_ctx *ctx, size_t lo, size_t cnt, int method, int level_or_accel, const uint8_t *d_blocks,
            uint64_t stride, uint32_t block_size, const int32_t *d_pre_status, uint32_t *d_blk, uint32_t *h_blk,
            const uint32_t *first_blkno, cryogpu_alloc_page_fn alloc, cryogpu_page_ptr_fn page_ptr, void *arg,
            uint32_t created_xid, uint32_t *npages, uint32_t *comp_size, int32_t *status, uint64_t &h2d, uint64_t &d2h)
{
    const uint64_t bound = cryogpu_compress_bound(method, block_size), cstride = (bound + 15) & ~(uint64_t) 15;
    const uint32_t cap_pages = pg_pages_needed(bound);
    const size_t   pstride = (size_t) cap_pages * PG_PAGE, meta = (cnt * 12 + 255) & ~(size_t) 255;
    int            rc;

    if ((rc = host_reserve(ctx->h_out[0], cnt * pstride + meta)) != CRYOGPU_OK ||
        (rc = dev_reserve(ctx->d_out[0], cnt * pstride + meta)) != CRYOGPU_OK ||
        (rc = dev_reserve(ctx->pgw, cnt * cstride + meta)) != CRYOGPU_OK)
        return rc;
    uint8_t  *ho = (uint8_t *) ctx->h_out[0].p, *dout = (uint8_t *) ctx->d_out[0].p;
    uint8_t  *comp = (uint8_t *) ctx->pgw.p, *dm = dout + cnt * pstride;
    uint32_t *d_np = (uint32_t *) dm, *d_cs = (uint32_t *) (dm + cnt * 4);
    int32_t  *d_st = (int32_t *) (dm + cnt * 8), *d_cst = (int32_t *) (comp + cnt * cstride);
    const uint8_t *hm = ho + cnt * pstride;

    CU(cudaStreamWaitEvent(ctx->stream, ctx->busy, 0));
    rc = compress_device_locked(ctx, ctx->stream, cnt, method, level_or_accel, d_blocks, stride, block_size, comp, cstride,
                                (uint32_t) cstride, d_cs, d_cst);
    if (rc != CRYOGPU_OK)
        return rc;
    /* a failed build overrides what the encoders made of the unwritten block: its status, compressed size 0 */
    if (d_pre_status)
    {
        k_pages_status<<<(unsigned) ((cnt + 255) / 256), 256, 0, ctx->stream>>>(d_pre_status, nullptr, d_cst, d_cs, nullptr,
                                                                               (uint32_t) cnt);
        CU(cudaGetLastError());
    }
    CU(cudaMemcpyAsync(ho + cnt * pstride + cnt * 4, d_cs, cnt * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    d2h += cnt * 4;
    /* the block numbers, in the order cryo_preserve takes them: block by block, page by page */
    const uint32_t *h_cs = (const uint32_t *) (hm + cnt * 4);

    for (size_t i = 0; i < cnt; i++)
    {
        const uint32_t np = pg_pages_needed(h_cs[i]);

        h_blk[i * cap_pages] = first_blkno[lo + i];
        for (uint32_t k = 1; k < cap_pages; k++)
            h_blk[i * cap_pages + k] = k < np ? alloc(arg) : PG_INVALID;
    }
    CU(cudaMemcpyAsync(d_blk, h_blk, cnt * cap_pages * 4, cudaMemcpyHostToDevice, ctx->stream));
    h2d += cnt * cap_pages * 4;
    k_pages_split<<<(unsigned) cnt, 256, 0, ctx->stream>>>(comp, cstride, d_cs, d_cst, (uint32_t) method, created_xid, d_blk,
                                                          cap_pages, dout, pstride, d_np, d_st);
    CU(cudaGetLastError());
    CU(cudaEventRecord(ctx->busy, ctx->stream));
    CU(cudaMemcpyAsync(ho + cnt * pstride, dm, meta, cudaMemcpyDeviceToHost, ctx->stream));
    for (size_t i = 0; i < cnt; i++)
    {
        const uint32_t np = pg_pages_needed(h_cs[i]);

        CU(cudaMemcpyAsync(ho + i * pstride, dout + i * pstride, (size_t) np * PG_PAGE, cudaMemcpyDeviceToHost, ctx->stream));
        d2h += (size_t) np * PG_PAGE;
    }
    CU(cudaStreamSynchronize(ctx->stream));
    d2h += meta;
    memcpy(npages + lo, hm, cnt * 4);
    memcpy(comp_size + lo, hm + cnt * 4, cnt * 4);
    memcpy(status + lo, hm + cnt * 8, cnt * 4);
    for (size_t i = 0; i < cnt; i++)
        if (status[lo + i] == CRYOGPU_ST_OK)
            for (uint32_t k = 0; k < npages[lo + i]; k++)
            {
                void *p = page_ptr(arg, h_blk[i * cap_pages + k]);

                if (!p)
                    return fail(CRYOGPU_E_ARG, "page_ptr returned NULL for block %u", h_blk[i * cap_pages + k]);
                memcpy(p, ho + i * pstride + (size_t) k * PG_PAGE, PG_PAGE);
            }
    return CRYOGPU_OK;
}

extern "C" int
cryogpu_compress_pages_alloc_host(cryogpu_ctx *ctx, size_t n, int method, int level_or_accel, const void *const *src,
                                  uint32_t block_size, const uint32_t *first_blkno, cryogpu_alloc_page_fn alloc,
                                  cryogpu_page_ptr_fn page_ptr, void *arg, uint32_t created_xid, uint32_t *npages,
                                  uint32_t *comp_size, int32_t *status)
{
    if (!ctx)
        return fail(CRYOGPU_E_ARG, "ctx is NULL");
    if (method != CRYOGPU_LZ4 && method != CRYOGPU_ZSTD)
        return fail(CRYOGPU_E_METHOD, "unknown compression method %d", method);
    if (n == 0)
        return CRYOGPU_OK;
    if (!src || !first_blkno || !alloc || !page_ptr || !npages || !comp_size || !status)
        return fail(CRYOGPU_E_ARG, "NULL argument");
    if (block_size == 0 || block_size > (1u << 27))
        return fail(CRYOGPU_E_ARG, "block_size out of range");
    const uint64_t stride = ((uint64_t) block_size + 15) & ~(uint64_t) 15;
    const uint32_t cap_pages = pg_pages_needed(cryogpu_compress_bound(method, block_size));
    uint64_t       h2d = 0, d2h = 0;
    std::lock_guard<std::recursive_mutex> hold(ctx->mu);

    CU(cudaSetDevice(ctx->device));
    for (size_t lo = 0; lo < n; lo += PG_HOST_CHUNK)
    {
        const size_t cnt = std::min<size_t>(PG_HOST_CHUNK, n - lo);
        const size_t blk_bytes = (cnt * cap_pages * 4 + 255) & ~(size_t) 255;
        int          rc;

        if ((rc = host_reserve(ctx->h_in[0], cnt * stride + blk_bytes)) != CRYOGPU_OK ||
            (rc = dev_reserve(ctx->d_in[0], cnt * stride + blk_bytes)) != CRYOGPU_OK)
            return rc;
        uint8_t *hi = (uint8_t *) ctx->h_in[0].p, *di = (uint8_t *) ctx->d_in[0].p;

        if (is_pinned(src[lo]))                         /* callers that hold pinned block images */
            for (size_t i = 0; i < cnt; i++)
                CU(cudaMemcpyAsync(di + i * stride, src[lo + i], block_size, cudaMemcpyHostToDevice, ctx->stream));
        else
        {
            host_pool(ctx)->run(cnt, [&](size_t i) { memcpy(hi + i * stride, src[lo + i], block_size); });
            CU(cudaMemcpyAsync(di, hi, cnt * stride, cudaMemcpyHostToDevice, ctx->stream));
        }
        h2d += cnt * stride;
        rc = flush_chunk(ctx, lo, cnt, method, level_or_accel, di, stride, block_size, nullptr, (uint32_t *) (di + cnt * stride),
                         (uint32_t *) (hi + cnt * stride), first_blkno, alloc, page_ptr, arg, created_xid, npages, comp_size,
                         status, h2d, d2h);
        if (rc != CRYOGPU_OK)
            return rc;
    }
    ctx->last_h2d = h2d;
    ctx->last_d2h = d2h;
    return CRYOGPU_OK;
}

/* ------------------------------------------------ cryo blocks from packed tuples */

/* entry (off, len) of a batch whose data is data_size bytes: can its tuple go into a block of block_size bytes? */
static bool
entry_in_data(uint64_t off, uint32_t len, uint64_t data_size, uint32_t block_size)
{
    return off != UINT64_MAX && len <= block_size && off <= data_size && len <= data_size - off;
}

extern "C" int
cryogpu_build_blocks_device(cryogpu_ctx *ctx, size_t n, const uint8_t *d_data, uint64_t data_size, const uint64_t *d_tup_off,
                            const uint32_t *d_tup_len, const uint64_t *d_block_first, uint32_t block_size, uint8_t *d_dst,
                            uint64_t dst_stride, int32_t *d_status, void *stream)
{
    if (!ctx)
        return fail(CRYOGPU_E_ARG, "ctx is NULL");
    if (block_size < 16 || block_size > (1u << 27) || (block_size & 7) || n > 0x7fffffffu)
        return fail(CRYOGPU_E_ARG, "block_size must be a multiple of 8 in [16, 128 MiB]");
    if (n == 0)
        return CRYOGPU_OK;
    if ((data_size && !d_data) || !d_tup_off || !d_tup_len || !d_block_first || !d_dst || !d_status)
        return fail(CRYOGPU_E_ARG, "NULL device pointer");
    if (((uintptr_t) d_dst & 15) || (dst_stride & 15) || dst_stride < block_size || ((uintptr_t) d_tup_off & 7) ||
        ((uintptr_t) d_block_first & 7) || ((uintptr_t) d_tup_len & 3))
        return fail(CRYOGPU_E_ARG, "d_dst, dst_stride multiples of 16, stride >= block_size; tup_off, block_first 8-byte aligned");
    cudaStream_t st = stream ? (cudaStream_t) stream : ctx->stream;

    CU(cudaSetDevice(ctx->device));
    std::lock_guard<std::recursive_mutex> g(ctx->mu);

    CU(cudaStreamWaitEvent(st, ctx->busy, 0));
    k_block_build<<<(unsigned) n, BLK_THREADS, BLK_SMEM, st>>>(d_data, 0, data_size, (const tup_u64 *) d_tup_off, d_tup_len,
                                                              (const tup_u64 *) d_block_first, block_size, d_dst, dst_stride,
                                                              d_status);
    CU(cudaGetLastError());
    CU(cudaEventRecord(ctx->busy, st));
    return CRYOGPU_OK;
}

/*
 * The COPY flush from packed tuples.  Per chunk the bus carries the chunk's entries, its block_first row and the byte
 * span of data its well-formed entries cover (for a writer that appends in order: exactly the chunk's tuples, about
 * 22 KB per block of narrow rows against the 1 MiB image); the blocks are built in HBM and go through flush_chunk.
 */
extern "C" int
cryogpu_compress_tuples_pages_alloc_host(cryogpu_ctx *ctx, size_t n, int method, int level_or_accel, const void *data,
                                         uint64_t data_size, const uint64_t *tup_off, const uint32_t *tup_len,
                                         const uint64_t *block_first, uint32_t block_size, const uint32_t *first_blkno,
                                         cryogpu_alloc_page_fn alloc, cryogpu_page_ptr_fn page_ptr, void *arg,
                                         uint32_t created_xid, uint32_t *npages, uint32_t *comp_size, int32_t *status)
{
    if (!ctx)
        return fail(CRYOGPU_E_ARG, "ctx is NULL");
    if (method != CRYOGPU_LZ4 && method != CRYOGPU_ZSTD)
        return fail(CRYOGPU_E_METHOD, "unknown compression method %d", method);
    if (block_size < 16 || block_size > (1u << 27) || (block_size & 7))
        return fail(CRYOGPU_E_ARG, "block_size must be a multiple of 8 in [16, 128 MiB]");
    if (n == 0)
        return CRYOGPU_OK;
    if (!block_first || !first_blkno || !alloc || !page_ptr || !npages || !comp_size || !status)
        return fail(CRYOGPU_E_ARG, "NULL argument");
    for (size_t i = 0; i < n; i++)
        if (block_first[i + 1] < block_first[i])
            return fail(CRYOGPU_E_ARG, "block_first must not decrease");
    if (block_first[n] > block_first[0] && (!tup_off || !tup_len || (data_size && !data)))
        return fail(CRYOGPU_E_ARG, "NULL argument");
    const uint64_t stride = ((uint64_t) block_size + 15) & ~(uint64_t) 15;
    const uint32_t cap_pages = pg_pages_needed(cryogpu_compress_bound(method, block_size));
    uint64_t       h2d = 0, d2h = 0;
    std::lock_guard<std::recursive_mutex> hold(ctx->mu);

    CU(cudaSetDevice(ctx->device));
    const bool data_pinned = data && is_pinned(data), ent_pinned = tup_off && is_pinned(tup_off) && is_pinned(tup_len);

    for (size_t lo = 0; lo < n; lo += PG_HOST_CHUNK)
    {
        const size_t   cnt = std::min<size_t>(PG_HOST_CHUNK, n - lo);
        const uint64_t e0 = block_first[lo], ne = block_first[lo + cnt] - e0;
        uint64_t       b0 = UINT64_MAX, b1 = 0;

        /* the bytes the chunk's well-formed entries cover, from a 16-byte boundary (the kernel rejects the others) */
        for (uint64_t e = e0; e < e0 + ne; e++)
            if (tup_len[e] && entry_in_data(tup_off[e], tup_len[e], data_size, block_size))
            {
                b0 = std::min(b0, tup_off[e]);
                b1 = std::max(b1, tup_off[e] + tup_len[e]);
            }
        b0 = b0 == UINT64_MAX ? 0 : b0 & ~(uint64_t) 15;
        b1 = std::max(b0, b1);
        /* device: blocks | page rows | block_first (cnt + 1) | tup_off | tup_len | status | span (+ 16: the copies read
         * whole aligned words); pinned staging: page rows | block_first | tup_off, tup_len, span if the caller's are not */
        const size_t blk_bytes = tp_al(cnt * cap_pages * 4), bf_bytes = tp_al((cnt + 1) * 8), to_bytes = tp_al(ne * 8),
                     tl_bytes = tp_al(ne * 4), st_bytes = tp_al(cnt * 4), span = b1 - b0, sp_bytes = tp_al(span + 16);
        const size_t d_total = cnt * stride + blk_bytes + bf_bytes + to_bytes + tl_bytes + st_bytes + sp_bytes;
        const size_t h_total = blk_bytes + bf_bytes + (ent_pinned ? 0 : to_bytes + tl_bytes) + (data_pinned ? 0 : sp_bytes);
        int          rc;

        if ((rc = host_reserve(ctx->h_in[0], h_total)) != CRYOGPU_OK || (rc = dev_reserve(ctx->d_in[0], d_total)) != CRYOGPU_OK)
            return rc;
        uint8_t  *hi = (uint8_t *) ctx->h_in[0].p, *di = (uint8_t *) ctx->d_in[0].p;
        uint32_t *d_blk = (uint32_t *) (di + cnt * stride);
        uint64_t *d_bf = (uint64_t *) ((uint8_t *) d_blk + blk_bytes), *d_to = (uint64_t *) ((uint8_t *) d_bf + bf_bytes);
        uint32_t *d_tl = (uint32_t *) ((uint8_t *) d_to + to_bytes);
        int32_t  *d_bst = (int32_t *) ((uint8_t *) d_tl + tl_bytes);
        uint8_t  *d_span = (uint8_t *) d_bst + st_bytes;
        uint64_t *h_bf = (uint64_t *) (hi + blk_bytes);
        uint8_t  *h_rest = (uint8_t *) h_bf + bf_bytes;
        const uint64_t *src_to = tup_off + e0;
        const uint32_t *src_tl = tup_len + e0;
        const uint8_t  *src_span = (const uint8_t *) data + b0;

        for (size_t i = 0; i <= cnt; i++)
            h_bf[i] = block_first[lo + i] - e0;
        if (!ent_pinned && ne)
        {
            memcpy(h_rest, src_to, ne * 8);
            memcpy(h_rest + to_bytes, src_tl, ne * 4);
            src_to = (const uint64_t *) h_rest;
            src_tl = (const uint32_t *) (h_rest + to_bytes);
            h_rest += to_bytes + tl_bytes;
        }
        if (!data_pinned && span)
        {
            host_pool(ctx)->run((span + (1u << 20) - 1) >> 20, [&](size_t part) {
                const size_t at = part << 20;

                memcpy(h_rest + at, src_span + at, std::min<size_t>(1u << 20, span - at));
            });
            src_span = h_rest;
        }
        CU(cudaMemcpyAsync(d_bf, h_bf, (cnt + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
        h2d += (cnt + 1) * 8;
        if (ne)
        {
            CU(cudaMemcpyAsync(d_to, src_to, ne * 8, cudaMemcpyHostToDevice, ctx->stream));
            CU(cudaMemcpyAsync(d_tl, src_tl, ne * 4, cudaMemcpyHostToDevice, ctx->stream));
            h2d += ne * 12;
        }
        if (span)
        {
            CU(cudaMemcpyAsync(d_span, src_span, span, cudaMemcpyHostToDevice, ctx->stream));
            h2d += span;
        }
        CU(cudaStreamWaitEvent(ctx->stream, ctx->busy, 0));
        k_block_build<<<(unsigned) cnt, BLK_THREADS, BLK_SMEM, ctx->stream>>>(d_span, b0, data_size, (const tup_u64 *) d_to, d_tl,
                                                                             (const tup_u64 *) d_bf, block_size, di, stride,
                                                                             d_bst);
        CU(cudaGetLastError());
        rc = flush_chunk(ctx, lo, cnt, method, level_or_accel, di, stride, block_size, d_bst, d_blk, (uint32_t *) hi, first_blkno,
                         alloc, page_ptr, arg, created_xid, npages, comp_size, status, h2d, d2h);
        if (rc != CRYOGPU_OK)
            return rc;
    }
    ctx->last_h2d = h2d;
    ctx->last_d2h = d2h;
    return CRYOGPU_OK;
}

/* ----------------------------------------------------- tuple-level work (f-4) */

extern "C" int
cryogpu_tuple_stats_device(cryogpu_ctx *ctx, size_t n, const uint8_t *d_blocks, uint64_t stride, uint32_t block_size,
                           const int32_t *d_status, uint32_t *d_ntuples, uint64_t *d_tuple_bytes, int32_t *d_valid,
                           void *stream)
{
    if (!ctx)
        return fail(CRYOGPU_E_ARG, "ctx is NULL");
    if (n == 0)
        return CRYOGPU_OK;
    if (!d_blocks || !d_ntuples || !d_tuple_bytes || !d_valid)
        return fail(CRYOGPU_E_ARG, "NULL device pointer");
    if (((uintptr_t) d_blocks & 7) || (stride & 7) || block_size < 16 || stride < block_size || n > 0x7fffffffu)
        return fail(CRYOGPU_E_ARG, "blocks must be 8-byte aligned, block_size >= 16, stride >= block_size");
    cudaStream_t st = stream ? (cudaStream_t) stream : ctx->stream;

    CU(cudaSetDevice(ctx->device));
    k_tuple_stats<<<(unsigned) ((n + 7) / 8), 256, 0, st>>>(d_blocks, stride, block_size, d_status, d_ntuples,
                                                            (unsigned long long *) d_tuple_bytes, d_valid, (uint32_t) n);
    CU(cudaGetLastError());
    return CRYOGPU_OK;
}

/*
 * Count pushdown for the host-pointer caller: compressed blocks in, per block the number of tuples, their
 * bytes and the decode status out; the decoded blocks never leave HBM.
 */
extern "C" int
cryogpu_decompress_count_host(cryogpu_ctx *ctx, size_t n, const int32_t *methods, const void *const *src,
                              const uint32_t *src_size, uint32_t block_size, uint32_t *ntuples, uint64_t *tuple_bytes,
                              int32_t *status)
{
    if (!ctx)
        return fail(CRYOGPU_E_ARG, "ctx is NULL");
    if (n == 0)
        return CRYOGPU_OK;
    if (!methods || !src || !src_size || !ntuples || !tuple_bytes || !status)
        return fail(CRYOGPU_E_ARG, "NULL argument");
    if (block_size < 16 || block_size > (1u << 27))
        return fail(CRYOGPU_E_ARG, "block_size out of range");
    const uint64_t stride = ((uint64_t) block_size + 15) & ~(uint64_t) 15;
    const size_t   chunk = 512;
    uint64_t       h2d = 0, d2h = 0;
    std::lock_guard<std::recursive_mutex> hold(ctx->mu);

    CU(cudaSetDevice(ctx->device));
    for (size_t lo = 0; lo < n; lo += chunk)
    {
        const size_t cnt = std::min(chunk, n - lo);
        size_t       in_bytes = 0;

        for (size_t i = 0; i < cnt; i++)
            in_bytes += ((size_t) src_size[lo + i] + 15) & ~(size_t) 15;
        /* staging in: streams | offsets u64 | sizes u32 | methods i32 ; out: ntuples u32 | status i32 | valid i32 | bytes u64 */
        const size_t in_al = (in_bytes + 255) & ~(size_t) 255, meta_in = cnt * 16, meta_out = cnt * 24;
        int          rc;

        if ((rc = host_reserve(ctx->h_in[0], in_al + meta_in + 16)) != CRYOGPU_OK ||
            (rc = dev_reserve(ctx->d_in[0], in_al + meta_in + 16)) != CRYOGPU_OK ||
            (rc = host_reserve(ctx->h_out[0], meta_out)) != CRYOGPU_OK ||
            (rc = dev_reserve(ctx->d_out[0], cnt * stride + meta_out)) != CRYOGPU_OK)
            return rc;
        uint8_t  *hi = (uint8_t *) ctx->h_in[0].p, *di = (uint8_t *) ctx->d_in[0].p, *dout = (uint8_t *) ctx->d_out[0].p;
        uint64_t *h_off = (uint64_t *) (hi + in_al);
        uint32_t *h_sz = (uint32_t *) (hi + in_al + cnt * 8);
        int32_t  *h_me = (int32_t *) (hi + in_al + cnt * 12);
        size_t    at = 0;

        for (size_t i = 0; i < cnt; i++)
        {
            memcpy(hi + at, src[lo + i], src_size[lo + i]);
            h_off[i] = at;
            h_sz[i] = src_size[lo + i];
            h_me[i] = methods[lo + i];
            at += ((size_t) src_size[lo + i] + 15) & ~(size_t) 15;
        }
        CU(cudaMemcpyAsync(di, hi, in_al + meta_in, cudaMemcpyHostToDevice, ctx->stream));
        h2d += in_al + meta_in;
        uint8_t  *dm = dout + cnt * stride;
        uint32_t *d_nt = (uint32_t *) dm;
        int32_t  *d_st = (int32_t *) (dm + cnt * 4), *d_ok = (int32_t *) (dm + cnt * 8);
        uint64_t *d_by = (uint64_t *) (dm + cnt * 16);          /* cnt * 12 rounded up to 8-byte alignment: cnt * 16 */
        uint32_t *d_osz = (uint32_t *) (dm + cnt * 12);

        CU(cudaStreamWaitEvent(ctx->stream, ctx->busy, 0));
        rc = decompress_device_locked(ctx, ctx->stream, cnt, (int32_t *) (di + in_al + cnt * 12), di, (uint64_t *) (di + in_al),
                                      (uint32_t *) (di + in_al + cnt * 8), dout, stride, block_size, d_osz, d_st);
        if (rc != CRYOGPU_OK)
            return rc;
        k_tuple_stats<<<(unsigned) ((cnt + 7) / 8), 256, 0, ctx->stream>>>(dout, stride, block_size, d_st, d_nt,
                                                                          (unsigned long long *) d_by, d_ok, (uint32_t) cnt);
        CU(cudaGetLastError());
        CU(cudaEventRecord(ctx->busy, ctx->stream));
        CU(cudaMemcpyAsync(ctx->h_out[0].p, dm, meta_out, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        d2h += meta_out;
        const uint8_t *hm = (const uint8_t *) ctx->h_out[0].p;

        memcpy(ntuples + lo, hm, cnt * 4);
        memcpy(status + lo, hm + cnt * 4, cnt * 4);
        memcpy(tuple_bytes + lo, hm + cnt * 16, cnt * 8);
        /* a decoded block whose item ids point outside it is reported as malformed */
        const int32_t *h_ok = (const int32_t *) (hm + cnt * 8);

        for (size_t i = 0; i < cnt; i++)
            if (status[lo + i] == CRYOGPU_ST_OK && !h_ok[i])
                status[lo + i] = CRYOGPU_ST_FORMAT;
    }
    ctx->last_h2d = h2d;
    ctx->last_d2h = d2h;
    return CRYOGPU_OK;
}

/* ------------------------------------------------------- batched tuple fetch */

static size_t
tp_al(size_t v)
{
    return (v + 255) & ~(size_t) 255;
}

/*
 * Select and scan of one batch on st (ctx->mu held, st ordered after ctx->busy).  work: 4n + 4 words of the context's
 * tuple area: cnt[n] | bytes[n] | byte_first[n + 1] | (room for block_first[n + 1] and need[2] of the host calls).
 */
static int
tuples_place(cudaStream_t st, size_t n, const uint8_t *d_blocks, uint64_t stride, uint32_t block_size,
             const int32_t *d_block_status, const tup_u64 *d_sel_off, const uint32_t *d_sel_pos, uint64_t ent0, uint64_t byte0,
             uint64_t data_cap, uint64_t tup_cap, tup_u64 *d_block_first, int32_t *d_status, tup_u64 *d_need, tup_u64 *work)
{
    if (n)
        k_tuple_select<<<(unsigned) ((n + 7) / 8), 256, 0, st>>>(d_blocks, stride, block_size, d_block_status, d_sel_off,
                                                                 d_sel_pos, work, work + n, d_status, (uint32_t) n);
    k_tuple_scan<<<1, TUP_SCAN_THREADS, 64 * sizeof(tup_u64), st>>>((uint32_t) n, work, work + n, d_status, ent0, byte0, tup_cap,
                                                                    data_cap, d_block_first, work + 2 * n, d_need);
    CU(cudaGetLastError());
    return CRYOGPU_OK;
}

static int
tuples_gather(cudaStream_t st, size_t n, const uint8_t *d_blocks, uint64_t stride, uint32_t block_size, const int32_t *d_status,
              const tup_u64 *d_sel_off, const uint32_t *d_sel_pos, const tup_u64 *d_block_first, const tup_u64 *work, TupOut o)
{
    if (n)
        k_tuple_gather<<<(unsigned) ((n + 7) / 8), 256, 0, st>>>(d_blocks, stride, block_size, d_status, d_sel_off, d_sel_pos,
                                                                 d_block_first, work + 2 * n, o, (uint32_t) n);
    CU(cudaGetLastError());
    return CRYOGPU_OK;
}

extern "C" int
cryogpu_tuples_device(cryogpu_ctx *ctx, size_t n, const uint8_t *d_blocks, uint64_t stride, uint32_t block_size,
                      const int32_t *d_block_status, const uint64_t *d_sel_off, const uint32_t *d_sel_pos, uint8_t *d_data,
                      uint64_t data_cap, uint64_t *d_tup_off, uint32_t *d_tup_len, uint64_t tup_cap, uint64_t *d_block_first,
                      int32_t *d_status, uint64_t *d_need, void *stream)
{
    if (!ctx)
        return fail(CRYOGPU_E_ARG, "ctx is NULL");
    if (!d_blocks || !d_block_first || !d_status || !d_need || (d_sel_off && !d_sel_pos) || (data_cap && !d_data) ||
        (tup_cap && (!d_tup_off || !d_tup_len)))
        return fail(CRYOGPU_E_ARG, "NULL device pointer");
    if (((uintptr_t) d_blocks & 7) || (stride & 7) || block_size < 16 || block_size > (1u << 27) || stride < block_size ||
        ((uintptr_t) d_data & 15) || ((uintptr_t) d_tup_off & 7) || ((uintptr_t) d_block_first & 7) ||
        ((uintptr_t) d_sel_off & 7) || ((uintptr_t) d_need & 7) || n > 0x7fffffffu)
        return fail(CRYOGPU_E_ARG, "blocks, stride, block_first, sel_off, tup_off 8-byte aligned, data 16-byte aligned, "
                                   "16 <= block_size <= stride");
    cudaStream_t st = stream ? (cudaStream_t) stream : ctx->stream;

    CU(cudaSetDevice(ctx->device));
    std::lock_guard<std::recursive_mutex> g(ctx->mu);

    CU(cudaStreamWaitEvent(st, ctx->busy, 0));
    int rc = dev_reserve(ctx->tpw, (4 * n + 4) * sizeof(tup_u64));

    if (rc != CRYOGPU_OK)
        return rc;
    tup_u64 *work = (tup_u64 *) ctx->tpw.p;
    const TupOut o = {d_data, (tup_u64 *) d_tup_off, d_tup_len, 0, 0};

    if ((rc = tuples_place(st, n, d_blocks, stride, block_size, d_block_status, (const tup_u64 *) d_sel_off, d_sel_pos, 0, 0,
                           data_cap, tup_cap, (tup_u64 *) d_block_first, d_status, (tup_u64 *) d_need, work)) != CRYOGPU_OK ||
        (rc = tuples_gather(st, n, d_blocks, stride, block_size, d_status, (const tup_u64 *) d_sel_off, d_sel_pos,
                            (const tup_u64 *) d_block_first, work, o)) != CRYOGPU_OK)
        return rc;
    CU(cudaEventRecord(ctx->busy, st));
    return CRYOGPU_OK;
}

/*
 * Tuple fetch of one chunk of a host call, blocks [lo, lo + cnt), decoded into d_blocks with their statuses in d_st by
 * work already enqueued on ctx->stream (ctx->mu held).  Entries and bytes continue from ent_base / byte_base, which
 * advance by what the chunk needs.  Two round trips: the placement (so that only the bytes that fit are staged and
 * copied), then the packed tuples, straight into the caller's buffers when they are pinned.
 */
static int
tuples_chunk_host(cryogpu_ctx *ctx, size_t lo, size_t cnt, const uint8_t *d_blocks, uint64_t stride, uint32_t block_size,
                  int32_t *d_st, const uint64_t *sel_off, const uint32_t *sel_pos, void *data, uint64_t data_cap,
                  uint64_t *tup_off, uint32_t *tup_len, uint64_t tup_cap, uint64_t *block_first, int32_t *status,
                  uint64_t &ent_base, uint64_t &byte_base, uint64_t &h2d, uint64_t &d2h)
{
    const size_t m = sel_off ? (size_t) (sel_off[lo + cnt] - sel_off[lo]) : 0;
    const size_t work_bytes = tp_al((4 * cnt + 4) * 8), sel_bytes = sel_off ? tp_al((cnt + 1) * 8) + tp_al(m * 4 + 4) : 0;
    const size_t meta_words = 2 * (cnt + 1) + 2;        /* byte_first | block_first | need */
    int          rc;

    if ((rc = dev_reserve(ctx->tpw, work_bytes + sel_bytes)) != CRYOGPU_OK ||
        (rc = host_reserve(ctx->h_tpw, sel_bytes + meta_words * 8 + cnt * 4)) != CRYOGPU_OK)
        return rc;
    tup_u64 *work = (tup_u64 *) ctx->tpw.p, *d_sel_off = nullptr;
    uint32_t *d_sel_pos = nullptr;
    uint8_t  *hw = (uint8_t *) ctx->h_tpw.p, *hm = hw + sel_bytes;

    if (sel_off)
    {
        uint64_t *hs = (uint64_t *) hw;

        for (size_t i = 0; i <= cnt; i++)
            hs[i] = sel_off[lo + i] - sel_off[lo];
        memcpy(hw + tp_al((cnt + 1) * 8), sel_pos + sel_off[lo], m * 4);
        d_sel_off = (tup_u64 *) ((uint8_t *) work + work_bytes);
        d_sel_pos = (uint32_t *) ((uint8_t *) d_sel_off + tp_al((cnt + 1) * 8));
        CU(cudaMemcpyAsync(d_sel_off, hw, sel_bytes, cudaMemcpyHostToDevice, ctx->stream));
        h2d += sel_bytes;
    }
    tup_u64 *d_bf = work + 3 * cnt + 1, *d_need = d_bf + cnt + 1;

    rc = tuples_place(ctx->stream, cnt, d_blocks, stride, block_size, d_st, d_sel_off, d_sel_pos, ent_base, byte_base, data_cap,
                      tup_cap, d_bf, d_st, d_need, work);
    if (rc != CRYOGPU_OK)
        return rc;
    CU(cudaMemcpyAsync(hm, work + 2 * cnt, meta_words * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaMemcpyAsync(hm + meta_words * 8, d_st, cnt * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    d2h += meta_words * 8 + cnt * 4;
    const uint64_t *h_byte_first = (const uint64_t *) hm, *h_bf = h_byte_first + cnt + 1, *h_need = h_bf + cnt + 1;
    const int32_t  *h_st = (const int32_t *) (hm + meta_words * 8);
    uint64_t        fit_e = 0, fit_b = 0;

    /* the blocks that fit: one range of entries and bytes from ent_base / byte_base (once a block crosses a capacity,
     * every later block with entries does) */
    for (size_t i = 0; i < cnt; i++)
        if (h_st[i] == CRYOGPU_ST_OK && h_bf[i + 1] > h_bf[i])
        {
            fit_e = h_bf[i + 1] - ent_base;
            fit_b = h_byte_first[i + 1] - byte_base;
        }
    if (fit_e)
    {
        const size_t db = tp_al(fit_b), ob = tp_al(fit_e * 8), total = db + ob + fit_e * 4;
        const bool   direct = is_pinned(data) && is_pinned(tup_off) && is_pinned(tup_len);

        if ((rc = dev_reserve(ctx->tpo, total)) != CRYOGPU_OK || (!direct && (rc = host_reserve(ctx->h_tpo, total)) != CRYOGPU_OK))
            return rc;
        uint8_t     *o = (uint8_t *) ctx->tpo.p;
        const TupOut to = {o, (tup_u64 *) (o + db), (uint32_t *) (o + db + ob), ent_base, byte_base};

        if ((rc = tuples_gather(ctx->stream, cnt, d_blocks, stride, block_size, d_st, d_sel_off, d_sel_pos, d_bf, work, to)) !=
            CRYOGPU_OK)
            return rc;
        if (direct)
        {
            CU(cudaMemcpyAsync((uint8_t *) data + byte_base, o, fit_b, cudaMemcpyDeviceToHost, ctx->stream));
            CU(cudaMemcpyAsync(tup_off + ent_base, o + db, fit_e * 8, cudaMemcpyDeviceToHost, ctx->stream));
            CU(cudaMemcpyAsync(tup_len + ent_base, o + db + ob, fit_e * 4, cudaMemcpyDeviceToHost, ctx->stream));
            CU(cudaStreamSynchronize(ctx->stream));
        }
        else
        {
            uint8_t *h = (uint8_t *) ctx->h_tpo.p;

            CU(cudaMemcpyAsync(h, o, fit_b, cudaMemcpyDeviceToHost, ctx->stream));
            CU(cudaMemcpyAsync(h + db, o + db, ob + fit_e * 4, cudaMemcpyDeviceToHost, ctx->stream));
            CU(cudaStreamSynchronize(ctx->stream));
            memcpy((uint8_t *) data + byte_base, h, fit_b);
            memcpy(tup_off + ent_base, h + db, fit_e * 8);
            memcpy(tup_len + ent_base, h + db + ob, fit_e * 4);
        }
        d2h += fit_b + fit_e * 12;
    }
    CU(cudaEventRecord(ctx->busy, ctx->stream));
    memcpy(status + lo, h_st, cnt * 4);
    memcpy(block_first + lo, h_bf, cnt * 8);
    ent_base += h_need[1];
    byte_base += h_need[0];
    return CRYOGPU_OK;
}

static int
check_tuples_host_args(const cryogpu_ctx *ctx, uint32_t block_size, const uint64_t *sel_off, const uint32_t *sel_pos,
                       const void *data, uint64_t data_cap, const uint64_t *tup_off, const uint32_t *tup_len, uint64_t tup_cap,
                       const uint64_t *block_first, const int32_t *status, const uint64_t *need)
{
    if (!ctx)
        return fail(CRYOGPU_E_ARG, "ctx is NULL");
    if (!block_first || !status || !need || (sel_off && !sel_pos) || (data_cap && !data) || (tup_cap && (!tup_off || !tup_len)))
        return fail(CRYOGPU_E_ARG, "NULL argument");
    if (block_size < 16 || block_size > (1u << 27))
        return fail(CRYOGPU_E_ARG, "block_size out of range");
    return CRYOGPU_OK;
}

#define TUP_HOST_CHUNK 256u

extern "C" int
cryogpu_decompress_tuples_host(cryogpu_ctx *ctx, size_t n, const int32_t *methods, const void *const *src,
                               const uint32_t *src_size, uint32_t block_size, const uint64_t *sel_off, const uint32_t *sel_pos,
                               void *data, uint64_t data_cap, uint64_t *tup_off, uint32_t *tup_len, uint64_t tup_cap,
                               uint64_t *block_first, int32_t *status, uint64_t *need)
{
    int rc = check_tuples_host_args(ctx, block_size, sel_off, sel_pos, data, data_cap, tup_off, tup_len, tup_cap, block_first,
                                    status, need);

    if (rc != CRYOGPU_OK)
        return rc;
    if (n && (!methods || !src || !src_size))
        return fail(CRYOGPU_E_ARG, "NULL argument");
    const uint64_t stride = ((uint64_t) block_size + 15) & ~(uint64_t) 15;
    uint64_t       h2d = 0, d2h = 0, ent = 0, bytes = 0;
    std::lock_guard<std::recursive_mutex> hold(ctx->mu);

    CU(cudaSetDevice(ctx->device));
    for (size_t lo = 0; lo < n; lo += TUP_HOST_CHUNK)
    {
        const size_t cnt = std::min<size_t>(TUP_HOST_CHUNK, n - lo);
        size_t       in_bytes = 0;

        for (size_t i = 0; i < cnt; i++)
            in_bytes += ((size_t) src_size[lo + i] + 15) & ~(size_t) 15;
        /* staging in: streams | offsets u64 | sizes u32 | methods i32 ; device out: blocks | out_size u32 | status i32 */
        const size_t in_al = tp_al(in_bytes), meta_in = cnt * 16;

        if ((rc = host_reserve(ctx->h_in[0], in_al + meta_in + 16)) != CRYOGPU_OK ||
            (rc = dev_reserve(ctx->d_in[0], in_al + meta_in + 16)) != CRYOGPU_OK ||
            (rc = dev_reserve(ctx->d_out[0], cnt * stride + cnt * 8)) != CRYOGPU_OK)
            return rc;
        uint8_t  *hi = (uint8_t *) ctx->h_in[0].p, *di = (uint8_t *) ctx->d_in[0].p, *dout = (uint8_t *) ctx->d_out[0].p;
        uint64_t *h_off = (uint64_t *) (hi + in_al);
        uint32_t *h_sz = (uint32_t *) (hi + in_al + cnt * 8);
        int32_t  *h_me = (int32_t *) (hi + in_al + cnt * 12);
        size_t    at = 0;

        for (size_t i = 0; i < cnt; i++)
        {
            memcpy(hi + at, src[lo + i], src_size[lo + i]);
            h_off[i] = at;
            h_sz[i] = src_size[lo + i];
            h_me[i] = methods[lo + i];
            at += ((size_t) src_size[lo + i] + 15) & ~(size_t) 15;
        }
        CU(cudaMemcpyAsync(di, hi, in_al + meta_in, cudaMemcpyHostToDevice, ctx->stream));
        h2d += in_al + meta_in;
        uint32_t *d_osz = (uint32_t *) (dout + cnt * stride);
        int32_t  *d_st = (int32_t *) (dout + cnt * stride + cnt * 4);

        CU(cudaStreamWaitEvent(ctx->stream, ctx->busy, 0));
        rc = decompress_device_locked(ctx, ctx->stream, cnt, (int32_t *) (di + in_al + cnt * 12), di, (uint64_t *) (di + in_al),
                                      (uint32_t *) (di + in_al + cnt * 8), dout, stride, block_size, d_osz, d_st);
        if (rc != CRYOGPU_OK)
            return rc;
        rc = tuples_chunk_host(ctx, lo, cnt, dout, stride, block_size, d_st, sel_off, sel_pos, data, data_cap, tup_off, tup_len,
                               tup_cap, block_first, status, ent, bytes, h2d, d2h);
        if (rc != CRYOGPU_OK)
            return rc;
    }
    block_first[n] = ent;
    need[0] = bytes;
    need[1] = ent;
    ctx->last_h2d = h2d;
    ctx->last_d2h = d2h;
    return CRYOGPU_OK;
}

extern "C" int
cryogpu_decompress_pages_tuples_host(cryogpu_ctx *ctx, size_t n, const void *const *pages, const uint32_t *page_blkno,
                                     const uint32_t *chain_off, uint32_t block_size, const uint64_t *sel_off,
                                     const uint32_t *sel_pos, void *data, uint64_t data_cap, uint64_t *tup_off,
                                     uint32_t *tup_len, uint64_t tup_cap, uint64_t *block_first, int32_t *status,
                                     int32_t *methods, uint32_t *comp_size, uint64_t *need)
{
    int rc = check_tuples_host_args(ctx, block_size, sel_off, sel_pos, data, data_cap, tup_off, tup_len, tup_cap, block_first,
                                    status, need);

    if (rc != CRYOGPU_OK)
        return rc;
    if (n && (!pages || !page_blkno || !chain_off || !methods))
        return fail(CRYOGPU_E_ARG, "NULL argument");
    const uint64_t stride = ((uint64_t) block_size + 15) & ~(uint64_t) 15;
    uint64_t       h2d = 0, d2h = 0, ent = 0, bytes = 0;
    std::lock_guard<std::recursive_mutex> hold(ctx->mu);

    CU(cudaSetDevice(ctx->device));
    for (size_t lo = 0; lo < n; lo += PG_HOST_CHUNK)
    {
        const size_t   cnt = std::min<size_t>(PG_HOST_CHUNK, n - lo);
        const uint32_t e0 = chain_off[lo], e1 = chain_off[lo + cnt], ne = e1 - e0;

        if (e1 < e0)
            return fail(CRYOGPU_E_ARG, "chain_off must not decrease");
        if (ne == 0)
        {
            for (size_t i = 0; i < cnt; i++)
            {
                status[lo + i] = CRYOGPU_ST_EMPTY_BLOCK;
                block_first[lo + i] = ent;
                methods[lo + i] = 0;
                if (comp_size)
                    comp_size[lo + i] = 0;
            }
            continue;
        }
        /* staging in: pages | slot | blkno | chain_off (cnt + 1); device out: blocks | out_size | status | methods | comp_size */
        const size_t pg_bytes = (size_t) ne * PG_PAGE, meta_in = tp_al((size_t) ne * 8 + (cnt + 1) * 4);

        if ((rc = host_reserve(ctx->h_in[0], pg_bytes + meta_in)) != CRYOGPU_OK ||
            (rc = dev_reserve(ctx->d_in[0], pg_bytes + meta_in)) != CRYOGPU_OK ||
            (rc = host_reserve(ctx->h_out[0], cnt * 8)) != CRYOGPU_OK ||
            (rc = dev_reserve(ctx->d_out[0], cnt * stride + cnt * 16)) != CRYOGPU_OK)
            return rc;
        uint8_t  *hi = (uint8_t *) ctx->h_in[0].p, *di = (uint8_t *) ctx->d_in[0].p, *dout = (uint8_t *) ctx->d_out[0].p;
        uint32_t *h_slot = (uint32_t *) (hi + pg_bytes), *h_blk = h_slot + ne, *h_coff = h_blk + ne;

        host_pool(ctx)->run((ne + 255) / 256, [&](size_t part) {
            for (uint32_t e = (uint32_t) part * 256u; e < ne && e < (uint32_t) (part + 1) * 256u; e++)
            {
                memcpy(hi + (size_t) e * PG_PAGE, pages[e0 + e], PG_PAGE);
                h_slot[e] = e;
                h_blk[e] = page_blkno[e0 + e];
            }
        });
        for (size_t i = 0; i <= cnt; i++)
            h_coff[i] = chain_off[lo + i] - e0;
        CU(cudaMemcpyAsync(di, hi, pg_bytes + meta_in, cudaMemcpyHostToDevice, ctx->stream));
        h2d += pg_bytes + meta_in;
        uint8_t *dm = dout + cnt * stride;
        int32_t *d_st = (int32_t *) (dm + cnt * 4);

        rc = cryogpu_decompress_pages_device(ctx, cnt, di, (uint32_t *) (di + pg_bytes), (uint32_t *) (di + pg_bytes) + ne,
                                             (uint32_t *) (di + pg_bytes) + 2 * (size_t) ne, ne, dout, stride, block_size,
                                             (uint32_t *) dm, d_st, (int32_t *) (dm + cnt * 8), (uint32_t *) (dm + cnt * 12),
                                             ctx->stream);
        if (rc != CRYOGPU_OK)
            return rc;
        /* methods | comp_size: read once the chunk's tuples are back (tuples_chunk_host waits for the stream) */
        CU(cudaMemcpyAsync(ctx->h_out[0].p, dm + cnt * 8, cnt * 8, cudaMemcpyDeviceToHost, ctx->stream));
        d2h += cnt * 8;
        rc = tuples_chunk_host(ctx, lo, cnt, dout, stride, block_size, d_st, sel_off, sel_pos, data, data_cap, tup_off, tup_len,
                               tup_cap, block_first, status, ent, bytes, h2d, d2h);
        if (rc != CRYOGPU_OK)
            return rc;
        memcpy(methods + lo, ctx->h_out[0].p, cnt * 4);
        if (comp_size)
            memcpy(comp_size + lo, (const uint8_t *) ctx->h_out[0].p + cnt * 4, cnt * 4);
    }
    block_first[n] = ent;
    need[0] = bytes;
    need[1] = ent;
    ctx->last_h2d = h2d;
    ctx->last_d2h = d2h;
    return CRYOGPU_OK;
}

/* -------------------------------------------------------------- host API */

/* blocks per pipeline chunk: bounds device/pinned staging to ~128 MiB per lane */
static size_t
chunk_blocks(uint32_t block_size)
{
    size_t c = (128u << 20) / block_size;

    return c < 1 ? 1 : c;
}

/*
 * Chunk of the host decompress call.  A chunk is one batch for the kernels, and a batch of a few hundred
 * blocks or less is latency-bound (a whole table in 128-block chunks spent 12 of its 16 ms there): a large
 * call is cut into about four chunks (two lanes, so copies and kernels still overlap) of at most 1 GiB.
 * CRYOGPU_HOST_CHUNK overrides (blocks).
 */
static size_t
decompress_chunk_blocks(uint32_t block_size, size_t n)
{
    static long forced = -1;

    if (forced < 0)
    {
        const char *e = getenv("CRYOGPU_HOST_CHUNK");

        forced = e && atol(e) > 0 ? atol(e) : 0;
    }
    if (forced)
        return (size_t) forced;
    const size_t lo = chunk_blocks(block_size), hi = std::max<size_t>(lo, ((size_t) 1 << 30) / block_size);

    return std::min(hi, std::max(lo, (n + 3) / 4));
}

static bool
is_pinned(const void *p)
{
    cudaPointerAttributes a;

    if (cudaPointerGetAttributes(&a, p) != cudaSuccess)
    {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost;
}

static bool
sparse_enabled(cryogpu_ctx *ctx)
{
    if (ctx->sparse < 0)
    {
        const char *e = getenv("CRYOGPU_SPARSE_D2H");

        ctx->sparse = (e && strcmp(e, "0") == 0) ? 0 : 1;
    }
    return ctx->sparse == 1;
}

static bool
zero_unmap_enabled(cryogpu_ctx *ctx)
{
    if (ctx->zero_unmap < 0)
    {
        const char *e = getenv("CRYOGPU_ZERO_UNMAP");

        ctx->zero_unmap = (e && strcmp(e, "1") == 0) ? 1 : 0;
    }
    return ctx->zero_unmap == 1;
}

extern "C" int
cryogpu_set_zero_by_unmap(cryogpu_ctx *ctx, int on)
{
    if (!ctx)
        return fail(CRYOGPU_E_ARG, "ctx is NULL");
    ctx->zero_unmap = on ? 1 : 0;
    return CRYOGPU_OK;
}

static HostPool *
host_pool(cryogpu_ctx *ctx)
{
    if (!ctx->pool)
    {
        const char *e = getenv("CRYOGPU_HOST_THREADS");
        int         n = e ? atoi(e) : (int) std::min(16u, std::max(1u, std::thread::hardware_concurrency()));

        ctx->pool = new HostPool();
        ctx->pool->start(n > 1 ? n - 1 : 0);        /* the calling thread works too */
    }
    return ctx->pool;
}

/* zero-fill with non-temporal stores: the run is far larger than any cache and is not read
 * back by this thread, so write-combining avoids the read-for-ownership of every line */
static void
zero_fill(uint8_t *p, size_t n)
{
#ifdef CRYO_HAVE_SSE2
    if (n >= 4096 && ((uintptr_t) p & 15u) == 0)
    {
        const __m128i z = _mm_setzero_si128();
        size_t        i = 0;

        for (; i + 64 <= n; i += 64)
        {
            _mm_stream_si128((__m128i *) (p + i), z);
            _mm_stream_si128((__m128i *) (p + i + 16), z);
            _mm_stream_si128((__m128i *) (p + i + 32), z);
            _mm_stream_si128((__m128i *) (p + i + 48), z);
        }
        _mm_sfence();
        if (i < n)
            memset(p + i, 0, n - i);
        return;
    }
#endif
    memset(p, 0, n);
}

/* place one sparse block: non-zero pages from the packed staging buffer, zeros elsewhere */
/*
 * A run of zero bytes in a caller's block.  unmap (cryogpu_set_zero_by_unmap): the caller has said that its
 * blocks are private anonymous memory (malloc / palloc / .bss: the reference's cache, cache.c:49, is), so the
 * whole OS pages inside the run are given back to the kernel instead of being written: MADV_DONTNEED makes
 * them read as zeros again, on demand, and a scan that only follows item ids never touches them.  The
 * first failure (a locked or special mapping) turns it off for the rest of the call.
 */
static void
zero_range(uint8_t *p, size_t n, std::atomic<int> *unmap)
{
    static const size_t os_page = (size_t) sysconf(_SC_PAGESIZE);

    if (unmap && unmap->load(std::memory_order_relaxed) && n >= 16 * os_page)
    {
        uint8_t *a = (uint8_t *) (((uintptr_t) p + os_page - 1) & ~(uintptr_t) (os_page - 1));
        uint8_t *b = (uint8_t *) (((uintptr_t) p + n) & ~(uintptr_t) (os_page - 1));

        if (b > a && madvise(a, (size_t) (b - a), MADV_DONTNEED) == 0)
        {
            if (a > p)
                memset(p, 0, (size_t) (a - p));
            if (p + n > b)
                memset(b, 0, (size_t) (p + n - b));
            return;
        }
        unmap->store(0, std::memory_order_relaxed);
    }
    zero_fill(p, n);
}

static void
place_sparse_block(uint8_t *dst, uint32_t block_size, const uint32_t *bits, const uint8_t *pages, std::atomic<int> *unmap)
{
    const uint32_t npages = (block_size + SP_PAGE - 1) / SP_PAGE;
    uint32_t       p = 0;

    while (p < npages)
    {
        uint32_t q = p;
        const bool nz = (bits[p >> 5] >> (p & 31)) & 1u;

        while (q < npages && (((bits[q >> 5] >> (q & 31)) & 1u) != 0) == nz)
            q++;
        const size_t lo = (size_t) p * SP_PAGE;
        const size_t hi = std::min<size_t>((size_t) q * SP_PAGE, block_size);

        if (nz)
        {
            memcpy(dst + lo, pages, hi - lo);
            pages += (size_t) (q - p) * SP_PAGE;
        }
        else
            zero_range(dst + lo, hi - lo, unmap);
        p = q;
    }
}

extern "C" int
cryogpu_decompress_host(cryogpu_ctx *ctx, size_t n, const int32_t *methods,
                        const void *const *src, const uint32_t *src_size, void *const *dst,
                        uint32_t block_size, uint32_t *out_size, int32_t *status)
{
    if (!ctx)
        return fail(CRYOGPU_E_ARG, "ctx is NULL");
    if (n == 0)
        return CRYOGPU_OK;
    if (!methods || !src || !src_size || !dst || !out_size || !status)
        return fail(CRYOGPU_E_ARG, "NULL argument");
    if (block_size == 0 || block_size > (1u << 27))
        return fail(CRYOGPU_E_ARG, "block_size out of range");
    std::lock_guard<std::recursive_mutex> g(ctx->mu);

    CU(cudaSetDevice(ctx->device));
    CU(cudaEventSynchronize(ctx->busy));        /* a device-resident call may still be using the work areas */
    const size_t   chunk = decompress_chunk_blocks(block_size, n);
    const uint64_t stride = ((uint64_t) block_size + 15) & ~(uint64_t) 15;
    const bool     dst_pinned = is_pinned(dst[0]);
    /* sparse return pays when a batch is worth a second kernel and blocks have whole pages */
    const bool     sparse = sparse_enabled(ctx) && n >= 4 && block_size >= 16 * SP_PAGE &&
                            block_size <= SP_MAXPAGES * SP_PAGE;
    if (n > chunk)
    {
        int rc = make_lane_streams(ctx, 1);     /* a second chunk will be in flight */

        if (rc != CRYOGPU_OK)
            return rc;
    }
    cudaStream_t   lanes[2] = {ctx->stream, ctx->stream2};
    size_t         pending_lo[2] = {0, 0}, pending_n[2] = {0, 0};
    uint64_t       h2d = 0, d2h = 0;
    std::atomic<int> unmap{zero_unmap_enabled(ctx) && !dst_pinned ? 1 : 0};

    /* dense return of lane l's chunk, enqueued on its stream */
    auto dense_d2h = [&](int l, size_t lo, size_t cnt) -> int {
        cudaStream_t st = lanes[l];

        if (dst_pinned)
        {
            /* straight into the caller's pinned blocks; merge contiguous runs */
            size_t i = 0;

            while (i < cnt)
            {
                size_t j = i + 1;

                while (j < cnt && stride == block_size &&
                       (uint8_t *) dst[lo + j] == (uint8_t *) dst[lo + j - 1] + block_size)
                    j++;
                CU(cudaMemcpyAsync(dst[lo + i], (uint8_t *) ctx->d_out[l].p + i * stride,
                                   (j - i - 1) * stride + block_size, cudaMemcpyDeviceToHost, st));
                i = j;
            }
        }
        else
        {
            int rc = host_reserve(ctx->h_out[l], cnt * stride);

            if (rc != CRYOGPU_OK)
                return rc;
            CU(cudaMemcpyAsync(ctx->h_out[l].p, ctx->d_out[l].p, cnt * stride, cudaMemcpyDeviceToHost, st));
        }
        d2h += cnt * (uint64_t) block_size;
        return CRYOGPU_OK;
    };
    auto dense_finish = [&](int l, size_t lo, size_t cnt) -> int {
        CU(cudaStreamSynchronize(lanes[l]));
        if (!dst_pinned)
            for (size_t i = 0; i < cnt; i++)
                memcpy(dst[lo + i], (uint8_t *) ctx->h_out[l].p + i * stride, block_size);
        return CRYOGPU_OK;
    };

    /* finish a lane: wait, then hand results to the caller */
    auto drain = [&](int l) -> int {
        if (pending_n[l] == 0)
            return CRYOGPU_OK;
        CU(cudaStreamSynchronize(lanes[l]));
        size_t   lo = pending_lo[l], cnt = pending_n[l];
        uint8_t *hm = (uint8_t *) ctx->h_meta[l].p;
        uint32_t *h_osz = (uint32_t *) (hm + cnt * 16);
        int32_t  *h_st = (int32_t *) (hm + cnt * 20);

        memcpy(out_size + lo, h_osz, cnt * 4);
        memcpy(status + lo, h_st, cnt * 4);
        pending_n[l] = 0;
        if (!sparse)
            return dense_finish(l, lo, cnt);
        const uint32_t *h_bits = (const uint32_t *) ctx->h_sp[l].p;
        const uint32_t *h_off = h_bits + cnt * SP_WORDS;
        const uint32_t  total = h_off[cnt];

        if ((uint64_t) total * SP_PAGE * 2 > cnt * (uint64_t) block_size)
        {
            /* mostly non-zero pages: the plain copy is the cheaper one */
            int rc = dense_d2h(l, lo, cnt);

            return rc != CRYOGPU_OK ? rc : dense_finish(l, lo, cnt);
        }
        int rc = host_reserve(ctx->h_stage[l], (size_t) total * SP_PAGE + SP_PAGE);

        if (rc != CRYOGPU_OK)
            return rc;
        if (total)
            CU(cudaMemcpyAsync(ctx->h_stage[l].p, ctx->d_stage[l].p, (size_t) total * SP_PAGE,
                               cudaMemcpyDeviceToHost, lanes[l]));
        d2h += (uint64_t) total * SP_PAGE;
        CU(cudaStreamSynchronize(lanes[l]));
        const uint8_t *pages = (const uint8_t *) ctx->h_stage[l].p;

        host_pool(ctx)->run(cnt, [&](size_t i) {
            place_sparse_block((uint8_t *) dst[lo + i], block_size, h_bits + i * SP_WORDS,
                               pages + (size_t) h_off[i] * SP_PAGE, &unmap);
        });
        return CRYOGPU_OK;
    };

    int lane = 0;

    for (size_t lo = 0; lo < n; lo += chunk, lane ^= 1)
    {
        size_t cnt = std::min(chunk, n - lo);
        int    rc = drain(lane);

        if (rc != CRYOGPU_OK)
            return rc;
        /* meta layout (host and device): off u64[cnt] | size u32[cnt] | method i32[cnt] ->
         * out_size u32[cnt] | status i32[cnt]   (offsets cnt*{0,8,12,16,20}) */
        size_t in_bytes = 0;

        for (size_t i = 0; i < cnt; i++)
            in_bytes += ((size_t) src_size[lo + i] + 15) & ~(size_t) 15;
        if ((rc = host_reserve(ctx->h_in[lane], in_bytes + 16)) != CRYOGPU_OK ||
            (rc = host_reserve(ctx->h_meta[lane], cnt * 24)) != CRYOGPU_OK ||
            (rc = dev_reserve(ctx->d_in[lane], in_bytes + 16)) != CRYOGPU_OK ||
            (rc = dev_reserve(ctx->d_meta[lane], cnt * 24)) != CRYOGPU_OK ||
            (rc = dev_reserve(ctx->d_out[lane], cnt * stride)) != CRYOGPU_OK ||
            (rc = dev_reserve(ctx->scratch, std::min(chunk, n) * (size_t) ZSTDD_SCRATCH_BYTES * 2)) != CRYOGPU_OK)
            return rc;
        /* work areas by the size of this call (the drop-in's calls are one block each, from every backend);
         * a missing one only selects the kernels that do without it */
        void *zpbuf = nullptr, *lzw = nullptr;
        bool  any_zstd = false, any_lz4 = false;       /* the methods are the host's here: no zstd work area (2.2 x the
                                                        * chunk's output) for a chunk without a zstd block */

        for (size_t i = 0; i < cnt; i++)
        {
            any_zstd = any_zstd || methods[lo + i] == CRYOGPU_ZSTD;
            any_lz4 = any_lz4 || methods[lo + i] == CRYOGPU_LZ4;
        }
        if (any_zstd && zstd_kernel_variant() == 3 &&
            dev_reserve(ctx->zp[lane], zp_bytes(std::min(chunk, n), block_size)) == CRYOGPU_OK)
            zpbuf = ctx->zp[lane].p;
        if (any_lz4 && block_size <= LZ4C_MAXCAP &&
            dev_reserve(ctx->lzw[lane], lz4c_bytes(std::min(chunk, n), ctx->sm_count)) == CRYOGPU_OK)
            lzw = ctx->lzw[lane].p;
        cudaGetLastError();
        const size_t sp_bytes = (cnt * (SP_WORDS + 1) + 1) * 4;

        if (sparse &&
            ((rc = dev_reserve(ctx->d_stage[lane], cnt * stride + SP_PAGE)) != CRYOGPU_OK ||
             (rc = dev_reserve(ctx->d_sp[lane], sp_bytes)) != CRYOGPU_OK ||
             (rc = host_reserve(ctx->h_sp[lane], sp_bytes)) != CRYOGPU_OK))
            return rc;
        uint8_t  *hm = (uint8_t *) ctx->h_meta[lane].p;
        uint64_t *h_off = (uint64_t *) hm;
        uint32_t *h_sz = (uint32_t *) (hm + cnt * 8);
        int32_t  *h_me = (int32_t *) (hm + cnt * 12);
        size_t    p = 0;

        for (size_t i = 0; i < cnt; i++)
        {
            h_off[i] = p;
            h_sz[i] = src_size[lo + i];
            h_me[i] = methods[lo + i];
            if (src_size[lo + i])
                memcpy((uint8_t *) ctx->h_in[lane].p + p, src[lo + i], src_size[lo + i]);
            p += ((size_t) src_size[lo + i] + 15) & ~(size_t) 15;
        }
        cudaStream_t st = lanes[lane];
        uint8_t     *dm = (uint8_t *) ctx->d_meta[lane].p;

        CU(cudaMemcpyAsync(ctx->d_in[lane].p, ctx->h_in[lane].p, in_bytes + 16, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(dm, hm, cnt * 16, cudaMemcpyHostToDevice, st));
        h2d += in_bytes + 16 + cnt * 16;
        uint8_t *scr = (uint8_t *) ctx->scratch.p + (size_t) lane * std::min(chunk, n) * ZSTDD_SCRATCH_BYTES;

        k_flag_unknown_methods<<<(unsigned) ((cnt + 255) / 256), 256, 0, st>>>(
            (int32_t *) (dm + cnt * 12), cnt, (uint32_t *) (dm + cnt * 16), (int32_t *) (dm + cnt * 20));
        /* (a chunk without blocks of a method does not launch that method's kernels: the drop-in's one-block call) */
        if (any_lz4)
            launch_lz4_decode(st, cnt, (int32_t *) (dm + cnt * 12), (uint8_t *) ctx->d_in[lane].p,
                              (uint64_t *) dm, (uint32_t *) (dm + cnt * 8),
                              (uint8_t *) ctx->d_out[lane].p, stride, block_size,
                              (uint32_t *) (dm + cnt * 16), (int32_t *) (dm + cnt * 20), lzw, ctx->sm_count);
        if (any_zstd)
            launch_zstd_decode(st, cnt, (int32_t *) (dm + cnt * 12), (uint8_t *) ctx->d_in[lane].p,
                               (uint64_t *) dm, (uint32_t *) (dm + cnt * 8),
                               (uint8_t *) ctx->d_out[lane].p, stride, block_size,
                               (uint32_t *) (dm + cnt * 16), (int32_t *) (dm + cnt * 20), scr,
                               ctx->predef, zpbuf, ctx->zaux[lane], ctx->zev[lane], ctx->sm_count);
        CU(cudaGetLastError());
        CU(cudaMemcpyAsync(hm + cnt * 16, dm + cnt * 16, cnt * 8, cudaMemcpyDeviceToHost, st));
        d2h += cnt * 8;
        if (sparse)
        {
            uint32_t *d_bits = (uint32_t *) ctx->d_sp[lane].p;
            uint32_t *d_off = d_bits + cnt * SP_WORDS;

            CU(cudaMemsetAsync(d_off + cnt, 0, 4, st));
            k_page_compact<<<(unsigned) cnt, 256, 0, st>>>((uint8_t *) ctx->d_out[lane].p, stride, block_size,
                                                          d_bits, d_off, d_off + cnt,
                                                          (uint8_t *) ctx->d_stage[lane].p);
            CU(cudaGetLastError());
            CU(cudaMemcpyAsync(ctx->h_sp[lane].p, ctx->d_sp[lane].p, sp_bytes, cudaMemcpyDeviceToHost, st));
            d2h += sp_bytes;
        }
        else if ((rc = dense_d2h(lane, lo, cnt)) != CRYOGPU_OK)
            return rc;
        pending_lo[lane] = lo;
        pending_n[lane] = cnt;
    }
    int rc = drain(0);

    if (rc == CRYOGPU_OK)
        rc = drain(1);
    ctx->last_h2d = h2d;
    ctx->last_d2h = d2h;
    return rc;
}

extern "C" int
cryogpu_compress_host(cryogpu_ctx *ctx, size_t n, int method, int level_or_accel,
                      const void *const *src, uint32_t block_size, void *const *dst,
                      uint32_t dst_cap, uint32_t *dst_size, int32_t *status)
{
    if (!ctx)
        return fail(CRYOGPU_E_ARG, "ctx is NULL");
    if (method != CRYOGPU_LZ4 && method != CRYOGPU_ZSTD)
        return fail(CRYOGPU_E_METHOD, "unknown compression method %d", method);
    if (n == 0)
        return CRYOGPU_OK;
    if (!src || !dst || !dst_size || !status)
        return fail(CRYOGPU_E_ARG, "NULL argument");
    if (block_size == 0 || block_size > (1u << 27))
        return fail(CRYOGPU_E_ARG, "block_size out of range");
    const uint64_t bound = cryogpu_compress_bound(method, block_size);

    if (dst_cap < bound)
        return fail(CRYOGPU_E_ARG, "dst_cap %u below cryogpu_compress_bound %llu", dst_cap,
                    (unsigned long long) bound);
    std::lock_guard<std::recursive_mutex> g(ctx->mu);

    CU(cudaSetDevice(ctx->device));
    CU(cudaEventSynchronize(ctx->busy));
    const size_t   chunk = chunk_blocks(block_size);
    const uint64_t sstride = ((uint64_t) block_size + 15) & ~(uint64_t) 15;
    const uint64_t dstride = (bound + 15) & ~(uint64_t) 15;
    const size_t   lane_scratch = (compress_scratch_bytes(method, block_size, std::min(chunk, n), ctx->sm_count) + 255) &
                                  ~(size_t) 255;
    const bool     src_pinned = is_pinned(src[0]);
    if (n > chunk)
    {
        int rc = make_lane_streams(ctx, 1);     /* a second chunk will be in flight */

        if (rc != CRYOGPU_OK)
            return rc;
    }
    cudaStream_t   lanes[2] = {ctx->stream, ctx->stream2};
    size_t         pending_lo[2] = {0, 0}, pending_n[2] = {0, 0};

    auto drain = [&](int l) -> int {
        if (pending_n[l] == 0)
            return CRYOGPU_OK;
        CU(cudaStreamSynchronize(lanes[l]));
        size_t    lo = pending_lo[l], cnt = pending_n[l];
        uint32_t *h_sz = (uint32_t *) ctx->h_meta[l].p;
        int32_t  *h_st = (int32_t *) ((uint8_t *) ctx->h_meta[l].p + cnt * 4);

        for (size_t i = 0; i < cnt; i++)
        {
            dst_size[lo + i] = h_sz[i];
            status[lo + i] = h_st[i];
            if (h_st[i] == CRYOGPU_ST_OK)
                memcpy(dst[lo + i], (uint8_t *) ctx->h_out[l].p + i * dstride, h_sz[i]);
        }
        pending_n[l] = 0;
        return CRYOGPU_OK;
    };

    int lane = 0;

    for (size_t lo = 0; lo < n; lo += chunk, lane ^= 1)
    {
        size_t cnt = std::min(chunk, n - lo);
        int    rc = drain(lane);

        if (rc != CRYOGPU_OK)
            return rc;
        if ((rc = dev_reserve(ctx->d_in[lane], cnt * sstride)) != CRYOGPU_OK ||
            (rc = dev_reserve(ctx->d_out[lane], cnt * dstride)) != CRYOGPU_OK ||
            (rc = dev_reserve(ctx->d_meta[lane], cnt * 8)) != CRYOGPU_OK ||
            (rc = host_reserve(ctx->h_meta[lane], cnt * 8)) != CRYOGPU_OK ||
            (rc = host_reserve(ctx->h_out[lane], cnt * dstride)) != CRYOGPU_OK ||
            (rc = dev_reserve(ctx->scratch, 2 * lane_scratch)) != CRYOGPU_OK)
            return rc;
        if (!src_pinned && (rc = host_reserve(ctx->h_in[lane], cnt * sstride)) != CRYOGPU_OK)
            return rc;
        cudaStream_t st = lanes[lane];

        if (src_pinned)
            for (size_t i = 0; i < cnt; i++)
                CU(cudaMemcpyAsync((uint8_t *) ctx->d_in[lane].p + i * sstride, src[lo + i], block_size,
                                   cudaMemcpyHostToDevice, st));
        else
        {
            for (size_t i = 0; i < cnt; i++)
                memcpy((uint8_t *) ctx->h_in[lane].p + i * sstride, src[lo + i], block_size);
            CU(cudaMemcpyAsync(ctx->d_in[lane].p, ctx->h_in[lane].p, cnt * sstride,
                               cudaMemcpyHostToDevice, st));
        }
        uint8_t *dm = (uint8_t *) ctx->d_meta[lane].p;
        uint8_t *scr = (uint8_t *) ctx->scratch.p + (size_t) lane * lane_scratch;

        rc = launch_compress(st, cnt, method, level_or_accel, (uint8_t *) ctx->d_in[lane].p, sstride, block_size,
                             (uint8_t *) ctx->d_out[lane].p, dstride, (uint32_t) bound, (uint32_t *) dm,
                             (int32_t *) (dm + cnt * 4), scr, ctx->sm_count);
        if (rc != CRYOGPU_OK)
            return rc;
        CU(cudaMemcpyAsync(ctx->h_meta[lane].p, dm, cnt * 8, cudaMemcpyDeviceToHost, st));
        /* compressed sizes are unknown until the kernel ends: bring back whole slots when the
         * batch is tiny, otherwise sizes first and then only the used prefix of every slot */
        if (cnt <= 4)
            CU(cudaMemcpyAsync(ctx->h_out[lane].p, ctx->d_out[lane].p, cnt * dstride,
                               cudaMemcpyDeviceToHost, st));
        else
        {
            CU(cudaStreamSynchronize(st));
            uint32_t *h_sz = (uint32_t *) ctx->h_meta[lane].p;

            for (size_t i = 0; i < cnt; i++)
                CU(cudaMemcpyAsync((uint8_t *) ctx->h_out[lane].p + i * dstride,
                                   (uint8_t *) ctx->d_out[lane].p + i * dstride,
                                   std::min<uint64_t>(h_sz[i], dstride), cudaMemcpyDeviceToHost, st));
        }
        pending_lo[lane] = lo;
        pending_n[lane] = cnt;
    }
    int rc = drain(0);

    if (rc == CRYOGPU_OK)
        rc = drain(1);
    return rc;
}

/* ------------------------------------------------------------- multi GPU */

template <typename F>
static int
run_sharded(int nctx, size_t n, F fn)
{
    std::vector<std::thread> th;
    std::vector<int>         rc(nctx, CRYOGPU_OK);
    std::vector<std::string> msg(nctx);

    for (int k = 0; k < nctx; k++)
    {
        size_t lo = n * k / nctx, hi = n * (k + 1) / nctx;

        if (hi == lo)
            continue;
        th.emplace_back([&, k, lo, hi]() {
            rc[k] = fn(k, lo, hi - lo);
            if (rc[k] != CRYOGPU_OK)
                msg[k] = g_err;
        });
    }
    for (auto &t : th)
        t.join();
    for (int k = 0; k < nctx; k++)
        if (rc[k] != CRYOGPU_OK)
            return fail(rc[k], "gpu shard %d: %s", k, msg[k].c_str());
    return CRYOGPU_OK;
}

extern "C" int
cryogpu_decompress_host_multi(cryogpu_ctx *const *ctxs, int nctx, size_t n, const int32_t *methods,
                              const void *const *src, const uint32_t *src_size, void *const *dst,
                              uint32_t block_size, uint32_t *out_size, int32_t *status)
{
    if (!ctxs || nctx < 1)
        return fail(CRYOGPU_E_ARG, "no contexts");
    return run_sharded(nctx, n, [&](int k, size_t lo, size_t cnt) {
        return cryogpu_decompress_host(ctxs[k], cnt, methods + lo, src + lo, src_size + lo, dst + lo,
                                       block_size, out_size + lo, status + lo);
    });
}

extern "C" int
cryogpu_compress_host_multi(cryogpu_ctx *const *ctxs, int nctx, size_t n, int method,
                            int level_or_accel, const void *const *src, uint32_t block_size,
                            void *const *dst, uint32_t dst_cap, uint32_t *dst_size, int32_t *status)
{
    if (!ctxs || nctx < 1)
        return fail(CRYOGPU_E_ARG, "no contexts");
    return run_sharded(nctx, n, [&](int k, size_t lo, size_t cnt) {
        return cryogpu_compress_host(ctxs[k], cnt, method, level_or_accel, src + lo, block_size,
                                     dst + lo, dst_cap, dst_size + lo, status + lo);
    });
}

#ifdef CX_PROF
/* development aid: phase cycle counters of CTA 0 of the CTA-per-block decoders; not part of include/cryogpu.h */
extern "C" int
cryogpu_debug_cxprof(unsigned long long *out32, int reset)
{
    unsigned long long zero[32] = {0};

    cudaDeviceSynchronize();
    if (out32)
        cudaMemcpyFromSymbol(out32, cx_prof, sizeof(zero));
    if (reset)
        cudaMemcpyToSymbol(cx_prof, zero, sizeof(zero));
    return 0;
}
#endif

#ifdef ZP_TIMELINE
/* development aid: read (and optionally reset) the pipeline timeline; not part of include/cryogpu.h */
extern "C" int
cryogpu_debug_timeline(unsigned long long *out32, int reset)
{
    unsigned long long init[32];

    cudaDeviceSynchronize();
    if (out32)
        cudaMemcpyFromSymbol(out32, zp_tl, sizeof(init));
    if (reset)
    {
        for (int i = 0; i < 32; i++)
            init[i] = (i & 1) ? 0ull : ~0ull;
        cudaMemcpyToSymbol(zp_tl, init, sizeof(init));
    }
    return 0;
}
#endif
