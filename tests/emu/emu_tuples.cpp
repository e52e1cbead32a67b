/*
 * tests/emu/emu_tuples.cpp -- TEST INFRASTRUCTURE ONLY.
 * The tuple-fetch kernel bodies (pg_cryogen_b200/csrc/cryo_tuples.cuh) on the CPU through cuda_emu.h, launched as
 * cryogpu.cu launches them, so the `-m "not gpu"` suite can hold them against the restatement in tests/tuple_oracle.c.
 * Built by tests/test_emu_tuples.py.  Never part of libcryogpu.so.
 */
#define CRYO_EMU 1
#include "cuda_emu.h"
#include "../../pg_cryogen_b200/csrc/cryo_tuples.cuh"

/* the tuple fetch as cryogpu.cu launches it: k_tuple_select (a warp per block, 8 per CTA), k_tuple_scan (one CTA),
 * k_tuple_gather (a warp per block); ent0 / byte0 = 0.  work: 3 x (n + 1) words */
extern "C" int
emu_tuples(const uint8_t *blocks, uint64_t stride, uint32_t block_size, uint32_t n, const int32_t *block_status,
           const unsigned long long *sel_off, const uint32_t *sel_pos, uint8_t *data, unsigned long long data_cap,
           unsigned long long *tup_off, uint32_t *tup_len, unsigned long long tup_cap, unsigned long long *block_first,
           int32_t *status, unsigned long long *need, unsigned long long *work)
{
    if (((uintptr_t) blocks | stride) & 7u || ((uintptr_t) data & 15u) || block_size < 16)
        return -1;
    unsigned long long *cnt = work, *bytes = work + (n + 1), *byte_first = work + 2 * (size_t) (n + 1);

    emu::launch(dim3((n + 7u) / 8u), dim3(256), 0, [&]() {
        const uint32_t b = blockIdx.x * 8u + (threadIdx.x >> 5), lane = threadIdx.x & 31u;

        if (b < n)
            tup_select_block(blocks + b * stride, block_size, block_status ? block_status[b] : ST_OK, sel_off, sel_pos, b,
                             cnt + b, bytes + b, status + b, lane);
    });
    emu::launch(dim3(1), dim3(TUP_SCAN_THREADS), 64 * sizeof(unsigned long long), [&]() {
        tup_scan(n, cnt, bytes, status, 0, 0, tup_cap, data_cap, block_first, byte_first, need,
                 (unsigned long long *) CRYO_SMEM_BASE(), threadIdx.x, TUP_SCAN_THREADS);
    });
    const TupOut o = {data, tup_off, tup_len, 0, 0};

    emu::launch(dim3((n + 7u) / 8u), dim3(256), 0, [&]() {
        const uint32_t b = blockIdx.x * 8u + (threadIdx.x >> 5), lane = threadIdx.x & 31u;

        if (b < n && status[b] == ST_OK)
            tup_gather_block(blocks + b * stride, block_size, sel_off, sel_pos, b, block_first[b], byte_first[b], o, lane);
    });
    return 0;
}
