/*
 * tests/emu/emu_build.cpp -- TEST INFRASTRUCTURE ONLY.
 * The block-build kernel body (blk_build_block, pg_cryogen_b200/csrc/cryo_tuples.cuh) on the CPU through cuda_emu.h,
 * launched as cryogpu.cu launches k_block_build, so the `-m "not gpu"` suite can hold it against blockgen.pack_block.
 * Built by tests/test_emu_build.py.  Never part of libcryogpu.so.
 */
#define CRYO_EMU 1
#include "cuda_emu.h"
#include "../../pg_cryogen_b200/csrc/cryo_tuples.cuh"

/* cryogpu_build_blocks_device's launch: one CTA of BLK_THREADS per block, data_lo = 0 */
extern "C" int
emu_build_blocks(uint32_t n, const uint8_t *data, unsigned long long data_size, const unsigned long long *tup_off,
                 const uint32_t *tup_len, const unsigned long long *block_first, uint32_t block_size, uint8_t *dst,
                 uint64_t dst_stride, int32_t *status)
{
    if ((block_size & 7u) || block_size < 16 || ((uintptr_t) dst & 15u) || (dst_stride & 15u) || dst_stride < block_size)
        return -1;
    emu::launch(dim3(n), dim3(BLK_THREADS), BLK_SMEM, [&]() {
        const uint32_t b = blockIdx.x;

        blk_build_block(data, 0, data_size, tup_off, tup_len, block_first, b, block_size, dst + b * dst_stride, status + b,
                        (uint32_t *) CRYO_SMEM_BASE(), threadIdx.x);
    });
    return 0;
}
