/*
 * tests/emu/emu_encode_multi.cpp -- TEST INFRASTRUCTURE ONLY.
 * The encoder work loops (lz4_encode_worker / zstd_encode_worker) on the CPU through cuda_emu.h, over a batch of
 * blocks in the caller's strided slots, so that the `-m "not gpu"` suite sees what a block's stream depends on: the
 * bytes after it in its source slot, the bytes after dst_cap in its destination slot, and the other blocks that
 * share the work queue.  Built by tests/test_emu_encode_contract.py.  Never part of libcryogpu.so.
 *
 * cuda_emu.h runs the CTAs of a grid one after another, so the first would take every work item; here ncta
 * emulated CTAs of `warps` warps each are the fibers of ONE emulated launch, interleaved by its scheduler, and
 * take items from one queue as the device's persistent CTAs do.  Each has its own shared-memory tables and, for
 * zstd, its own global scratch, as k_lz4_encode / k_zstd_encode give them.
 */
#define CRYO_EMU 1
#include "cuda_emu.h"
#include "../../pg_cryogen_b200/csrc/lz4_encode.cuh"
#include "../../pg_cryogen_b200/csrc/zstd_encode.cuh"

#include <vector>

/* method 0 = LZ4 (level = acceleration), 1 = zstd.  src, dst, src_stride and dst_stride 16-byte aligned, as
 * cryogpu_compress_device requires.  Returns 0, or -1 for arguments the device call would refuse. */
extern "C" int
emu_encode_multi(int method, int level, const uint8_t *src, uint64_t src_stride, uint32_t n, uint32_t nblocks,
                 uint8_t *dst, uint64_t dst_stride, uint32_t dst_cap, uint32_t *dst_size, int32_t *status, uint32_t ncta,
                 uint32_t warps)
{
    if (((uintptr_t) src & 15) || (src_stride & 15) || ((uintptr_t) dst & 15) || (dst_stride & 15) ||
        src_stride < n || dst_stride < dst_cap || nblocks == 0 || ncta == 0 || warps == 0 || warps > 16)
        return -1;
    const uint32_t nwarps = ncta * warps;
    std::vector<uint32_t> queue(64 + nblocks, 0);      /* [0]: next work item; [64 + b]: finished items of block b */

    if (method == 0)
    {
        const size_t per = lz4e_scratch_bytes(n);
        std::vector<uint8_t> scr(nblocks * per + 64, 0x55);
        uint8_t *sc = (uint8_t *) (((uintptr_t) scr.data() + 15) & ~(uintptr_t) 15);

        emu::launch(dim3(1), dim3(32 * nwarps), (size_t) nwarps * LZ4E_HASH_BYTES + 64, [&]() {
            const uint32_t warp = threadIdx.x >> 5;

            lz4_encode_worker(src, src_stride, n, dst, dst_stride, dst_cap, level, dst_size, status, sc, per, nblocks,
                              queue.data(), queue.data() + 64,
                              reinterpret_cast<uint16_t *>(CRYO_SMEM_BASE() + warp * LZ4E_HASH_BYTES), threadIdx.x & 31);
        });
        return 0;
    }
    if (n > ZSE_MAXBLK * (uint64_t) ZSE_BLOCK)
        return -1;
    std::vector<uint8_t> scr((size_t) ncta * zstde_scratch_bytes(n) + 64, 0x55);
    std::vector<uint32_t> bmeta((size_t) nblocks * ZSE_MAXBLK, 0xCDCDCDCDu);
    uint8_t *sc = (uint8_t *) (((uintptr_t) scr.data() + 15) & ~(uintptr_t) 15);

    emu::launch(dim3(1), dim3(32 * nwarps), (size_t) nwarps * ZSE_PER_WARP + 512, [&]() {
        const uint32_t warp = threadIdx.x >> 5, cta = warp / warps;

        zstd_encode_worker(src, src_stride, n, dst, dst_stride, dst_cap, level, dst_size, status,
                           sc + cta * zstde_scratch_bytes(n) + (size_t) (warp % warps) * ZSE_SCR_PER_WARP, nblocks,
                           queue.data(), queue.data() + 64, bmeta.data(), CRYO_SMEM_BASE() + warp * ZSE_PER_WARP,
                           threadIdx.x & 31);
    });
    return 0;
}
