// seqik_stream.cuh -- shared-memory staging and the persistent TMA tile pipeline of the streaming kernels
// (seqik_kernels.cu: FK, align apply, head apply; seqik_fk_grad.cu: FK backward).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "seqik_tma.cuh"

// 128-bit copy between global and shared memory when both ends are 16-byte aligned and the count is a multiple of 4
__device__ __forceinline__ void stage_in(float* __restrict__ dst, const float* __restrict__ src, int n) {
    if ((n & 3) == 0 && (((uintptr_t)src) & 15) == 0) {
        const float4* s4 = reinterpret_cast<const float4*>(src); float4* d4 = reinterpret_cast<float4*>(dst);
        for (int i = threadIdx.x; i < (n >> 2); i += blockDim.x) d4[i] = __ldg(s4 + i);
    } else {
        for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = __ldg(src + i);
    }
}
__device__ __forceinline__ void stage_out(float* __restrict__ dst, const float* __restrict__ src, int n) {
    if ((n & 3) == 0 && (((uintptr_t)dst) & 15) == 0) {
        const float4* s4 = reinterpret_cast<const float4*>(src); float4* d4 = reinterpret_cast<float4*>(dst);
        for (int i = threadIdx.x; i < (n >> 2); i += blockDim.x) __stcs(d4 + i, s4[i]);
    } else {
        for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
    }
}

// ---- persistent, TMA-fed tile pipeline for the streaming kernels (sm_100a) -------------------------------------------------
// A few CTAs per SM walk over tiles of 256 units.  A single thread moves the tiles with the bulk-copy engine
// (cp.async.bulk, 1-D; SASS UBLKCP): the input tiles of the NEXT tile land in shared memory behind an mbarrier while the
// current tile is computed, and the output tile leaves through a bulk store (double-buffered) -- no thread issues a global
// load or store and no register holds data in flight.  Measured on the FK kernel: 0.70 -> 0.91 of the HBM copy peak.
// Bulk copies need 16-byte aligned addresses and sizes: the launchers check and fall back to the plain kernels (which
// also take the ragged last tile).
// The pipeline itself.  `Op` describes one streaming computation over tiles of TILE = 256 units:
//   N_IN input streams with (per-tile) byte counts in_bytes(i, tile) [0 = stream absent] from in_src(i, tile), placed at the
//   128-byte aligned offsets IN_OFF[i] of a stage; compute(tid, tile, stage) fills the stage's output region (OUT_OFF);
//   store(tile, out) issues the bulk store(s) of that region.  STAGE_BYTES per stage, two stages.
constexpr int TILE = 256;
template <class Op>
__global__ void __launch_bounds__(TILE) tma_tile_kernel(const Op op, int64_t n_tiles) {
    extern __shared__ __align__(128) unsigned char tile_smem[];
    uint64_t* bar = reinterpret_cast<uint64_t*>(tile_smem + 2 * Op::STAGE_BYTES);
    const int tid = threadIdx.x;
    if (tid == 0) {
        mbar_init(&bar[0], 1); mbar_init(&bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    auto load = [&](int64_t tile, int st) {                      // thread 0 only
        uint32_t total = 0;
#pragma unroll
        for (int i = 0; i < Op::N_IN; ++i) total += op.in_bytes(i, tile);
        mbar_expect_tx(&bar[st], total);
#pragma unroll
        for (int i = 0; i < Op::N_IN; ++i) {
            const uint32_t nb = op.in_bytes(i, tile);
            if (nb) tma_load_1d(tile_smem + st * Op::STAGE_BYTES + Op::in_off(i), op.in_src(i, tile), nb, &bar[st]);
        }
    };
    if (tid == 0 && (int64_t)blockIdx.x < n_tiles) load(blockIdx.x, 0);
    int it = 0;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
        const int st = it & 1;
        unsigned char* stage = tile_smem + st * Op::STAGE_BYTES;
        if (tid == 0) {
            const int64_t next = tile + gridDim.x;
            if (next < n_tiles) load(next, st ^ 1);              // its previous reader finished before the last barrier
            tma_store_wait_read<1>();                            // the store issued two tiles ago has drained this stage's output
        }
        mbar_wait(&bar[st], (uint32_t)(it >> 1) & 1u);
        __syncthreads();
        op.compute(tid, tile, stage);
        fence_async_smem();                                      // generic-proxy writes of the output -> visible to the bulk store
        __syncthreads();
        if (tid == 0) { op.store(tile, stage + Op::OUT_OFF); tma_commit(); }
    }
    if (tid == 0) tma_store_wait_read<0>();                      // shared memory must outlive the stores that read it
}
template <class Op>
static void launch_tiles(const Op& op, int64_t n_tiles, cudaStream_t st) {
    int dev = 0, n_sm = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
    constexpr int smem = 2 * Op::STAGE_BYTES + 16;
    // (per device and idempotent, so simply set on every call: a host-side table lookup)
    cudaFuncSetAttribute(tma_tile_kernel<Op>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    cudaFuncSetAttribute(tma_tile_kernel<Op>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    const int fit = (227 * 1024) / (smem + 1024);               // CTAs that fit one SM's 227 KB (1 KB reserved per CTA)
    const int64_t cap = (int64_t)n_sm * (fit < 1 ? 1 : (fit > 4 ? 4 : fit));
    tma_tile_kernel<Op><<<(unsigned)(n_tiles < cap ? n_tiles : cap), TILE, smem, st>>>(op, n_tiles);
}
