// K1 (head form): conv1x1 as a GEMM on the 5th-gen tensor cores, one CTA per 128-row tile.  It runs the head convs with f32
// output (scalar conv, policy conv2, attention convs), the layers conv_i2c.cu / tower8k.cu / heads8.cu do not take.  Every head conv
// is 1x1 (net_spec.cpp rejects any other), so a tile needs no tap shifts and no zero padding.
//
// Replaces the per-layer `cudnnConvolutionBiasActivationForward` (fp32 NCHW) of the reference's CUDA executor (kn-cuda-eval 0.7.3
// planner, evidence docs/conv_bn_sm_flow.svg; call site rust/kz-core/src/network/cudnn.rs:73).
//
// GEMM view (per layer):  D[M=positions, N=cout] = sum_ci A[M, ci] * W[N, ci]
//   * activations are dense channels-last bf16 rows [position][cin_pad], one row per square; one M tile = 128 rows, loaded by a
//     2-D tensor map (c, row) with box (64, 128) at (c0, tile * 128); rows past the buffer are zero-filled
//   * both operands land in shared memory in the canonical K-major SWIZZLE_128B layout, tcgen05.mma
//     (cta_group::1, kind::f16, M=128, N=cout_pad, K=16) accumulates fp32 in TMEM
//   * epilogue (4 warps): tcgen05.ld -> +bias (BN folded on the host) -> relu -> +residual -> bf16 / f32 store (conv_epilogue.cuh)
//   * persistent CTAs, warp-specialised: warp 0 TMA producer, warp 1 MMA issuer (+TMEM owner),
//     warps 2..5 epilogue; smem ring of `stages` (A,B) slots; two TMEM accumulators so the epilogue of
//     tile i overlaps the MMAs of tile i+1.
//   * two instances: bf16 rows (kind::f16, K = 16, 64 channels per k-block) and, for the TF32 precision, f32 rows holding TF32-exact
//     values (kind::tf32, K = 8, 32 channels per k-block); a k-block is one 128-byte row in both, so the stage layout is the same.
//     The output is f32 and is not rounded: the tail kernel's CUDA-core FCs read it.
#include "conv_epilogue.cuh"
#include "kernels.cuh"
#include "tc_common.cuh"

namespace kzb {
namespace {

constexpr int kTileM = 128;
constexpr int kABytes = kTileM * 128;            // 16 KiB: one 128-byte smem row (= one swizzle span) per tile row
constexpr int kMmasPerKBlock = 4;                 // 32 bytes of K each: K = 16 bf16 or K = 8 TF32
constexpr int kThreads = 192;

using namespace tc;

struct SmemLayout {
    uint8_t* stage_base;
    uint64_t* full;
    uint64_t* empty;
    uint64_t* tmem_full;
    uint64_t* tmem_empty;
    uint32_t* tmem_ptr;
    float* bias;
};

__device__ __forceinline__ SmemLayout carve(uint8_t* base, int n, int stages) {
    SmemLayout s;
    s.stage_base = base;
    uint8_t* p = base + size_t(stages) * (kABytes + n * 128);
    s.full = reinterpret_cast<uint64_t*>(p);
    s.empty = s.full + stages;
    s.tmem_full = s.empty + stages;
    s.tmem_empty = s.tmem_full + 2;
    s.tmem_ptr = reinterpret_cast<uint32_t*>(s.tmem_empty + 2);
    s.bias = reinterpret_cast<float*>(s.tmem_ptr + 4);
    return s;
}

template <typename T>
__global__ void __launch_bounds__(kThreads, 1)
    conv_tc_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b, const ConvTcParams p) {
    extern __shared__ uint8_t smem_raw[];
    // SWIZZLE_128B atoms need 1024-byte alignment
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const SmemLayout sm = carve(smem, p.n, p.stages);
    constexpr int kBlockK = 128 / int(sizeof(T));  // channels per k-block
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    const int stage_bytes = kABytes + p.n * 128;
    const int my_tiles = (p.num_tiles - int(blockIdx.x) + int(gridDim.x) - 1) / int(gridDim.x);

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_a)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_b)) : "memory");
        for (int i = 0; i < p.stages; i++) {
            mbar_init(&sm.full[i], 1);
            mbar_init(&sm.empty[i], 1);
        }
        for (int i = 0; i < 2; i++) {
            mbar_init(&sm.tmem_full[i], 1);
            mbar_init(&sm.tmem_empty[i], 4);  // one arrive per epilogue warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(sm.tmem_ptr)),
                     "r"(uint32_t(p.tmem_cols))
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    for (int i = threadIdx.x; i < p.n; i += kThreads) sm.bias[i] = p.bias[i];
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *sm.tmem_ptr;
    const uint32_t acc_stride = uint32_t(p.tmem_cols / 2);

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int ti = 0; ti < my_tiles; ti++) {
                const int tile = int(blockIdx.x) + ti * int(gridDim.x);
                for (int kb = 0; kb < p.kblocks; kb++) {
                    mbar_wait(&sm.empty[stage], phase ^ 1);
                    uint8_t* a_dst = sm.stage_base + size_t(stage) * stage_bytes;
                    uint8_t* b_dst = a_dst + kABytes;
                    mbar_expect_tx(&sm.full[stage], uint32_t(stage_bytes));
                    tma_load_2d(&tmap_a, &sm.full[stage], a_dst, kb * kBlockK, tile * kTileM);
                    tma_load_2d(&tmap_b, &sm.full[stage], b_dst, kb * kBlockK, 0);
                    if (++stage == p.stages) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer
        // whole warp walks the loops (uniform datapath for the address arithmetic); lane 0 issues MMAs + commits
        const uint32_t idesc = umma_idesc<T>(kTileM, p.n);
        const uint64_t desc_hi = umma_desc_sw128_hi();
        int stage = 0;
        uint32_t phase = 0;
        for (int local = 0; local < my_tiles; local++) {
            const int buf = local & 1;
            const uint32_t buf_phase = (local >> 1) & 1;
            mbar_wait(&sm.tmem_empty[buf], buf_phase ^ 1);
            tc_fence_after();
            const uint32_t tmem_d = tmem_base + buf * acc_stride;
            for (int it = 0; it < p.kblocks; it++) {
                mbar_wait(&sm.full[stage], phase);
                tc_fence_after();
                const uint32_t a_lo = umma_desc_lo(smem_u32(sm.stage_base + size_t(stage) * stage_bytes));
                const uint32_t b_lo = a_lo + (kABytes >> 4);
                if (lane == 0) {
#pragma unroll
                    for (int k = 0; k < kMmasPerKBlock; k++) {
                        // advancing 32 bytes along K stays inside the 128-byte swizzle span
                        if constexpr (sizeof(T) == 4)
                            umma_tf32(tmem_d, desc_hi | uint64_t(a_lo + 2 * k), desc_hi | uint64_t(b_lo + 2 * k), idesc, (it | k) != 0);
                        else
                            umma_bf16(tmem_d, desc_hi | uint64_t(a_lo + 2 * k), desc_hi | uint64_t(b_lo + 2 * k), idesc,
                                      (it | k) != 0);
                    }
                    // frees the smem slot once these MMAs have read it
                    umma_commit(&sm.empty[stage]);
                }
                __syncwarp();
                if (++stage == p.stages) {
                    stage = 0;
                    phase ^= 1;
                }
            }
            if (lane == 0) umma_commit(&sm.tmem_full[buf]);  // accumulator complete -> epilogue
            __syncwarp();
        }
    } else {
        // ------------------------------------------------------------------ epilogue (warps 2..5)
        const int quarter = warp % 4;  // TMEM lanes [32*quarter, 32*quarter+32) are the ones this warp may read
        for (int local = 0; local < my_tiles; local++) {
            const int tile = int(blockIdx.x) + local * int(gridDim.x);
            const int buf = local & 1;
            const uint32_t buf_phase = (local >> 1) & 1;
            conv_epilogue_tile(p, sm.bias, tile, quarter, lane, tmem_base + buf * acc_stride, &sm.tmem_full[buf], buf_phase, &sm.tmem_empty[buf], 0,
                               p.n_store);
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(uint32_t(p.tmem_cols))
                     : "memory");
    }
}

}  // namespace

size_t conv_tc_smem_bytes(int n, int stages) {
    return 1024 /*alignment slack*/ + size_t(stages) * (kABytes + size_t(n) * 128) + (2 * stages + 4) * 8 + 16 + size_t(n) * 4;
}

int conv_tc_pick_stages(int n) {
    const size_t budget = 227 * 1024;
    int stages = 8;
    while (stages > 2 && conv_tc_smem_bytes(n, stages) > budget) stages--;
    return stages;
}

void conv_tc_prepare() {
    cudaFuncSetAttribute(conv_tc_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    cudaFuncSetAttribute(conv_tc_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
}

void launch_conv_tc(const CUtensorMap& tmap_a, const CUtensorMap& tmap_b, const ConvTcParams& p, int grid, cudaStream_t s) {
    if (p.num_tiles <= 0) return;
    if (p.tf32)
        conv_tc_kernel<float><<<std::min(grid, p.num_tiles), kThreads, conv_tc_smem_bytes(p.n, p.stages), s>>>(tmap_a, tmap_b, p);
    else
        conv_tc_kernel<__nv_bfloat16><<<std::min(grid, p.num_tiles), kThreads, conv_tc_smem_bytes(p.n, p.stages), s>>>(tmap_a, tmap_b, p);
}

}  // namespace kzb
