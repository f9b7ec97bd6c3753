// K1i: conv3x3 (and conv1x1: p.taps = 1) as an implicit GEMM on DENSE rows -- TMA im2col loads + the CTA-pair MMA.  The layers of every board the
// 8x8 whole-tower kernel does not cover (go 9x9 / 19x19, wide nets), and the head 1x1 convs of every net the fused heads kernel does not cover.
//
// GEMM view: D[pixels, cout] += A_tap[pixels, 64 ch] * W_tap[cout, 64 ch] over 9 taps x cin/64 k-blocks.  Activations are plain
// channels-last rows [board][y][x][C] with NO padding rows: the TMA engine's im2col mode (cuTensorMapEncodeIm2col, bounding box
// corners -1 / -1 for a 3x3 filter with zero padding 1) walks 128 consecutive output pixels across ranks and boards, adds the tap
// offset and zero-fills whatever falls off the board, so every row the tensor core multiplies is a real square (the padded-row
// layout it replaced spent 19 % of the MMAs on zero rows on 9x9, 10 % on 19x19).  Each 128-pixel tile is re-loaded per
// tap (16 KB, SWIZZLE_128B) next to the half weight tile (slice/2 x 64, up to 16 KB): exactly the shared-memory traffic of a plain
// 2-SM GEMM.
//
// Two CTAs of a cluster own 256 consecutive pixels (128 each); each stages its own pixels and HALF of every weight tile; the
// leader issues tcgen05.mma.cta_group::2 with M = 256 and both CTAs' TMEM receive their own 128 rows x (n / n_split) columns.
// Synchronisation (L = leader = cluster rank 0, P = peer); only L's MMA thread issues, one barrier wait per stage:
//   full[s] (L's copy)     armed by L's producer with the bytes of BOTH CTAs; P's TMA loads complete their bytes on L's barrier
//                          (cp.async.bulk.tensor .cta_group::2, peer bit of the barrier address cleared)
//   empty[s]               L's commit, multicast to both CTAs: the MMAs that read the stage are done
//   tmem_full[b]           L's commit, multicast: accumulator b is complete in both CTAs' TMEM
//   tmem_empty[b] (on L)   8 arrivals: the 4 epilogue warps of L (local) and of P (remote) have drained accumulator b
// Epilogue (warps 2..5, one TMEM lane quarter = 32 pixel rows each; thread = row): 32 output channels at a time,
// tcgen05.ld -> +bias -> relu -> +residual -> bf16, through a per-warp ring of four 2 KB SWIZZLE_64B staging boxes: the residual box
// arrives by TMA two chunks ahead, is updated IN PLACE and leaves by TMA store -- no per-thread global loads / stores, and a code
// body of a few hundred instructions (a per-thread epilogue with global loads / stores unrolled to 90 KB of code and kept the
// epilogue warps busy 80-90 % of a tile's MMA time: profiles/r02_go_kernels.md).
// Output channels in slices (p.n_split): a work item is one 256-pixel tile x one slice of n / n_split output channels, so every MMA
// has N = n / n_split <= 256 (the cta_group::2 limit; also the largest TMA box and half of a CTA's 512 TMEM columns, since an
// accumulator pair takes 2 N columns).  Layers wider than 256 always run in slices; small batches split further to fill the SMs
// (executor.cu).  The bias of a chunk is read from global memory (one 128-byte line, the same for every lane) rather than staged:
// shared memory and the stage count do not depend on the width.
// p.pdl: launched with programmatic stream serialization -- set-up and the first weight tiles overlap the previous layer's tail.
//
// Two instances, one per operand type T; a k-block is one 128-byte row in either:
//   bf16  (p.tf32 = 0): 64 channels per k-block, kind::f16 MMAs of K = 16, bf16 rows, 2 KB SWIZZLE_64B staging boxes
//   float (p.tf32 = 1): 32 channels per k-block, kind::tf32 MMAs of K = 8 on f32 values that are TF32-exact; f32 rows, 4 KB
//                       SWIZZLE_128B staging boxes, and every value the tower form stores rounded to TF32 (tf32_round), since it is
//                       the next layer's MMA operand.  Twice the k-blocks of bf16 for the same channels, so twice the stages per layer.
// Stages, the pair logic, PDL, n_split and the barrier protocol are the same in both.
//
// Each comes in two forms (kHead, p.head) that differ only in the epilogue:
//   tower form: relu on the whole layer or none, optional residual, output in the operand type (the next layer's MMA operand)
//   head form (the head 1x1 convs: scalar conv merged with the extra policy conv, policy conv2, the attention convs): relu on output
//               channels < p.relu_n, no residual, f32 output that is NOT rounded (the tail kernel's CUDA-core FCs read it), through
//               4 KB SWIZZLE_128B staging boxes in both operand types.  The MMA width p.n is the stored width rounded up to 32; the
//               output map's inner dimension is the stored width, so the TMA store clips the padding columns.
#include <type_traits>

#include "kernels.cuh"
#include "tc_common.cuh"

namespace kzb {
namespace {

constexpr int kTileM = 128;
constexpr int kThreads = 192;
constexpr uint32_t kABytes = kTileM * 128;    // one im2col tile: 128 pixels x one 128-byte k-block
constexpr uint32_t kStageBytes = 2 * kABytes;  // + a half weight tile of up to 128 rows
constexpr int kMmasPerStage = 4;               // 32 bytes of K each: K = 16 bf16 or K = 8 TF32
constexpr int kChunk = 32;                     // output channels per epilogue step
constexpr int kStgBufs = 4;                    // per epilogue warp
template <typename T>
constexpr int kBlockKOf = 128 / int(sizeof(T));  // channels per k-block
template <typename T>
constexpr uint32_t kStgBytesOf = 32 * kChunk * sizeof(T);  // one staging box: 32 rows x 32 channels
constexpr uint16_t kPairMask = 3;
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;

using namespace tc;

struct SmemLayout {
    uint8_t* stages;   // [stage][A 16 KB | B 16 KB], 1024-byte aligned
    uint8_t* staging;  // [epilogue warp][kStgBufs][kStgBytes]
    uint64_t *full, *empty, *tmem_full, *tmem_empty, *res_full;
    uint32_t* tmem_ptr;
};

template <typename T>
__device__ __forceinline__ SmemLayout carve(uint8_t* base, int stages) {
    SmemLayout s;
    s.stages = base;
    s.staging = base + size_t(stages) * kStageBytes;
    s.full = reinterpret_cast<uint64_t*>(s.staging + 4 * kStgBufs * kStgBytesOf<T>);
    s.empty = s.full + stages;
    s.tmem_full = s.empty + stages;
    s.tmem_empty = s.tmem_full + 2;
    s.res_full = s.tmem_empty + 2;
    s.tmem_ptr = reinterpret_cast<uint32_t*>(s.res_full + 4 * kStgBufs);
    return s;
}

// im2col load of kTileM pixels x one k-block of channels starting at base pixel (w, h, n) (bounding-box coordinates: output pixel - 1),
// tap offset (off_w, off_h) in 0..2; issued by either CTA of the pair, bytes completed on the LEADER's barrier
__device__ __forceinline__ void tma2_load_im2col(const CUtensorMap* map, uint64_t* bar, void* dst, int c, int w, int h, int n, uint16_t off_w,
                                                 uint16_t off_h) {
    asm volatile(
        "cp.async.bulk.tensor.4d.im2col.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2], "
        "{%7, %8};" ::"r"(smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c), "r"(w), "r"(h), "r"(n), "h"(off_w), "h"(off_h)
        : "memory");
}
__device__ __forceinline__ void tma2_load_2d(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(map)),
                 "r"(smem_u32(src)), "r"(c0), "r"(c1)
                 : "memory");
}
template <int kPending>
__device__ __forceinline__ void tma_store_wait_read() {  // at most kPending of this thread's store groups still read shared memory
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(kPending) : "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
template <typename T>
__device__ __forceinline__ void umma2(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    if constexpr (sizeof(T) == 4)
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t"
            "}" ::"r"(tmem_d),
            "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
            : "memory");
    else
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
            "}" ::"r"(tmem_d),
            "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
            : "memory");
}
__device__ __forceinline__ void umma2_commit(uint64_t* bar) {  // arrives on `bar` in both CTAs of the pair
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
                 "h"(kPairMask)
                 : "memory");
}

template <typename T, bool kHead>
__global__ void __launch_bounds__(kThreads, 1)
    conv_i2c_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_bh, const __grid_constant__ CUtensorMap tmap_out,
                    const __grid_constant__ CUtensorMap tmap_res, const ConvTcParams p) {
    using Out = std::conditional_t<kHead, float, T>;  // element type of the stored output
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const SmemLayout sm = carve<Out>(smem, p.stages);
    constexpr int kBlockK = kBlockKOf<T>;
    constexpr uint32_t kStgBytes = kStgBytesOf<Out>;
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    const uint32_t rank = cluster_ctarank();
    const bool leader = rank == 0;
    const int n_eff = p.n / p.n_split;                      // output channels per work item
    const uint32_t b_bytes = uint32_t(n_eff / 2) * 128u;    // this CTA's half of a weight tile
    const int num_pairs = (p.num_tiles + 1) / 2;            // pair tiles of 256 pixels
    const int num_items = num_pairs * p.n_split;
    const int cluster_id = int(blockIdx.x) / 2, num_clusters = int(gridDim.x) / 2;
    const int area = p.lay.W * p.lay.H;
    const int taps = p.taps, pad = p.taps == 9 ? 1 : 0;  // 3x3 with zero padding 1, or 1x1

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_a)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_bh)) : "memory");
        for (int i = 0; i < p.stages; i++) {
            mbar_init(&sm.full[i], 1);
            mbar_init(&sm.empty[i], 1);
        }
        for (int i = 0; i < 2; i++) {
            mbar_init(&sm.tmem_full[i], 1);
            mbar_init(&sm.tmem_empty[i], 8);  // 4 epilogue warps of each CTA (only the leader's copy is used)
        }
        for (int i = 0; i < 4 * kStgBufs; i++) mbar_init(&sm.res_full[i], 1);
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_out)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_res)) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(sm.tmem_ptr)),
                     "r"(uint32_t(p.tmem_cols))
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();  // the peer's barriers exist before anything is committed to / completes on them
    tc_fence_after();
    const uint32_t tmem_base = *sm.tmem_ptr;
    const uint32_t acc_stride = uint32_t(p.tmem_cols / 2);
    if (p.pdl) grid_dep_launch_dependents();  // the next layer may set itself up while this one computes

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer (both CTAs: own pixels, own weight half)
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            int pre = 0;  // stages whose barrier is armed and whose weight half is in flight already
            if (p.pdl) {
                // weights do not depend on the previous layer: fill the ring's weight halves before waiting for it
                if (cluster_id < num_items) {
                    const int n0 = (cluster_id % p.n_split) * n_eff;
                    for (; pre < p.stages && pre < taps * p.kblocks; pre++) {
                        if (leader) mbar_expect_tx(&sm.full[pre], 2 * (kABytes + b_bytes));
                        tma2_load_2d(&tmap_bh, &sm.full[pre], sm.stages + size_t(pre) * kStageBytes + kABytes, (pre % taps) * p.cin_pad + (pre / taps) * kBlockK,
                                     n0 + int(rank) * (n_eff / 2));
                    }
                }
                grid_dep_wait();  // the activations are the previous layer's output
            }
            for (int item = cluster_id; item < num_items; item += num_clusters) {
                const int pt = item / p.n_split, n0 = (item % p.n_split) * n_eff;
                const int pix = (2 * pt + int(rank)) * kTileM;  // first pixel of this CTA's tile (may lie past the batch: rows never stored)
                const int img = pix / area, rem = pix - img * area;
                const int h0 = rem / p.lay.W, w0 = rem - h0 * p.lay.W;
                for (int kb = 0; kb < p.kblocks; kb++) {
                    for (int tap = 0; tap < taps; tap++) {
                        uint8_t* dst = sm.stages + size_t(stage) * kStageBytes;
                        if (pre > 0) {
                            pre--;
                        } else {
                            mbar_wait(&sm.empty[stage], phase ^ 1);
                            if (leader) mbar_expect_tx(&sm.full[stage], 2 * (kABytes + b_bytes));
                            tma2_load_2d(&tmap_bh, &sm.full[stage], dst + kABytes, tap * p.cin_pad + kb * kBlockK, n0 + int(rank) * (n_eff / 2));
                        }
                        tma2_load_im2col(&tmap_a, &sm.full[stage], dst, kb * kBlockK, w0 - pad, h0 - pad, img, uint16_t(tap % 3), uint16_t(tap / 3));
                        if (++stage == p.stages) {
                            stage = 0;
                            phase ^= 1;
                        }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA warp: only the leader's issues
        if (leader) {
            const uint32_t idesc = umma_idesc<T>(2 * kTileM, n_eff);
            const uint64_t hi = umma_desc_sw128_hi();
            int stage = 0;
            uint32_t phase = 0;
            int local = 0;
            for (int item = cluster_id; item < num_items; item += num_clusters, local++) {
                const int buf = local & 1;
                const uint32_t buf_phase = (local >> 1) & 1;
                mbar_wait_cluster(&sm.tmem_empty[buf], buf_phase ^ 1);
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + buf * acc_stride;
                const int steps = taps * p.kblocks;
                for (int it = 0; it < steps; it++) {
                    mbar_wait(&sm.full[stage], phase);  // both CTAs' pixels and both halves of the weight tile
                    tc_fence_after();
                    const uint32_t a_lo = umma_desc_lo(smem_u32(sm.stages + size_t(stage) * kStageBytes));
                    const uint32_t b_lo = a_lo + (kABytes >> 4);
                    if (lane == 0) {
#pragma unroll
                        for (int k = 0; k < kMmasPerStage; k++)
                            umma2<T>(tmem_d, hi | uint64_t(a_lo + 2 * k), hi | uint64_t(b_lo + 2 * k), idesc, (it != 0 || k != 0) ? 1u : 0u);
                        umma2_commit(&sm.empty[stage]);
                    }
                    __syncwarp();
                    if (++stage == p.stages) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
                if (lane == 0) umma2_commit(&sm.tmem_full[buf]);  // accumulator complete in both CTAs -> both epilogues
                __syncwarp();
            }
        }
    } else {
        // ------------------------------------------------------------------ epilogue (warps 2..5), each CTA drains its own 128 rows
        const int quarter = warp % 4;  // TMEM lanes [32*quarter, 32*quarter+32) are the ones this warp may read
        uint8_t* stg = sm.staging + size_t(quarter) * kStgBufs * kStgBytes;
        uint64_t* res_bar = sm.res_full + quarter * kStgBufs;
        const bool has_res = !kHead && p.has_res;
        const bool relu = p.relu_n > 0;  // tower form: whole layers only (relu_n is 0 or n)
        const uint32_t cpi = uint32_t(n_eff / kChunk);  // chunks per work item
        const uint32_t local_items = cluster_id < num_items ? uint32_t((num_items - cluster_id + num_clusters - 1) / num_clusters) : 0u;
        const uint32_t total = local_items * cpi;
        // chunk f of this warp: rows [row0, row0 + 32), output channels [col0, col0 + 32)
        auto coords = [&](uint32_t f, int& row0, int& col0) {
            const uint32_t li = f / cpi, c = f - li * cpi;
            const int item = cluster_id + int(li) * num_clusters;
            row0 = (2 * (item / p.n_split) + int(rank)) * kTileM + quarter * 32;
            col0 = (item % p.n_split) * n_eff + int(c) * kChunk;
        };
        auto load_res = [&](uint32_t f) {  // lane 0: residual box of chunk f into its staging buffer
            int row0, col0;
            coords(f, row0, col0);
            mbar_expect_tx(&res_bar[f % kStgBufs], kStgBytes);
            tma_load_2d(&tmap_res, &res_bar[f % kStgBufs], stg + (f % kStgBufs) * kStgBytes, col0, row0);
        };
        if (p.pdl) grid_dep_wait();  // the residual rows are the previous layers' output
        if (has_res && lane == 0) {
            if (total > 0) load_res(0);
            if (total > 1) load_res(1);
        }
        // 16-byte chunk index ^ the address bits above the row: SWIZZLE_64B (64-byte bf16 rows) bits 7..8, SWIZZLE_128B (128-byte f32
        // rows) bits 7..9
        const int sw = sizeof(Out) == 4 ? (lane & 7) : ((lane >> 1) & 3);
        constexpr int kVec = 16 / int(sizeof(Out));  // channels per 16-byte unit
#pragma unroll 1
        for (uint32_t f = 0; f < total; f++) {
            const uint32_t li = f / cpi, c = f - li * cpi, buf = li & 1, sb = f % kStgBufs;
            int row0, col0;
            coords(f, row0, col0);
            float bias[kChunk];  // one 128-byte line, the same address in every lane (a broadcast); issued before the waits below
#pragma unroll
            for (int j = 0; j < kChunk / 4; j++) {
                const float4 b = __ldg(reinterpret_cast<const float4*>(p.bias + col0) + j);
                bias[4 * j] = b.x;
                bias[4 * j + 1] = b.y;
                bias[4 * j + 2] = b.z;
                bias[4 * j + 3] = b.w;
            }
            if (c == 0) {
                mbar_wait(&sm.tmem_full[buf], (li >> 1) & 1);
                tc_fence_after();
            }
            uint32_t r[32];
            tmem_ld32(tmem_base + buf * acc_stride + (uint32_t(quarter * 32) << 16) + c * kChunk, r);
            tmem_ld_wait();
            if (c == cpi - 1) {  // the accumulator is in registers: the MMAs of the tile after next may overwrite it
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_remote(&sm.tmem_empty[buf], 0);  // the leader's barrier, from either CTA
            }
            if (has_res) {
                mbar_wait(&res_bar[sb], (f / kStgBufs) & 1);
            } else {
                if (lane == 0) tma_store_wait_read<kStgBufs - 1>();  // the store that last read this buffer (chunk f - 4) is done with it
                __syncwarp();
            }
            uint8_t* row_ptr = stg + sb * kStgBytes + lane * (kChunk * int(sizeof(Out)));
#pragma unroll
            for (int j = 0; j < kChunk / kVec; j++) {  // kVec channels = one 16-byte unit of the row
                float v[kVec];
#pragma unroll
                for (int k = 0; k < kVec; k++) {
                    float x = __uint_as_float(r[j * kVec + k]) + bias[j * kVec + k];
                    if constexpr (kHead)
                        v[k] = (col0 + j * kVec + k < p.relu_n && x < 0.0f) ? 0.0f : x;
                    else
                        v[k] = relu ? (x < 0.0f ? 0.0f : x) : x;  // NaN stays NaN, like torch / ONNX Relu
                }
                uint4* cell = reinterpret_cast<uint4*>(row_ptr + ((j ^ sw) << 4));
                if constexpr (kHead) {
                    *cell = make_uint4(__float_as_uint(v[0]), __float_as_uint(v[1]), __float_as_uint(v[2]), __float_as_uint(v[3]));
                } else if constexpr (sizeof(T) == 4) {
                    if (has_res) {  // the reference block is x + relu(bn(conv(...))): relu BEFORE the add (post_act.py:218-228)
                        const uint4 q = *cell;
                        v[0] += __uint_as_float(q.x);
                        v[1] += __uint_as_float(q.y);
                        v[2] += __uint_as_float(q.z);
                        v[3] += __uint_as_float(q.w);
                    }
                    *cell = make_uint4(__float_as_uint(tf32_round(v[0])), __float_as_uint(tf32_round(v[1])), __float_as_uint(tf32_round(v[2])),
                                       __float_as_uint(tf32_round(v[3])));
                } else {
                    if (has_res) {  // the reference block is x + relu(bn(conv(...))): relu BEFORE the add (post_act.py:218-228)
                        const uint4 q = *cell;
                        const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&q);
#pragma unroll
                        for (int k = 0; k < 4; k++) {
                            const float2 t = __bfloat1622float2(h[k]);
                            v[2 * k] += t.x;
                            v[2 * k + 1] += t.y;
                        }
                    }
                    *cell = make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
                }
            }
            fence_proxy_async_smem();  // generic-proxy writes -> visible to the TMA store
            __syncwarp();
            if (lane == 0) {
                tma_store_2d(&tmap_out, stg + sb * kStgBytes, col0, row0);
                tma_store_commit();
                if (has_res && f + 2 < total) {
                    tma_store_wait_read<2>();  // buffer (f + 2) % 4 was last read by the store of chunk f - 2
                    load_res(f + 2);
                }
            }
        }
        if (lane == 0) tma_store_wait_all();
    }

    tc_fence_before();
    __syncthreads();
    cluster_sync_all();  // no CTA leaves while the pair may still read its shared memory or signal its barriers
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(uint32_t(p.tmem_cols))
                     : "memory");
    }
}

}  // namespace

// the same for every layer width: the ring holds up to 128 weight rows per CTA (a slice of <= 256 channels), biases are not staged;
// out_esz: bytes per output element (2: bf16 tower layers, 4: TF32 tower layers and every head conv)
size_t conv_i2c_smem_bytes(int stages, int out_esz) {
    return 1024 /*alignment slack*/ + size_t(stages) * kStageBytes + 4 * kStgBufs * (32 * kChunk * size_t(out_esz)) + (2 * stages + 4 + 4 * kStgBufs) * 8 + 16;
}

// bf16 output: 6 stages; f32 output: 5 (its staging boxes take 32 KB more)
int conv_i2c_pick_stages(int out_esz) {
    const size_t budget = 227 * 1024;
    int stages = 6;
    while (stages > 2 && conv_i2c_smem_bytes(stages, out_esz) > budget) stages--;
    return stages;
}

void conv_i2c_prepare() {
    cudaFuncSetAttribute(conv_i2c_kernel<__nv_bfloat16, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    cudaFuncSetAttribute(conv_i2c_kernel<float, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    cudaFuncSetAttribute(conv_i2c_kernel<__nv_bfloat16, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    cudaFuncSetAttribute(conv_i2c_kernel<float, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
}

// tmap_a: im2col map over the dense channels-last activations (C, W, H, boards), one k-block x 128 pixels per load, SWIZZLE_128B;
// tmap_bh: weight map whose box holds p.n / p.n_split / 2 rows (this CTA's half of a slice); tmap_out / tmap_res: output / residual rows, box (32 channels, 32 rows),
// SWIZZLE_64B for bf16, SWIZZLE_128B for f32 (tmap_res is only read when p.has_res is set)
void launch_conv_i2c(const CUtensorMap& tmap_a, const CUtensorMap& tmap_bh, const CUtensorMap& tmap_out, const CUtensorMap& tmap_res,
                     const ConvTcParams& p, int grid, cudaStream_t s) {
    if (p.num_tiles <= 0) return;
    const int items = (p.num_tiles + 1) / 2 * p.n_split;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(unsigned(2 * std::min(grid / 2, items)));
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = conv_i2c_smem_bytes(p.stages, p.tf32 || p.head ? 4 : 2);
    cfg.stream = s;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = p.pdl ? 2 : 1;
    auto kernel = p.head ? (p.tf32 ? conv_i2c_kernel<float, true> : conv_i2c_kernel<__nv_bfloat16, true>)
                         : (p.tf32 ? conv_i2c_kernel<float, false> : conv_i2c_kernel<__nv_bfloat16, false>);
    cudaLaunchKernelEx(&cfg, kernel, tmap_a, tmap_bh, tmap_out, tmap_res, p);
}

}  // namespace kzb
