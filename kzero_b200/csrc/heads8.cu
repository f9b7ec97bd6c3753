// K1' + K3 fused for 8x8 boards with a conv policy head: everything after the tower in ONE persistent launch.
//
// Replaces, for this case, three launches of the generic conv kernel (policy conv1 C->Cp + relu, policy conv2
// Cp->Pc, scalar conv C->hc + relu; python/lib/model/post_act.py:10-23,54-88) and the tail kernel (heads.cu), which
// together were 15 % of a chess 16x128 step although they hold < 1 % of its FLOPs: every one of them round-trips its
// activations through L2/HBM (the fp32 policy map alone is 21 MB per 1024-board batch) and pays a launch + pipeline
// fill for two k-blocks of work.  Here a 128-row tile (= 2 boards) never leaves the SM:
//
//   TMA   X tile [128 pos][C] (bf16, SWIZZLE_128B)                                        2-stage ring
//   MMA1  D1[128 x Cp] = X . W1^T        MMA3  Ds[128 x 16] = X . Ws^T                    (weights resident in smem)
//   epi1  D1 + b1 -> relu -> bf16 -> H tile in shared memory, written directly in the K-major SWIZZLE_128B operand
//         layout (thread = position = TMEM lane, so a thread owns whole 16-byte channel chunks of its row);
//         Ds + bs -> relu -> S[board][c*64 + sq] (flatten order (channel, y, x), post_act.py:16)
//   MMA2  D2[128 x Pc] = H . W2^T
//   epi2  D2 + b2 -> fp32 logits L[board][pc*64 + sq] in shared memory (aliases H)
//   tail  per board: fc1 + relu + fc2 (post_act.py:17-19); then either
//           packed: value = tanh, wdl = softmax, legal-move gather through policy_src + softmax over the legal moves
//                   only (rust/kz-core/src/network/common.rs:59-86,102-114; shared with heads.cu in head_decode.cuh), or
//           planes: raw scalars + all P logits (twin of CudaExecutor::evaluate, network/cudnn.rs:73)
// MMA1/MMA3 of tile t+1 overlap epi2 + tail of tile t (D1/Ds are free once epi1 has drained them).
// Warp roles: warp 0 TMA producer, warp 1 MMA issuer (+TMEM owner), warps 2..5 epilogue/tail (thread = tile row).
#include "head_decode.cuh"
#include "tc_common.cuh"

namespace kzb {
namespace {

using namespace tc;

constexpr int kThreads = 192;
constexpr int kTile = 16384;   // one [128 rows][64 k] bf16 operand tile
constexpr int kXStages = 2;
constexpr int kMaxKb = 2;      // C, Cp <= 128
constexpr int kD1Col = 0, kD2Col = 128, kDsCol = 256;

struct SmemH {
    uint8_t* w1;   // kb x [n1][64]
    uint8_t* w2;   // kb2 x [n2][64]
    uint8_t* ws;   // kb x [16][64]
    uint8_t* x;    // kXStages x kb x 16 KiB
    uint8_t* hl;   // H: kb2 x 16 KiB, later the logits L [2][pc*64] f32
    float* s;      // [2][hc*64]
    float* fc1t;   // [hc*64][hs]
    float* b1;     // [n1]
    float* b2;     // [n2]
    float* bs;     // [16]
    uint64_t *w_full, *x_full, *x_empty, *d1_full, *h_full, *d2_full, *d2_free;
    uint32_t* tmem_ptr;
};

__host__ __device__ inline size_t hl_bytes(int kb2, int pc) {
    size_t h = size_t(kb2) * kTile, l = size_t(2) * pc * 64 * 4;
    return ((h > l ? h : l) + 1023) / 1024 * 1024;
}

__device__ __forceinline__ SmemH carve_h(uint8_t* base, const Heads8Params& p) {
    SmemH s;
    const int kb = p.kblocks, kb2 = p.n1 / 64;
    s.w1 = base;
    s.w2 = s.w1 + size_t(kb) * p.n1 * 128;
    s.ws = s.w2 + size_t(kb2) * p.n2 * 128;
    s.x = s.ws + size_t(kb) * 16 * 128;
    s.x = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(s.x) + 1023) & ~uintptr_t(1023));
    s.hl = s.x + size_t(kXStages) * kb * kTile;
    uint8_t* q = s.hl + hl_bytes(kb2, p.pc);
    s.s = reinterpret_cast<float*>(q);
    s.fc1t = s.s + 2 * p.hc * 64;
    s.b1 = s.fc1t + size_t(p.hc) * 64 * p.hs;
    s.b2 = s.b1 + p.n1;
    s.bs = s.b2 + p.n2;
    s.w_full = reinterpret_cast<uint64_t*>((reinterpret_cast<uintptr_t>(s.bs + 16) + 7) & ~uintptr_t(7));
    s.x_full = s.w_full + 1;
    s.x_empty = s.x_full + kXStages;
    s.d1_full = s.x_empty + kXStages;
    s.h_full = s.d1_full + 1;
    s.d2_full = s.h_full + 1;
    s.d2_free = s.d2_full + 1;
    s.tmem_ptr = reinterpret_cast<uint32_t*>(s.d2_free + 1);
    return s;
}

__device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 1, 128;" ::: "memory"); }

__global__ void __launch_bounds__(kThreads, 1)
    heads8_kernel(const __grid_constant__ Heads8Maps maps, const Heads8Params p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const SmemH sm = carve_h(smem, p);
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    const int kb = p.kblocks, kb2 = p.n1 / 64;
    // development aid: stamps [0] kernel start, [1] setup done, [2] end; per tile t (8 + 8t + k):
    //   k=0 d1_full seen, 1 epi1 done, 2 d2_full seen, 3 epi2 done (after barrier), 4 tail done, 5 MMA1 issued, 6 MMA2 issued
    unsigned long long* tl = p.timeline ? p.timeline + size_t(blockIdx.x) * 1024 : nullptr;
#define KZB_HSTAMP(t, k) do { if (tl && (t) < 100 && lane == 0) tl[8 + (t) * 8 + (k)] = clock64(); } while (0)
    if (tl && threadIdx.x == 0) tl[0] = clock64();

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&maps.x)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&maps.w1)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&maps.w2)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&maps.ws)) : "memory");
        mbar_init(sm.w_full, 1);
        for (int i = 0; i < kXStages; i++) {
            mbar_init(&sm.x_full[i], 1);
            mbar_init(&sm.x_empty[i], 1);
        }
        mbar_init(sm.d1_full, 1);
        mbar_init(sm.h_full, 128);
        mbar_init(sm.d2_full, 1);
        mbar_init(sm.d2_free, 128);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(sm.tmem_ptr)), "r"(512u)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *sm.tmem_ptr;
    if (tl && threadIdx.x == 0) tl[1] = clock64();

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer
        if (lane == 0) {
            // everything that stays resident: the three weight matrices (TMA tiles), biases and the fc1 matrix (bulk copies)
            const uint32_t fc1_bytes = uint32_t(p.hc) * 64 * p.hs * 4;
            mbar_expect_tx(sm.w_full, uint32_t(kb * p.n1 * 128 + kb2 * p.n2 * 128 + kb * 16 * 128) + fc1_bytes +
                                          uint32_t(p.n1 + p.n2 + 16) * 4);
            bulk_load_1d(sm.w_full, sm.fc1t, p.fc1_t, fc1_bytes);
            bulk_load_1d(sm.w_full, sm.b1, p.b1, uint32_t(p.n1) * 4);
            bulk_load_1d(sm.w_full, sm.b2, p.b2, uint32_t(p.n2) * 4);
            bulk_load_1d(sm.w_full, sm.bs, p.bs, 64);
            for (int k = 0; k < kb; k++) {
                tma_load_2d(&maps.w1, sm.w_full, sm.w1 + size_t(k) * p.n1 * 128, k * 64, 0);
                tma_load_2d(&maps.ws, sm.w_full, sm.ws + size_t(k) * 16 * 128, k * 64, 0);
            }
            for (int k = 0; k < kb2; k++) tma_load_2d(&maps.w2, sm.w_full, sm.w2 + size_t(k) * p.n2 * 128, k * 64, 0);
            if (p.pdl) grid_dep_wait();  // the tower's output rows; the weights above do not depend on it
            int stage = 0;
            uint32_t phase = 0;
            for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
                mbar_wait(&sm.x_empty[stage], phase ^ 1);
                mbar_expect_tx(&sm.x_full[stage], uint32_t(kb * kTile));
                for (int k = 0; k < kb; k++)
                    tma_load_2d(&maps.x, &sm.x_full[stage], sm.x + (size_t(stage) * kb + k) * kTile, k * 64, tile * 128);
                if (++stage == kXStages) {
                    stage = 0;
                    phase ^= 1;
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer
        const uint32_t idesc1 = umma_idesc_bf16(128, p.n1), idesc2 = umma_idesc_bf16(128, p.n2), idescs = umma_idesc_bf16(128, 16);
        const uint64_t hi = umma_desc_sw128_hi();
        mbar_wait(sm.w_full, 0);
        int stage = 0;
        uint32_t phase = 0;
        int local = 0;
        for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, local++) {
            const uint32_t par = uint32_t(local) & 1;
            // MMA1 + MMA3: D1 / Ds were drained by epi1 of the previous tile (implied by the h_full wait below)
            mbar_wait(&sm.x_full[stage], phase);
            tc_fence_after();
            if (lane == 0) {
                for (int k = 0; k < kb; k++) {
                    const uint32_t a_lo = umma_desc_lo(smem_u32(sm.x + (size_t(stage) * kb + k) * kTile));
                    const uint32_t b_lo = umma_desc_lo(smem_u32(sm.w1 + size_t(k) * p.n1 * 128));
                    const uint32_t s_lo = umma_desc_lo(smem_u32(sm.ws + size_t(k) * 16 * 128));
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        umma_bf16(tmem_base + kD1Col, hi | uint64_t(a_lo + 2 * j), hi | uint64_t(b_lo + 2 * j), idesc1, (k | j) != 0);
                        umma_bf16(tmem_base + kDsCol, hi | uint64_t(a_lo + 2 * j), hi | uint64_t(s_lo + 2 * j), idescs, (k | j) != 0);
                    }
                }
                umma_commit(&sm.x_empty[stage]);
                umma_commit(sm.d1_full);
            }
            KZB_HSTAMP(local, 5);
            __syncwarp();
            if (++stage == kXStages) {
                stage = 0;
                phase ^= 1;
            }
            // MMA2 once epi1 has written H, and epi2 of the previous tile has drained D2
            mbar_wait(sm.h_full, par);
            if (local > 0) mbar_wait(sm.d2_free, uint32_t(local - 1) & 1);
            tc_fence_after();
            if (lane == 0) {
                for (int k = 0; k < kb2; k++) {
                    const uint32_t a_lo = umma_desc_lo(smem_u32(sm.hl + size_t(k) * kTile));
                    const uint32_t b_lo = umma_desc_lo(smem_u32(sm.w2 + size_t(k) * p.n2 * 128));
#pragma unroll
                    for (int j = 0; j < 4; j++)
                        umma_bf16(tmem_base + kD2Col, hi | uint64_t(a_lo + 2 * j), hi | uint64_t(b_lo + 2 * j), idesc2, (k | j) != 0);
                }
                umma_commit(sm.d2_full);
            }
            KZB_HSTAMP(local, 6);
            __syncwarp();
        }
    } else {
        // ------------------------------------------------------------------ epilogue + tail (warps 2..5)
        const int quarter = warp % 4;
        const int row = quarter * 32 + lane;  // tile row = TMEM lane = board_in_tile * 64 + square
        const int tb = row >> 6, sq = row & 63;
        const uint32_t lane_addr = tmem_base + (uint32_t(quarter * 32) << 16);
        float* const L = reinterpret_cast<float*>(sm.hl);
        const int n_in = p.hc * 64;
        int local = 0;
        mbar_wait(sm.w_full, 0);  // biases + fc1 matrix are in shared memory
        for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, local++) {
            const uint32_t par = uint32_t(local) & 1;
            // every warp is done reading L / S of the previous tile before H / S are overwritten
            epi_bar();
            if (warp == 2 && local > 0) KZB_HSTAMP(local - 1, 4);
            mbar_wait(sm.d1_full, par);
            tc_fence_after();
            if (warp == 2) KZB_HSTAMP(local, 0);
            // ---- epi1: scalar conv -> S, policy conv1 -> H
            {
                uint32_t r[16];
                tmem_ld16(lane_addr + kDsCol, r);
                tmem_ld_wait();
                float bias[16];
#pragma unroll
                for (int c = 0; c < 16; c++) bias[c] = sm.bs[c];
#pragma unroll
                for (int c = 0; c < 16; c++) {
                    if (c < p.hc) {
                        float f = __uint_as_float(r[c]) + bias[c];
                        sm.s[tb * n_in + c * 64 + sq] = f < 0.0f ? 0.0f : f;
                    }
                }
            }
            for (int c0 = 0; c0 < p.n1; c0 += 32) {
                uint32_t r[32];
                tmem_ld32(lane_addr + kD1Col + c0, r);
                float bias[32];  // loaded before any store of this chunk (see epi2)
#pragma unroll
                for (int j = 0; j < 32; j++) bias[j] = sm.b1[c0 + j];
                tmem_ld_wait();
                uint8_t* hrow = sm.hl + size_t(c0 >> 6) * kTile + row * 128;
#pragma unroll
                for (int g = 0; g < 4; g++) {  // 8 channels = one 16-byte chunk of the 128-byte row, swizzled by the row
                    uint32_t pk[4];
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        float f0 = __uint_as_float(r[g * 8 + 2 * j]) + bias[g * 8 + 2 * j];
                        float f1 = __uint_as_float(r[g * 8 + 2 * j + 1]) + bias[g * 8 + 2 * j + 1];
                        f0 = f0 < 0.0f ? 0.0f : f0;
                        f1 = f1 < 0.0f ? 0.0f : f1;
                        pk[j] = pack_bf16(f0, f1);
                    }
                    const int chunk = ((c0 & 63) >> 3) + g;
                    *reinterpret_cast<uint4*>(hrow + ((chunk ^ (row & 7)) << 4)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // H (generic proxy) -> UMMA reads
            tc_fence_before();
            mbar_arrive(sm.h_full);
            if (warp == 2) KZB_HSTAMP(local, 1);

            // ---- epi2: policy conv2 -> fp32 logits L[board][pc*64 + sq]
            mbar_wait(sm.d2_full, par);
            tc_fence_after();
            if (warp == 2) KZB_HSTAMP(local, 2);
            for (int c0 = 0; c0 < p.n2; c0 += 16) {
                uint32_t r[16];
                tmem_ld16(lane_addr + kD2Col + c0, r);
                tmem_ld_wait();
                // biases first, then the stores: the compiler cannot move a shared-memory load across a shared-memory store
                // that may alias it, and with one warp per scheduler a load -> add -> store chain per element costs ~60 cycles
                float bias[16];
#pragma unroll
                for (int j = 0; j < 16; j++) bias[j] = sm.b2[c0 + j];
                float* lrow = L + size_t(tb * p.pc + c0) * 64 + sq;
#pragma unroll
                for (int j = 0; j < 16; j++)
                    if (c0 + j < p.pc) lrow[j * 64] = __uint_as_float(r[j]) + bias[j];
            }
            tc_fence_before();
            mbar_arrive(sm.d2_free);
            epi_bar();  // L and S complete
            if (warp == 2) KZB_HSTAMP(local, 3);

            // ---- tail: two warps per board; the even one runs the scalar head, both split the policy work
            const int b = tile * 2 + (quarter >> 1);
            if (b >= p.out.batch) continue;  // whole warps skip together; epi_bar at the loop top keeps the count (all 4 warps loop)
            const int wb = quarter >> 1, sub = quarter & 1;
            const float* S = sm.s + wb * n_in;
            const float* Lb = L + size_t(wb) * p.pc * 64;
            if (sub == 0) {
                // fc1 + relu: lane = hidden unit (hs <= 32), inputs ascending like the reference's Gemm
                float h = 0.0f;
                if (lane < p.hs) {
                    // four independent partial sums (inputs i = 4k + a) keep the FMA pipe busy; n_in is a multiple of 64
                    float h0 = 0.0f, h1 = 0.0f, h2 = 0.0f, h3 = 0.0f;
                    const float* w = sm.fc1t + lane;
#pragma unroll 4
                    for (int i = 0; i < n_in; i += 4) {
                        h0 = fmaf(w[(i + 0) * p.hs], S[i + 0], h0);
                        h1 = fmaf(w[(i + 1) * p.hs], S[i + 1], h1);
                        h2 = fmaf(w[(i + 2) * p.hs], S[i + 2], h2);
                        h3 = fmaf(w[(i + 3) * p.hs], S[i + 3], h3);
                    }
                    h = ((h0 + h1) + (h2 + h3)) + p.fc1_b[lane];
                    h = h < 0.0f ? 0.0f : h;
                }
                float sc[5];
#pragma unroll
                for (int k = 0; k < 5; k++) {
                    float part = lane < p.hs ? p.fc2_w[k * p.hs + lane] * h : 0.0f;
                    sc[k] = warp_sum(part) + p.fc2_b[k];
                }
                if (!p.out.packed) {
                    if (lane < 5) p.out.out_scalars[size_t(b) * 5 + lane] = sc[lane];
                } else if (lane == 0) {
                    decode_values(sc, b, p.out);
                }
            }
            auto logit = [&](int i) -> float {
                const int src = p.policy_src[i];
                return src >= 0 ? Lb[src] : 0.0f;  // -1: constant zero column
            };
            if (!p.out.packed) {
                for (int i = sub * 32 + lane; i < p.out.policy_len; i += 64) p.out.out_logits[size_t(b) * p.out.policy_len + i] = logit(i);
                continue;
            }
            if (sub == 1) legal_softmax<8>(p.out, b, lane, logit);  // up to 256 legal moves in registers (chess <= 218)
        }
    }

    tc_fence_before();
    __syncthreads();
    if (tl && threadIdx.x == 0) tl[2] = clock64();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

}  // namespace

size_t heads8_smem_bytes(const Heads8Params& p) {
    const int kb = p.kblocks, kb2 = p.n1 / 64;
    size_t b = 1024;
    b += size_t(kb) * p.n1 * 128 + size_t(kb2) * p.n2 * 128 + size_t(kb) * 16 * 128 + 1024;
    b += size_t(kXStages) * kb * kTile + hl_bytes(kb2, p.pc);
    b += (size_t(2) * p.hc * 64 + size_t(p.hc) * 64 * p.hs + p.n1 + p.n2 + 16) * 4;
    b += 16 * 8 + 64;
    return b;
}

bool heads8_supported(const Heads8Params& p) {
    return p.kblocks >= 1 && p.kblocks <= kMaxKb && p.n1 % 64 == 0 && p.n1 >= 64 && p.n1 <= 128 && p.n2 % 16 == 0 && p.n2 >= 16 &&
           p.n2 <= 128 && p.pc <= p.n2 && p.hc >= 1 && p.hc <= 15 && p.hs >= 1 && p.hs <= 32 && heads8_smem_bytes(p) <= 227 * 1024;
}

void heads8_prepare() { cudaFuncSetAttribute(heads8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024); }

void launch_heads8(const Heads8Maps& maps, const Heads8Params& p, int grid, cudaStream_t s) {
    if (p.num_tiles <= 0) return;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(unsigned(std::min(grid, p.num_tiles)));
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = heads8_smem_bytes(p);
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = p.pdl ? 1 : 0;
    cudaLaunchKernelEx(&cfg, heads8_kernel, maps, p);
}

}  // namespace kzb
