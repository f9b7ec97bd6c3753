// Epilogue of conv_tc.cu: one epilogue warp drains its 32 TMEM lanes of one 128-row accumulator tile.
// tcgen05.ld -> +bias (BN folded on the host) -> relu -> +residual -> bf16 / f32 store.
// Order matters: the reference block is x + relu(bn(conv(...))), relu BEFORE the add (python/lib/model/post_act.py:218-228).
#pragma once
#include "kernels.cuh"
#include "tc_common.cuh"

namespace kzb {

// `quarter` = warp % 4 selects the TMEM lanes [32*quarter, 32*quarter+32) this warp may read; `tmem_acc` is the
// accumulator's TMEM address (lane 0); waits for `tmem_full` at `buf_phase`, arrives on `tmem_empty` when done.
// The accumulator's columns [0, n_cols) are output channels [ch_base, ch_base + n_cols) (a CTA that owns only part of
// the output channels passes its slice; `bias` always holds all of them).
__device__ __forceinline__ void conv_epilogue_tile(const ConvTcParams& p, const float* bias, int tile, int quarter, int lane, uint32_t tmem_acc,
                                                   uint64_t* tmem_full, uint32_t buf_phase, uint64_t* tmem_empty, int ch_base, int n_cols) {
    using namespace tc;
    const int row = tile * 128 + quarter * 32 + lane;
    const bool store = row < p.valid_rows;

    // residual row (bf16) prefetched into registers BEFORE waiting for the accumulator, so its global
    // latency hides behind the MMAs of this tile (first 128 channels; the rest is loaded in the loop)
    constexpr int kResPrefetch = 16;  // uint4 = 8 channels each
    uint4 resq[kResPrefetch];
    const bool has_res = p.res != nullptr && store;
    if (has_res) {
        const uint4* rp = reinterpret_cast<const uint4*>(static_cast<const __nv_bfloat16*>(p.res) + size_t(row) * p.res_stride + ch_base);
#pragma unroll
        for (int j = 0; j < kResPrefetch; j++)
            if (j * 8 < n_cols) resq[j] = rp[j];
    }

    mbar_wait(tmem_full, buf_phase);
    tc_fence_after();
    const uint32_t taddr = tmem_acc + (uint32_t(quarter * 32) << 16);

#pragma unroll
    for (int cc = 0; cc < 8; cc++) {  // 32 columns per iteration, n <= 256
        const int c0 = cc * 32;
        if (c0 >= n_cols) break;
        const bool second = c0 + 16 < n_cols;
        uint32_t r[32];
        tmem_ld16(taddr + c0, r);
        if (second) tmem_ld16(taddr + c0 + 16, r + 16);
        tmem_ld_wait();
#pragma unroll
        for (int h = 0; h < 2; h++) {
            if (h == 1 && !second) break;
            const int col = c0 + h * 16, ch = ch_base + col;
            float v[16];
#pragma unroll
            for (int j = 0; j < 16; j++) {
                float f = __uint_as_float(r[h * 16 + j]) + bias[ch + j];
                if (ch + j < p.relu_n) f = f < 0.0f ? 0.0f : f;  // NaN stays NaN, like torch/ONNX Relu
                v[j] = f;
            }
            if (has_res) {
                uint4 q0, q1;
                if (cc < kResPrefetch / 4) {
                    q0 = resq[cc * 4 + h * 2];
                    q1 = resq[cc * 4 + h * 2 + 1];
                } else {
                    const uint4* rp = reinterpret_cast<const uint4*>(static_cast<const __nv_bfloat16*>(p.res) + size_t(row) * p.res_stride + ch);
                    q0 = rp[0];
                    q1 = rp[1];
                }
                const __nv_bfloat16* h0 = reinterpret_cast<const __nv_bfloat16*>(&q0);
                const __nv_bfloat16* h1 = reinterpret_cast<const __nv_bfloat16*>(&q1);
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    v[j] += __bfloat162float(h0[j]);
                    v[8 + j] += __bfloat162float(h1[j]);
                }
            }
            if (store) {
                if (p.out_f32) {
                    float4* op = reinterpret_cast<float4*>(static_cast<float*>(p.out) + size_t(row) * p.out_stride + ch);
#pragma unroll
                    for (int j = 0; j < 4; j++) op[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                } else {
                    uint4* op = reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(p.out) + size_t(row) * p.out_stride + ch);
                    op[0] = make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
                    op[1] = make_uint4(pack_bf16(v[8], v[9]), pack_bf16(v[10], v[11]), pack_bf16(v[12], v[13]), pack_bf16(v[14], v[15]));
                }
            }
        }
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0 && tmem_empty != nullptr) mbar_arrive(tmem_empty);  // nullptr: the caller signals (a barrier in another CTA)
}

}  // namespace kzb
