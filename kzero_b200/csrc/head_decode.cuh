// The output decode of packed evaluations, shared by both head kernels (heads.cu, heads8.cu): the GPU form of the reference's
// decode_output (rust/kz-core/src/network/common.rs:16-114), one warp per board.  The kernels differ in how they compute the
// scalars and gather a logit; what the reference does with them lives here only.
#pragma once
#include "kernels.cuh"

namespace kzb {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// a softmax sum of board b is not > 0 (NaN logits): the reference panics here (common.rs:110); err_flag may be host memory
__device__ __forceinline__ void report_bad_sum(const HeadOutputs& o, int b) { *reinterpret_cast<volatile int*>(o.err_flag) = 1 + b; }

// lane 0: value = tanh(s0), wdl = softmax(s1..3), moves_left = s4 (common.rs:59-74)
__device__ __forceinline__ void decode_values(const float sc[5], int b, const HeadOutputs& o) {
    float* ov = o.out_values + size_t(b) * 5;
    ov[0] = tanhf(sc[0]);
    float mx = fmaxf(sc[1], fmaxf(sc[2], sc[3]));
    float e0 = expf(sc[1] - mx), e1 = expf(sc[2] - mx), e2 = expf(sc[3] - mx);
    float sum = (e0 + e1) + e2;
    if (!(sum > 0.0f)) report_bad_sum(o, b);
    ov[1] = e0 / sum;
    ov[2] = e1 / sum;
    ov[3] = e2 / sum;
    ov[4] = sc[4];
}

// whole warp: softmax over the legal moves of board b only (common.rs:76-86 + softmax_in_place :102-114).  Legal index
// mv_idx[j] is remapped through the board's symmetry, then logit(i) gives policy entry i; an index outside the policy gets a NaN
// logit, which the sum check reports.  Lists of up to 32 * kRegMoves moves keep their logits in registers; longer ones gather
// every logit again in each pass rather than staging it in out_probs, which may be host memory.  Either way each lane adds its
// own moves in ascending order, so both forms give the same bits.
template <int kRegMoves, class Logit>
__device__ __forceinline__ void legal_softmax(const HeadOutputs& o, int b, int lane, Logit logit) {
    const uint32_t o0 = o.mv_off[b], o1 = o.mv_off[b + 1];
    const int n = int(o1 - o0);
    if (n <= 0) return;  // terminal board: empty policy (common.rs:77)
    const int32_t* pmap = o.sym ? o.policy_map + size_t(o.sym[b]) * o.policy_len : nullptr;
    auto gather = [&](int j) -> float {
        uint32_t idx = o.mv_idx[o0 + j];
        if (pmap && idx < uint32_t(o.policy_len)) idx = uint32_t(pmap[idx]);
        return idx < uint32_t(o.policy_len) ? logit(int(idx)) : NAN;
    };
    float mx = -INFINITY, sum = 0.0f;
    if (n <= 32 * kRegMoves) {
        float l[kRegMoves];
#pragma unroll
        for (int k = 0; k < kRegMoves; k++) {
            const int j = lane + 32 * k;
            l[k] = -INFINITY;
            if (j < n) {
                l[k] = gather(j);
                mx = fmaxf(mx, l[k]);
            }
        }
        mx = warp_max(mx);
#pragma unroll
        for (int k = 0; k < kRegMoves; k++) {
            const int j = lane + 32 * k;
            if (j < n) {
                l[k] = expf(l[k] - mx);
                sum += l[k];
            }
        }
        sum = warp_sum(sum);
        if (!(sum > 0.0f) && lane == 0) report_bad_sum(o, b);
#pragma unroll
        for (int k = 0; k < kRegMoves; k++) {
            const int j = lane + 32 * k;
            if (j < n) o.out_probs[o0 + j] = l[k] / sum;
        }
        return;
    }
    for (int j = lane; j < n; j += 32) mx = fmaxf(mx, gather(j));
    mx = warp_max(mx);
    for (int j = lane; j < n; j += 32) sum += expf(gather(j) - mx);
    sum = warp_sum(sum);
    if (!(sum > 0.0f) && lane == 0) report_bad_sum(o, b);
    for (int j = lane; j < n; j += 32) o.out_probs[o0 + j] = expf(gather(j) - mx) / sum;
}

}  // namespace kzb
