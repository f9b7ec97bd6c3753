// K3: everything after the head convolutions, one warp per position, warp-shuffle reductions.
//
// Replaces, for this path:
//   - the scalar head's Flatten/Gemm/Relu/Gemm steps (python/lib/model/post_act.py:15-19), which the
//     reference executes as separate cuBLAS launches,
//   - the policy Flatten/Gather/Concat plumbing (post_act.py:76-88, 102-112) and the attention head's
//     slice / reshape / bmm / scale / Gather chain (post_act.py:130-141), evaluated only for the requested indices,
//   - and, in packed mode, the CPU-side decode_output (rust/kz-core/src/network/common.rs:16-100):
//     value = tanh(s0), wdl = softmax(s1..3), moves_left = s4, policy = softmax over the LEGAL moves only
//     (gathered by the host-supplied move_to_index list), so only n_legal probabilities per position cross
//     PCIe instead of the full [B, P] logit matrix.  The decode itself is shared with heads8.cu (head_decode.cuh).
// HBM/latency-bound: algorithmic bytes per position = hc*A*4 + (n_legal or P)*4 read, (5 + n_legal or P)*4 written.
#include "head_decode.cuh"

namespace kzb {
namespace {

constexpr int kWarpsPerBlock = 4;
constexpr int kMaxHiddenPerLane = 4;  // hs <= 128
constexpr size_t kMaxSmem = 227 * 1024;

// STAGED: the warp copies its board's fc1 inputs to shared memory first (kWarpsPerBlock * hc * area floats a block).  Boards too
// large for that (above about 60 x 60 squares at hc = 4, go-256 at any hc) read them from global memory instead, in the same order,
// so both forms give the same bits.
template <bool PACKED, int HPL, bool STAGED>  // HPL = hidden units per lane = ceil(hs / 32)
__global__ void __launch_bounds__(kWarpsPerBlock * 32) heads_tail_kernel(HeadsTailParams p) {
    extern __shared__ float smem[];
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    const int b = blockIdx.x * kWarpsPerBlock + warp;
    if (b >= p.out.batch) return;  // whole warp exits together, no block-level sync below

    const int area = p.lay.W * p.lay.H;
    const int n_in = p.hc * area;
    float* s_in = smem + size_t(warp) * n_in;  // flatten order (channel, y, x), post_act.py:16
    auto fc1_in = [&](int i) -> float {
        return STAGED ? s_in[i] : p.s1[size_t(p.lay.row(b, i % area)) * p.s1_stride + i / area];
    };

    if (STAGED)
        for (int i = lane; i < n_in; i += 32) {
            int c = i / area, sq = i % area;
            s_in[i] = p.s1[size_t(p.lay.row(b, sq)) * p.s1_stride + c];
        }
    float extra = 0.0f;
    if (p.extra_w) {
        float e = 0.0f;
        for (int sq = lane; sq < area; sq += 32) e += p.extra_w[sq] * p.s1[size_t(p.lay.row(b, sq)) * p.s1_stride + p.hc];
        extra = warp_sum(e) + p.extra_b;
    }
    __syncwarp();

    // fc1 + relu: lane owns hidden units lane, lane+32, ...; 8 inputs per step so 8*HPL independent
    // weight loads are in flight (the loop is latency-bound otherwise); accumulation order stays i-ascending
    float h[HPL];
#pragma unroll
    for (int u = 0; u < HPL; u++) h[u] = 0.0f;
    for (int i0 = 0; i0 < n_in; i0 += 8) {
        float w[8][HPL], v[8];
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const int i = i0 + k;
            const bool ok = i < n_in;
            v[k] = ok ? fc1_in(i) : 0.0f;
#pragma unroll
            for (int u = 0; u < HPL; u++) {
                const int j = lane + 32 * u;
                w[k][u] = (ok && j < p.hs) ? __ldg(p.fc1_t + size_t(i) * p.hs + j) : 0.0f;
            }
        }
#pragma unroll
        for (int k = 0; k < 8; k++)
#pragma unroll
            for (int u = 0; u < HPL; u++) h[u] = fmaf(w[k][u], v[k], h[u]);
    }
#pragma unroll
    for (int u = 0; u < HPL; u++) {
        const int j = lane + 32 * u;
        float t = j < p.hs ? h[u] + p.fc1_b[j] : 0.0f;
        h[u] = t < 0.0f ? 0.0f : t;
    }
    // fc2: 5 outputs
    float sc[5];
#pragma unroll
    for (int k = 0; k < 5; k++) {
        float part = 0.0f;
#pragma unroll
        for (int u = 0; u < HPL; u++) {
            int j = lane + 32 * u;
            if (j < p.hs) part = fmaf(p.fc2_w[k * p.hs + j], h[u], part);
        }
        sc[k] = warp_sum(part) + p.fc2_b[k];
    }

    auto logit = [&](int i) -> float {
        if (p.att_entries) {  // attention head: q_from(from square) . q_to(to square / under-promotion slot) / sqrt(Q)
            const AttEntryDev e = p.att_entries[i];
            const float* a = p.att + size_t(p.lay.row(b, e.a_sq)) * p.att_stride + e.a_chan;
            const float* c = p.att + size_t(p.lay.row(b, e.b_sq)) * p.att_stride + e.b_chan;
            float acc = 0.0f;
            for (int q = 0; q < p.att_q; q++) acc = fmaf(a[q * e.a_stride], c[q * e.b_stride], acc);
            return acc / p.att_div;
        }
        int src = p.policy_src[i];
        if (src >= 0) return p.pm[size_t(p.lay.row(b, src % area)) * p.pm_stride + src / area];
        return src == -1 ? 0.0f : extra;
    };

    if (!PACKED) {
        if (lane < 5) p.out.out_scalars[size_t(b) * 5 + lane] = sc[lane];
        for (int i = lane; i < p.out.policy_len; i += 32) p.out.out_logits[size_t(b) * p.out.policy_len + i] = logit(i);
        return;
    }
    if (lane == 0) decode_values(sc, b, p.out);
    legal_softmax<12>(p.out, b, lane, logit);  // up to 384 legal moves stay in registers (chess <= 218, go-19 <= 362)
}

}  // namespace

void heads_tail_prepare() {
#define KZB_OPT_IN(PACKED, HPL) \
    cudaFuncSetAttribute(heads_tail_kernel<PACKED, HPL, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kMaxSmem))
    KZB_OPT_IN(true, 1);
    KZB_OPT_IN(true, 2);
    KZB_OPT_IN(true, 4);
    KZB_OPT_IN(false, 1);
    KZB_OPT_IN(false, 2);
    KZB_OPT_IN(false, 4);
#undef KZB_OPT_IN
}

void launch_heads_tail(const HeadsTailParams& p, cudaStream_t s) {
    if (p.out.batch <= 0) return;
    int blocks = (p.out.batch + kWarpsPerBlock - 1) / kWarpsPerBlock;
    const size_t stage = size_t(kWarpsPerBlock) * p.hc * p.lay.W * p.lay.H * sizeof(float);
    const bool staged = stage <= kMaxSmem;
    const size_t smem = staged ? stage : 0;
    const int hpl = (p.hs + 31) / 32;
#define KZB_TAIL(PACKED, HPL)                                                                       \
    (staged ? heads_tail_kernel<PACKED, HPL, true><<<blocks, kWarpsPerBlock * 32, smem, s>>>(p) \
            : heads_tail_kernel<PACKED, HPL, false><<<blocks, kWarpsPerBlock * 32, smem, s>>>(p))
    if (p.out.packed) {
        if (hpl <= 1) KZB_TAIL(true, 1);
        else if (hpl == 2) KZB_TAIL(true, 2);
        else KZB_TAIL(true, 4);
    } else {
        if (hpl <= 1) KZB_TAIL(false, 1);
        else if (hpl == 2) KZB_TAIL(false, 2);
        else KZB_TAIL(false, 4);
    }
#undef KZB_TAIL
}

}  // namespace kzb
