// fp32-accurate conv (precision 0): CUDA-core implicit GEMM, plain FMA, no TF32, no tensor cores.
// Exists so the whole path can be checked against the oracle at <= 1e-4 max-abs (BASELINE.json
// north_star "fp32 path"), and so index arithmetic of the tensor-core path has an on-device twin.
// It is a correctness mode, not the throughput mode: the bf16 tcgen05 kernels in tower8k.cu and conv_i2c.cu are.
//
// GEMM view: M = positions (batch*H*W), N = cout, K = taps*cin.  Tile 64x64x16, 256 threads, 4x4 per thread.
#include "kernels.cuh"

namespace kzb {
namespace {

constexpr int BM = 64, BN = 64, BK = 16, THREADS = 256;

__global__ void __launch_bounds__(THREADS) conv_fp32_kernel(ConvF32Params p) {
    __shared__ float As[BK][BM + 4];
    __shared__ float Bs[BK][BN + 4];

    const int W = p.lay.W, H = p.lay.H, area = W * H;
    const int n_pos = p.batch * area;
    const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
    const int t = threadIdx.x;
    const int tx = t % 16, ty = t / 16;

    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) acc[i][j] = 0.0f;

    // A loader: thread loads rows (t/16 + 16*i), k = t%16
    const int ak = t % 16;
    int a_b[4], a_y[4], a_x[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        int m = m0 + t / 16 + 16 * i;
        if (m < n_pos) {
            a_b[i] = m / area;
            int sq = m % area;
            a_y[i] = sq / W;
            a_x[i] = sq % W;
        } else {
            a_b[i] = -1;
            a_y[i] = a_x[i] = 0;
        }
    }
    const int bn = t % 64, bk0 = t / 64;

    for (int tap = 0; tap < p.taps; tap++) {
        const int dy = p.taps == 9 ? tap / 3 - 1 : 0;
        const int dx = p.taps == 9 ? tap % 3 - 1 : 0;
        for (int c0 = 0; c0 < p.cin; c0 += BK) {
#pragma unroll
            for (int i = 0; i < 4; i++) {
                float v = 0.0f;
                int yy = a_y[i] + dy, xx = a_x[i] + dx, ci = c0 + ak;
                if (a_b[i] >= 0 && yy >= 0 && yy < H && xx >= 0 && xx < W && ci < p.cin)
                    v = p.in[size_t(p.lay.row(a_b[i], yy * W + xx)) * p.in_stride + ci];
                As[ak][t / 16 + 16 * i] = v;
            }
#pragma unroll
            for (int i = 0; i < 4; i++) {
                int k = bk0 + 4 * i, ci = c0 + k, co = n0 + bn;
                float v = 0.0f;
                if (ci < p.cin && co < p.cout) v = p.w[(size_t(tap) * p.cin + ci) * p.cout + co];
                Bs[k][bn] = v;
            }
            __syncthreads();
#pragma unroll
            for (int k = 0; k < BK; k++) {
                float a[4], b[4];
#pragma unroll
                for (int i = 0; i < 4; i++) a[i] = As[k][ty * 4 + i];
#pragma unroll
                for (int j = 0; j < 4; j++) b[j] = Bs[k][tx * 4 + j];
#pragma unroll
                for (int i = 0; i < 4; i++)
#pragma unroll
                    for (int j = 0; j < 4; j++) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
            }
            __syncthreads();
        }
    }

#pragma unroll
    for (int i = 0; i < 4; i++) {
        int m = m0 + ty * 4 + i;
        if (m >= n_pos) continue;
        size_t row = p.lay.row(m / area, m % area);
#pragma unroll
        for (int j = 0; j < 4; j++) {
            int co = n0 + tx * 4 + j;
            if (co >= p.cout) continue;
            float v = acc[i][j] + p.bias[co];
            if (co < p.relu_n) v = v < 0.0f ? 0.0f : v;  // NaN stays NaN, like torch/ONNX Relu
            if (p.res) v += p.res[row * p.res_stride + co];
            p.out[row * p.out_stride + co] = v;
        }
    }
}

}  // namespace

void launch_conv_fp32(const ConvF32Params& p, cudaStream_t s) {
    if (p.batch <= 0) return;
    int n_pos = p.batch * p.lay.W * p.lay.H;
    dim3 grid((n_pos + BM - 1) / BM, (p.cout + BN - 1) / BN);
    conv_fp32_kernel<<<grid, THREADS, 0, s>>>(p);
}

}  // namespace kzb
