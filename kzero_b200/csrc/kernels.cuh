// Device-side parameter blocks and host launchers for the hot path's kernels (sm_100a only).
//   K2  encode      packed bitboards + scalars -> input planes          (encode.cu)      HBM-bound
//   K1  conv tower  implicit-GEMM conv3x3/1x1 on tcgen05 + TMA + TMEM   (tower8k.cu, conv_i2c.cu)  tensor-bound
//       conv fp32   CUDA-core fp32 implicit GEMM, the <=1e-4 parity mode (conv_fp32.cu)
//   K3  heads tail  scalar-head FCs, policy gather, masked softmax      (heads.cu, decode: head_decode.cuh)  HBM/latency-bound
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <cstring>

namespace kzb {

// Element type of the activation rows: bf16 (tensor-core path), f32 (CUDA-core fp32 path), or f32 rounded to TF32 (tensor-core
// TF32 path: every value a kind::tf32 MMA reads is stored TF32-exact, see tf32_round)
enum class Act { kBf16, kF32, kTf32 };

// f32 -> the nearest TF32 value (round to nearest, ties away from zero, the low 13 mantissa bits cleared), as a float.  The rule of
// cvt.rna.tf32.f32; a value at or above the midpoint between the largest TF32 value and 2^128 becomes Inf.  Inf stays Inf, NaN stays
// NaN (a plain add-and-mask would turn a NaN whose payload sits in the low 13 bits into Inf).  Host (weights) and device (epilogues,
// encode) use this one definition.
__host__ __device__ __forceinline__ float tf32_round(float x) {
#ifdef __CUDA_ARCH__
    uint32_t u = __float_as_uint(x);
#else
    uint32_t u;
    std::memcpy(&u, &x, 4);
#endif
    if ((u & 0x7F800000u) != 0x7F800000u)
        u += 0x1000u;  // finite: half an ulp of TF32 on the magnitude, carries into the exponent
    else if (u & 0x007FFFFFu)
        u |= 0x00400000u;  // NaN: quiet bit set, so the payload survives the mask
    u &= 0xFFFFE000u;
#ifdef __CUDA_ARCH__
    return __uint_as_float(u);
#else
    std::memcpy(&x, &u, 4);
    return x;
#endif
}

// Row index of square sq = y * W + x of board b inside an activation matrix [rows][channels]: every row is a real square
struct RowLayout {
    int W, H;
    __host__ __device__ int row(int b, int sq) const { return b * W * H + sq; }
};

// ---------------------------------------------------------------------------------------------- K2
struct EncodeParams {
    const uint8_t* bits;   // [batch][bits_stride]   LSB-first (bit_buffer.rs:27-35)
    const float* scalars;  // [batch][scalar_count]
    int batch, bits_stride, scalar_count, bool_channels;
    RowLayout lay;
    int c_pad;  // channels per row in the output (>= scalar_count + bool_channels, multiple of 8)
    void* out;  // [batch*W*H][c_pad] bf16 or f32 (f32 rounded to TF32 for Act::kTf32)
    // optional board symmetry (RandomSymmetryNetwork on the GPU, network/symmetry.rs:41-67): plane square sq of board b is
    // read from square square_src[sym[b]*A + sq] of the record; null = identity
    const uint8_t* sym;
    const int32_t* square_src;
    // k-chunk-major output only: the record's own board (<= 8x8), embedded top-left in the 8x8 grid the tower works on
    int rec_w, rec_h;
};
void launch_encode_nhwc(const EncodeParams& p, Act out, cudaStream_t s);
// exact twin of InputMapper::encode_input_full (mapping/mod.rs:40-63): out [batch][Cs+Cb][H*W] f32
void launch_encode_nchw_f32(const uint8_t* bits, const float* scalars, int batch, int bits_stride, int scalar_count,
                            int bool_channels, int area, float* out, cudaStream_t s);
// f32 NCHW [batch][C][H*W] -> rows [batch*W*H][c_pad] of element type `out_type`, zero pad channels
void launch_nchw_to_rows(const float* in, int batch, int channels, RowLayout lay, int c_pad, void* out, Act out_type,
                         cudaStream_t s);

// ---------------------------------------------------------------------------------------------- conv fp32
struct ConvF32Params {
    const float* in;  // [rows][in_stride]
    int in_stride;
    const float* w;     // [taps][cin][cout]
    const float* bias;  // [cout]
    const float* res;   // optional [rows][res_stride], added AFTER the relu (post_act.py:227-228)
    int res_stride;
    float* out;  // [rows][out_stride]
    int out_stride;
    int cin, cout, taps;  // taps 1 or 9
    int relu_n;           // relu on output channels < relu_n
    int batch;
    RowLayout lay;  // dense
};
void launch_conv_fp32(const ConvF32Params& p, cudaStream_t s);

// ---------------------------------------------------------------------------------------------- K1
struct ConvTcParams {
    int num_tiles;  // 128-row M tiles
    int taps;       // 1 or 9
    int kblocks;    // cin_pad / (channels per 128-byte k-block: 64 bf16 or 32 TF32)
    int cin_pad;
    int n;  // padded cout, the MMA width: multiple of 32, <= 1024 (UMMA N = n / n_split <= 256)
    RowLayout lay;
    const float* bias;  // [n]
    int relu_n;         // relu on output channels < relu_n (tower form: 0 or n)
    int has_res;        // tower form: add the residual rows (tmap_res) after the relu
    int stages;
    int tmem_cols;
    int n_split;  // slices of the output channels; a work item is one 256-pixel tile x n / n_split channels (n / n_split <= 256, multiple of 32)
    int pdl;      // launched with programmatic stream serialization (set-up and the first weight tiles overlap the previous layer's tail)
    int tf32;     // operands and activations are f32 rounded to TF32 (tcgen05 kind::tf32, 32 channels per k-block); 0: bf16
    int head;     // head form: f32 output, not rounded, no residual (the head 1x1 convs); 0: tower form, output in the operand type
};
// conv_i2c.cu: conv3x3 / conv1x1 (p.taps) on DENSE rows, activation tiles by TMA im2col, CTA-pair MMA (tmap_bh: weight box of p.n / p.n_split / 2 rows)
void launch_conv_i2c(const CUtensorMap& tmap_a_im2col, const CUtensorMap& tmap_bh, const CUtensorMap& tmap_out, const CUtensorMap& tmap_res,
                     const ConvTcParams& p, int grid, cudaStream_t s);
size_t conv_i2c_smem_bytes(int stages, int out_esz);
int conv_i2c_pick_stages(int out_esz);  // out_esz: bytes per output element
void conv_i2c_prepare();  // per-device (every instance): opt in to 227 KB dynamic shared memory

// whole-tower persistent kernel for 8x8 boards (tower8k.cu)
struct TowerLayerDev {
    int a_map;   // input activations: 0 = encoded planes, 1 = X (residual stream), 2 = T (block-internal)
    int w_map;   // 0 = first-layer weights, 1 = concatenated block weights
    int w_row0;  // first row of this layer inside its weight matrix
    int kblocks, cin_pad;
    int relu_n;
    int has_res;  // add X (same rows) after the relu
    int out_buf;  // 1 = X, 2 = T
    const float* bias;
    // second-generation kernel (tower8k.cu)
    int kchunks;       // 8-channel chunks staged per k-block (8, fewer for a narrow first layer)
    int ksteps;        // K=16 MMA steps per k-block and tap (kchunks / 2)
    int out_rowmajor;  // last layer: store [position][C] rows (what the head kernels read) instead of k-chunk-major
};
struct Tower8Params {
    int num_layers;
    const TowerLayerDev* layers;  // device memory
    int num_units;                // 4-board work units
    int valid_rows;
    int n, n_store;
    __nv_bfloat16* x;
    __nv_bfloat16* t;
    __nv_bfloat16* xt;  // channel-major copy of the residual stream: [unit][128 channels][256 positions]
    int stride;  // elements per row of X / T
    int b_slots, tmem_cols;
    int cluster;  // 1: every CTA streams its own weight tiles; 2: CTA pairs, each loads half of every tile and multicasts it
    // tower8k only: the real board inside the 8x8 grid (ataxx 7x7, ...): outputs on squares outside it are forced to zero after
    // every layer, so that they keep acting as the convolution's zero padding
    int board_w, board_h;
    // tower8k only: balanced board assignment (CTA c owns bal_base + (c < bal_rem) contiguous boards as two units of 4 / 3)
    int balanced, bal_base, bal_rem, bal_grid;
    int pdl;  // launched with programmatic stream serialization: set-up overlaps the encode kernel, which runs right before it
    unsigned long long* timeline;
    int debug;  // development aid (KZB_DEBUG): 1 = skip A loads, 2 = skip B loads, 4 = skip epilogue memory traffic
};
// second generation (tower8k.cu): k-chunk-major activations A[kc][board][y][x][8], every tap = a descriptor offset
struct Tower8kMaps {
    // second index: boards per unit - 3 (units of 3 or 4 boards)
    CUtensorMap a[3][2];    // loads: encoded planes, X, T -- dims (x*8+c8: 64, board, y: 8, kc), box (72, nb, 9, 1), no swizzle
    CUtensorMap w[2];       // loads: first-layer weights, concatenated block weights -- box (64, n / cluster), SWIZZLE_128B
    CUtensorMap out[3][2];  // stores: X, T k-chunk-major -- dims (64, kc, board, y), box (80, 4, nb, 1); [2] = X row-major (c, x, board, y), box (32, 8, nb, 1)
};
void launch_tower8k(const Tower8kMaps& maps, const Tower8Params& p, int grid, cudaStream_t s);
size_t tower8k_smem_bytes(int w_slots);
int tower8k_pick_b_slots();
int tower8k_max_local_units();
void tower8k_prepare();

// K2 / layout twins for the k-chunk-major tower input: out[kc][boards_total][64 squares][8 channels] bf16
void launch_encode_kc(const EncodeParams& p, int kc_total, int boards_total, cudaStream_t s);
void launch_nchw_to_kc(const float* in, int batch, int channels, int rec_w, int rec_h, int kc_total, int boards_total, void* out,
                       cudaStream_t s);

// ---------------------------------------------------------------------------------------------- K3
struct AttEntryDev {  // same layout as NetSpec::AttEntry
    int32_t a_chan, a_stride, a_sq, b_chan, b_stride, b_sq;
};
// What a head kernel writes for one batch: the raw scalars and logits (planes mode), or their decode (packed mode, head_decode.cuh)
struct HeadOutputs {
    int batch, policy_len;
    int packed;
    // planes mode (twin of CudaExecutor::evaluate, network/cudnn.rs:73)
    float* out_scalars;  // [batch][5] raw
    float* out_logits;   // [batch][P]
    // packed mode (fused decode_output, network/common.rs:16-114)
    const uint32_t* mv_idx;  // legal moves' policy indices, CSR
    const uint32_t* mv_off;  // [batch+1]
    // optional symmetry: legal index i of board b is looked up at policy_map[sym[b]*P + i] (unmap_eval, symmetry.rs:126-148)
    const uint8_t* sym;
    const int32_t* policy_map;
    float* out_values;  // [batch][5]: tanh(v), softmax(wdl), moves_left
    float* out_probs;   // CSR-aligned with mv_idx
    int* err_flag;      // set to 1+board (any failing board) when a softmax sum is not > 0 (common.rs:110); may be host memory
};

struct HeadsTailParams {
    HeadOutputs out;
    RowLayout lay;
    const float* s1;  // [rows][s1_stride]: ch 0..hc-1 relu(scalar conv), ch hc = extra policy conv (no relu)
    int s1_stride, hc;
    const float* pm;  // [rows][pm_stride]: policy conv map, channel pc at [row][pc]
    int pm_stride;
    const float* fc1_t;  // [hc*A][hs]  (transposed fc1 weight)
    const float* fc1_b;  // [hs]
    const float* fc2_w;  // [5][hs]
    const float* fc2_b;  // [5]
    int hs;
    const float* extra_w;  // [A] or null
    float extra_b;
    const int32_t* policy_src;  // [P]; null for the attention head
    // attention policy head (post_act.py:115-141): logit[i] = dot_q(E[a.sq][a.chan + q*a.stride], E[b.sq][b.chan + q*b.stride]) / att_div
    const float* att;  // [rows][att_stride]: concatenated outputs of the head's 1x1 convs
    int att_stride, att_q;
    float att_div;
    const AttEntryDev* att_entries;  // [P] or null
};
void heads_tail_prepare();  // per-device: opt in to 227 KB dynamic shared memory for the staged fc1 inputs
void launch_heads_tail(const HeadsTailParams& p, cudaStream_t s);

// ---------------------------------------------------------------------------------------------- K1' + K3 fused (heads8.cu)
struct Heads8Maps {
    CUtensorMap x;   // tower output rows [rows][c_pad] bf16, box (64, 128), SWIZZLE_128B
    CUtensorMap w1;  // policy conv1 [n1][c_pad], box (64, n1)
    CUtensorMap w2;  // policy conv2 [n2][n1],    box (64, n2)
    CUtensorMap ws;  // scalar conv  [16][c_pad], box (64, 16)
};
struct Heads8Params {
    HeadOutputs out;
    int num_tiles;  // 128-row tiles = pairs of 8x8 boards
    int kblocks;    // c_pad / 64
    int n1, n2;     // padded output channels of policy conv1 (multiple of 64) / conv2 (multiple of 16)
    int pc;         // real output channels of policy conv2
    int hc, hs;     // scalar head: conv channels, hidden size (<= 32)
    const float *b1, *b2, *bs;  // [n1], [n2], [16]
    const float* fc1_t;         // [hc*64][hs]
    const float* fc1_b;         // [hs]
    const float* fc2_w;         // [5][hs]
    const float* fc2_b;         // [5]
    const int32_t* policy_src;  // [P]: pc*64 + sq, or -1 for a constant-zero logit
    int pdl;  // launched with programmatic stream serialization: set-up and the resident weights' loads overlap the tower's tail
    unsigned long long* timeline;  // development aid (KZB_TIMELINE=heads8): per-CTA clock64() stamps
};
size_t heads8_smem_bytes(const Heads8Params& p);
bool heads8_supported(const Heads8Params& p);
void heads8_prepare();
void launch_heads8(const Heads8Maps& maps, const Heads8Params& p, int grid, cudaStream_t s);

}  // namespace kzb
