// K2: board-to-plane input encoding on the GPU.
//
// Reference: InputMapper::encode_input_full, rust/kz-core/src/mapping/mod.rs:40-63 -- on the CPU, one
// Vec::push per f32, then a 5.5 MB (chess, batch 1024) H2D copy of f32 NCHW planes.  Here the host
// uploads the packed record ((bits, scalars), 136 B per chess position -- the same bytes
// BinaryOutput::append_position writes, rust/kz-selfplay/src/binary_output.rs:218-247) and this kernel
// expands it straight into the channels-last bf16 activation matrix the conv tower reads.
//
// HBM-bound: algorithmic bytes per position = packed record in + (Cs+Cb)*A*sizeof(elem) out.
// One CTA per board, record staged in shared memory, 16-byte vectorised fully coalesced stores.
#include "kernels.cuh"

namespace kzb {
namespace {

constexpr int kEncodeThreads = 128;

template <typename T>
struct Vec8;
template <>
struct Vec8<__nv_bfloat16> {
    uint4 v;
    __device__ void set(int i, float f) {
        __nv_bfloat16 h = __float2bfloat16_rn(f);
        reinterpret_cast<__nv_bfloat16*>(&v)[i] = h;
    }
    __device__ void store(void* base, size_t vec_index) const { reinterpret_cast<uint4*>(base)[vec_index] = v; }
};
template <>
struct Vec8<float> {
    float4 a, b;
    __device__ void set(int i, float f) { reinterpret_cast<float*>(this)[i] = f; }
    __device__ void store(void* base, size_t vec_index) const {
        reinterpret_cast<float4*>(base)[vec_index * 2] = a;
        reinterpret_cast<float4*>(base)[vec_index * 2 + 1] = b;
    }
};
struct Tf32;  // f32 rows whose values are rounded to TF32: what the TF32 precision's first conv reads (scalar planes need not be exact)
template <>
struct Vec8<Tf32> : Vec8<float> {
    __device__ void set(int i, float f) { Vec8<float>::set(i, tf32_round(f)); }
};

template <typename T>
__global__ void __launch_bounds__(kEncodeThreads) encode_nhwc_kernel(EncodeParams p) {
    extern __shared__ uint8_t smem[];
    float* s_scalars = reinterpret_cast<float*>(smem);
    uint8_t* s_bits = smem + ((p.scalar_count * 4 + 15) / 16) * 16;

    const int b = blockIdx.x;
    for (int i = threadIdx.x; i < p.scalar_count; i += kEncodeThreads) s_scalars[i] = p.scalars[size_t(b) * p.scalar_count + i];
    for (int i = threadIdx.x; i < p.bits_stride; i += kEncodeThreads) s_bits[i] = p.bits[size_t(b) * p.bits_stride + i];
    __syncthreads();

    const int area = p.lay.W * p.lay.H;
    const int32_t* sym_row = p.sym ? p.square_src + size_t(p.sym[b]) * area : nullptr;
    const int groups = p.c_pad / 8;
    const int vecs = area * groups;
    const size_t vec_base = size_t(b) * area * groups;
    for (int v = threadIdx.x; v < vecs; v += kEncodeThreads) {
        int sq = v / groups, g = v % groups;
        const int src_sq = sym_row ? sym_row[sq] : sq;
        Vec8<T> out;
#pragma unroll
        for (int j = 0; j < 8; j++) {
            int c = g * 8 + j;
            float f = 0.0f;
            if (c < p.scalar_count) {
                f = s_scalars[c];  // mod.rs:54-56: each scalar broadcast over the plane
            } else if (c < p.scalar_count + p.bool_channels) {
                int i = (c - p.scalar_count) * area + src_sq;  // mod.rs:57-59, bit_buffer.rs:73-75
                f = float((s_bits[i >> 3] >> (i & 7)) & 1);
            }
            out.set(j, f);
        }
        out.store(p.out, vec_base + v);
    }
}

__global__ void encode_nchw_f32_kernel(const uint8_t* __restrict__ bits, const float* __restrict__ scalars, int batch,
                                       int bits_stride, int scalar_count, int bool_channels, int area,
                                       float* __restrict__ out) {
    const int full = (scalar_count + bool_channels) * area;
    size_t total = size_t(batch) * full;
    for (size_t idx = blockIdx.x * size_t(blockDim.x) + threadIdx.x; idx < total; idx += size_t(gridDim.x) * blockDim.x) {
        int b = int(idx / full), e = int(idx % full);
        float f;
        if (e < scalar_count * area) {
            f = scalars[size_t(b) * scalar_count + e / area];
        } else {
            int i = e - scalar_count * area;
            f = float((bits[size_t(b) * bits_stride + (i >> 3)] >> (i & 7)) & 1);
        }
        out[idx] = f;
    }
}

template <typename T>
__global__ void nchw_to_rows_kernel(const float* __restrict__ in, int batch, int channels, RowLayout lay, int c_pad,
                                    void* out) {
    const int area = lay.W * lay.H;
    const int groups = c_pad / 8;
    size_t total = size_t(batch) * area * groups;
    for (size_t v = blockIdx.x * size_t(blockDim.x) + threadIdx.x; v < total; v += size_t(gridDim.x) * blockDim.x) {
        int g = int(v % groups);
        size_t rr = v / groups;
        int b = int(rr / area), sq = int(rr % area);
        Vec8<T> o;
#pragma unroll
        for (int j = 0; j < 8; j++) {
            int c = g * 8 + j;
            float f = 0.0f;
            if (c < channels) f = in[(size_t(b) * channels + c) * area + sq];
            o.set(j, f);
        }
        o.store(out, v);
    }
}

// k-chunk-major input for the second-generation 8x8 tower (tower8k.cu): out[kc][board][square][8 channels] bf16.
// One CTA per board, thread = (kc, square), one 16-byte store each; 64 consecutive threads write 1 KiB contiguous.
template <bool PACKED>
__global__ void encode_kc_kernel(EncodeParams p, const float* __restrict__ nchw, int channels, int kc_total, int boards_total) {
    extern __shared__ uint8_t smem[];
    float* s_scalars = reinterpret_cast<float*>(smem);
    uint8_t* s_bits = smem + ((p.scalar_count * 4 + 15) / 16) * 16;
    const int b = blockIdx.x;
    // the tower kernel is launched with programmatic stream serialization: let it set itself up (it waits before it reads the planes)
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (PACKED) {
        for (int i = threadIdx.x; i < p.scalar_count; i += blockDim.x) s_scalars[i] = p.scalars[size_t(b) * p.scalar_count + i];
        for (int i = threadIdx.x; i < p.bits_stride; i += blockDim.x) s_bits[i] = p.bits[size_t(b) * p.bits_stride + i];
        __syncthreads();
    }
    const int rec_area = p.rec_w * p.rec_h;
    const int32_t* sym_row = (PACKED && p.sym) ? p.square_src + size_t(p.sym[b]) * rec_area : nullptr;
    for (int t = threadIdx.x; t < kc_total * 64; t += blockDim.x) {
        const int kc = t >> 6, sq = t & 63;
        // the record's board sits top-left in the 8x8 grid; squares outside it stay zero
        const int y = sq >> 3, x = sq & 7;
        const bool on_board = x < p.rec_w && y < p.rec_h;
        const int rec_sq = y * p.rec_w + x;
        const int src_sq = (sym_row && on_board) ? sym_row[rec_sq] : rec_sq;
        Vec8<__nv_bfloat16> out;
#pragma unroll
        for (int j = 0; j < 8; j++) {
            const int c = kc * 8 + j;
            float f = 0.0f;
            if (!on_board) {
            } else if (PACKED) {
                if (c < p.scalar_count) {
                    f = s_scalars[c];  // mod.rs:54-56
                } else if (c < p.scalar_count + p.bool_channels) {
                    const int i = (c - p.scalar_count) * rec_area + src_sq;  // mod.rs:57-59, bit_buffer.rs:73-75
                    f = float((s_bits[i >> 3] >> (i & 7)) & 1);
                }
            } else if (c < channels) {
                f = nchw[(size_t(b) * channels + c) * rec_area + rec_sq];
            }
            out.set(j, f);
        }
        out.store(p.out, (size_t(kc) * boards_total + b) * 64 + sq);
    }
}

}  // namespace

void launch_encode_kc(const EncodeParams& p, int kc_total, int boards_total, cudaStream_t s) {
    if (p.batch <= 0) return;
    size_t smem = ((p.scalar_count * 4 + 15) / 16) * 16 + p.bits_stride;
    encode_kc_kernel<true><<<p.batch, std::min(kc_total * 64, 512), smem, s>>>(p, nullptr, 0, kc_total, boards_total);
}

void launch_nchw_to_kc(const float* in, int batch, int channels, int rec_w, int rec_h, int kc_total, int boards_total, void* out,
                       cudaStream_t s) {
    if (batch <= 0) return;
    EncodeParams p{};
    p.batch = batch;
    p.out = out;
    p.rec_w = rec_w;
    p.rec_h = rec_h;
    encode_kc_kernel<false><<<batch, std::min(kc_total * 64, 512), 0, s>>>(p, in, channels, kc_total, boards_total);
}

void launch_encode_nhwc(const EncodeParams& p, Act out, cudaStream_t s) {
    if (p.batch <= 0) return;
    size_t smem = ((p.scalar_count * 4 + 15) / 16) * 16 + p.bits_stride;
    if (out == Act::kBf16)
        encode_nhwc_kernel<__nv_bfloat16><<<p.batch, kEncodeThreads, smem, s>>>(p);
    else if (out == Act::kTf32)
        encode_nhwc_kernel<Tf32><<<p.batch, kEncodeThreads, smem, s>>>(p);
    else
        encode_nhwc_kernel<float><<<p.batch, kEncodeThreads, smem, s>>>(p);
}

void launch_encode_nchw_f32(const uint8_t* bits, const float* scalars, int batch, int bits_stride, int scalar_count,
                            int bool_channels, int area, float* out, cudaStream_t s) {
    if (batch <= 0) return;
    size_t total = size_t(batch) * (scalar_count + bool_channels) * area;
    int blocks = int(std::min<size_t>((total + 255) / 256, 148 * 16));
    encode_nchw_f32_kernel<<<blocks, 256, 0, s>>>(bits, scalars, batch, bits_stride, scalar_count, bool_channels, area, out);
}

void launch_nchw_to_rows(const float* in, int batch, int channels, RowLayout lay, int c_pad, void* out, Act out_type,
                         cudaStream_t s) {
    if (batch <= 0) return;
    size_t total = size_t(batch) * lay.W * lay.H * (c_pad / 8);
    int blocks = int(std::min<size_t>((total + 255) / 256, 148 * 16));
    if (out_type == Act::kBf16)
        nchw_to_rows_kernel<__nv_bfloat16><<<blocks, 256, 0, s>>>(in, batch, channels, lay, c_pad, out);
    else if (out_type == Act::kTf32)
        nchw_to_rows_kernel<Tf32><<<blocks, 256, 0, s>>>(in, batch, channels, lay, c_pad, out);
    else
        nchw_to_rows_kernel<float><<<blocks, 256, 0, s>>>(in, batch, channels, lay, c_pad, out);
}

}  // namespace kzb
