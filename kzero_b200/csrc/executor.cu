#include "executor.hpp"

#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <stdexcept>

namespace kzb {

// ---------------------------------------------------------------------------------------------- utils
namespace {

thread_local std::string g_last_error;

void cuda_check(cudaError_t e, const char* what) {
    if (e != cudaSuccess) throw std::runtime_error(std::string("CUDA error in ") + what + ": " + cudaGetErrorString(e));
}
#define CK(expr) cuda_check((expr), #expr)

int round_up(int v, int m) { return (v + m - 1) / m * m; }
size_t align16(size_t v) { return (v + 15) / 16 * 16; }

// Widest tower / policy conv1 the tensor-core and fp32 paths take
constexpr int kMaxChannels = 1024;

// conv_i2c.cu: the fewest slices an n-channel layer runs in -- each at most 256 output channels (one cta_group::2 MMA, one TMA box,
// two accumulators in 512 TMEM columns) and a whole number of 32-channel epilogue chunks; 0 if there is no such split
int base_split(int n) {
    for (int s = 1; s <= n / 32; s++)
        if (n % s == 0 && n / s <= 256 && (n / s) % 32 == 0) return s;
    return 0;
}

// output width of a conv_i2c layer with c channels: a whole k-block up to 256 channels; above that a multiple of 64 (whole 32-channel
// chunks in both precisions after the small-batch halving) whose base slices hold at least 128 channels.  Most widths only round
// up to 64 (288 -> 320); 704 and 832, whose 64-multiples split only into 64-channel slices, become 768 (3 x 256) and 896 (4 x 224).
int i2c_width(int c, int kb) {
    if (c <= 256) return round_up(c, kb);
    int n = round_up(c, 64);
    while (n / base_split(n) < 128) n += 64;
    return n;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        cuda_check(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q), "cudaGetDriverEntryPoint");
        if (q != cudaDriverEntryPointSuccess || !p) throw std::runtime_error("cuTensorMapEncodeTiled not available in this driver");
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}

// tensor map (bf16 unless `dtype` says otherwise), SWIZZLE_128B, zero OOB fill.  dims/box innermost first; strides in bytes for
// dims 1..rank-1.
CUtensorMap make_tmap(void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes, const uint32_t* box,
                      bool swizzle128 = true, bool swizzle64 = false, CUtensorMapDataType dtype = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16) {
    CUtensorMap m;
    cuuint64_t gdim[5], gstr[4];
    cuuint32_t bdim[5], estr[5];
    for (int i = 0; i < rank; i++) {
        gdim[i] = dims[i];
        bdim[i] = box[i];
        estr[i] = 1;
        if (i > 0) gstr[i - 1] = strides_bytes[i - 1];
    }
    CUresult r = encode_tiled_fn()(&m, dtype, cuuint32_t(rank), base, gdim, gstr, bdim, estr,
                                   CU_TENSOR_MAP_INTERLEAVE_NONE,
                                   swizzle64 ? CU_TENSOR_MAP_SWIZZLE_64B : swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) throw std::runtime_error("cuTensorMapEncodeTiled failed with CUresult " + std::to_string(int(r)));
    return m;
}

typedef CUresult (*EncodeIm2colFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const int*,
                                   const int*, cuuint32_t, cuuint32_t, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// im2col map over channels-last activations [boards][H][W][C] of `dtype` (bf16 or f32) for a (2 * pad + 1)^2 filter with zero
// padding `pad`: a load brings `pixels` consecutive output pixels x `channels` channels, shifted by the instruction's tap offset,
// zero-filled off the board
CUtensorMap make_tmap_im2col(void* base, int C, int W, int H, int boards, int channels, int pixels, int pad, CUtensorMapDataType dtype) {
    static EncodeIm2colFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        cuda_check(cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &p, cudaEnableDefault, &q), "cudaGetDriverEntryPoint");
        if (q != cudaDriverEntryPointSuccess || !p) throw std::runtime_error("cuTensorMapEncodeIm2col not available in this driver");
        return reinterpret_cast<EncodeIm2colFn>(p);
    }();
    CUtensorMap m;
    const size_t esz = dtype == CU_TENSOR_MAP_DATA_TYPE_FLOAT32 ? 4 : 2;
    cuuint64_t gdim[4] = {cuuint64_t(C), cuuint64_t(W), cuuint64_t(H), cuuint64_t(boards)};
    cuuint64_t gstr[3] = {cuuint64_t(C) * esz, cuuint64_t(C) * esz * W, cuuint64_t(C) * esz * W * H};
    int lower[2] = {-pad, -pad}, upper[2] = {-pad, -pad};  // -padding, padding - (filter - 1)
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = fn(&m, dtype, 4, base, gdim, gstr, lower, upper, cuuint32_t(channels), cuuint32_t(pixels), estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) throw std::runtime_error("cuTensorMapEncodeIm2col failed with CUresult " + std::to_string(int(r)));
    // drivers up to CUDA 13.1 mis-encode im2col maps of tensors smaller than 128 KiB (bit 21 of the second descriptor word must be
    // clear); the same correction CUTLASS applies in make_im2col_tma_copy_desc
    int driver = 0;
    if (cudaDriverGetVersion(&driver) == cudaSuccess && driver <= 13010 && size_t(C) * esz * W * H * boards < 131072)
        reinterpret_cast<uint64_t*>(&m)[1] &= ~(1ull << 21);
    return m;
}

}  // namespace

void set_last_error(const std::string& msg) { g_last_error = msg; }
const char* last_error() { return g_last_error.c_str(); }

DeviceBuffer::~DeviceBuffer() {
    if (ptr) cudaFree(ptr);
}
void DeviceBuffer::alloc(size_t n, bool zero) {
    if (ptr) cudaFree(ptr);
    ptr = nullptr;
    bytes = n;
    if (n == 0) return;
    CK(cudaMalloc(&ptr, n));
    if (zero) CK(cudaMemset(ptr, 0, n));
}
PinnedBuffer::~PinnedBuffer() {
    if (ptr) cudaFreeHost(ptr);
}
void PinnedBuffer::alloc(size_t n) {
    if (ptr) cudaFreeHost(ptr);
    ptr = nullptr;
    bytes = n;
    if (n == 0) return;
    // mapped + portable: kernels of any device in this process may write results straight into it
    CK(cudaHostAlloc(&ptr, n, cudaHostAllocMapped | cudaHostAllocPortable));
}

template <typename T>
static void upload(DeviceBuffer& buf, const std::vector<T>& host) {
    buf.alloc(host.size() * sizeof(T), false);
    if (!host.empty()) CK(cudaMemcpy(buf.ptr, host.data(), host.size() * sizeof(T), cudaMemcpyHostToDevice));
}

// ---------------------------------------------------------------------------------------------- Net
Net::Net(int device, const void* onnx, size_t len, int max_batch, int precision)
    : Net(device, build_net_spec(parse_onnx(onnx, len)), max_batch, precision) {}

Net::Net(int device, NetSpec spec, int max_batch, int precision)
    : device_(device), max_batch_(max_batch), precision_(precision) {
    if (max_batch < 1) throw std::runtime_error("max_batch must be >= 1");
    if (precision < 0 || precision > 2) throw std::runtime_error("precision must be 0 (fp32), 1 (bf16) or 2 (tf32)");
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        throw std::runtime_error("no CUDA device available (this library has no CPU fallback): " + std::string(cudaGetErrorString(e)));
    if (device < 0 || device >= count) throw std::runtime_error("device index out of range");
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) throw std::runtime_error("libkzb200 is built for sm_100a (B200) only; found sm_" + std::to_string(prop.major) + std::to_string(prop.minor));
    num_sms_ = prop.multiProcessorCount;

    spec_ = std::move(spec);
    if (spec_.scalar_conv.cout + (spec_.has_extra ? 1 : 0) > 16) throw std::runtime_error("scalar head with more than 15 hidden channels is not supported");
    if (spec_.fc1.out > 128) throw std::runtime_error("scalar head hidden size > 128 is not supported");
    if (spec_.has_extra && spec_.extra_fc.out != 1) throw std::runtime_error("policy head with more than one extra move is not supported");
    if (spec_.channels > kMaxChannels)
        throw std::runtime_error("a tower of " + std::to_string(spec_.channels) + " channels is not supported (at most " +
                                 std::to_string(kMaxChannels) + ")");
    if (spec_.policy_conv1.cout > kMaxChannels)
        throw std::runtime_error("policy conv1 with " + std::to_string(spec_.policy_conv1.cout) + " output channels is not supported (at most " +
                                 std::to_string(kMaxChannels) + ")");
    if (spec_.policy_conv2.cout > 256)
        throw std::runtime_error("policy conv2 with " + std::to_string(spec_.policy_conv2.cout) +
                                 " output channels is not supported (at most 256)");
    if (precision != 0 && (spec_.board_w > 255 || spec_.board_h > 255))  // im2col coordinates
        throw std::runtime_error(std::string("boards wider or taller than 255 squares are not supported in ") + (precision == 1 ? "bf16" : "tf32") +
                                 "; use precision=fp32");

    CK(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
    if (const char* bs = std::getenv("KZB_BLOCKING_SYNC")) blocking_sync_ = bs[0] == '1';
    if (const char* ng = std::getenv("KZB_NO_GRAPH")) use_graph_ = ng[0] != '1';
    if (const char* tr = std::getenv("KZB_TRACE"))
        if (tr[0] == '1') trace_ = new double[5]();
    heads_tail_prepare();
    if (precision_ != 0)
        build_tc();
    else
        build_f32();

    if (embed8_ && !use_tower8k_) throw std::logic_error("internal: small board embedded in 8x8 without the masking tower kernel");

    // tail parameters (shared by both precisions).  When a small board is embedded in the 8x8 grid (embed8_), the flatten
    // order (channel, y, x) of the scalar head's fc1 and the policy provenance table are re-indexed to 8x8 squares; squares
    // outside the board get zero weights / are never referenced.
    const int area = spec_.area(), hs = spec_.fc1.out, hc = spec_.scalar_conv.cout;
    const int bw = spec_.board_w;
    auto sq8 = [&](int sq) { return embed8_ ? (sq / bw) * 8 + sq % bw : sq; };
    const int area_k = embed8_ ? 64 : area;
    std::vector<float> fc1_t(size_t(hc) * area_k * hs, 0.0f);
    for (int j = 0; j < hs; j++)
        for (int c = 0; c < hc; c++)
            for (int sq = 0; sq < area; sq++)
                fc1_t[(size_t(c) * area_k + sq8(sq)) * hs + j] = spec_.fc1.w[size_t(j) * hc * area + size_t(c) * area + sq];
    upload(d_fc1_t_, fc1_t);
    if (embed8_) {
        for (auto& v : spec_.policy_src)
            if (v >= 0) v = (v / area) * 64 + sq8(v % area);
        if (spec_.has_extra) {
            std::vector<float> ew(64, 0.0f);
            for (int sq = 0; sq < area; sq++) ew[size_t(sq8(sq))] = spec_.extra_fc.w[size_t(sq)];
            spec_.extra_fc.w = ew;
        }
    }
    upload(d_fc1_b_, spec_.fc1.b);
    upload(d_fc2_w_, spec_.fc2.w);
    upload(d_fc2_b_, spec_.fc2.b);
    if (spec_.has_extra) upload(d_extra_w_, spec_.extra_fc.w);
    upload(d_policy_src_, spec_.policy_src);
    static_assert(sizeof(NetSpec::AttEntry) == sizeof(AttEntryDev), "AttEntry layout");
    upload(d_att_entries_, spec_.att_entries);

    d_nchw_.alloc(size_t(max_batch_) * spec_.cin * area * 4, false);
    d_out_scalars_.alloc(size_t(max_batch_) * 5 * 4, false);
    d_out_logits_.alloc(size_t(max_batch_) * spec_.policy_len * 4, false);
    CK(cudaStreamSynchronize(stream_));
}

Net::~Net() {
    if (trace_ && trace_[4] > 0)  // KZB_TRACE=1: mean host-side microseconds per kzb_eval_packed phase
        std::fprintf(stderr, "[kzb trace] calls %.0f: stage+H2D enqueue %.1f us, launches+D2H enqueue %.1f us, sync wait %.1f us, copy out %.1f us\n",
                     trace_[4], trace_[0] / trace_[4], trace_[1] / trace_[4], trace_[2] / trace_[4], trace_[3] / trace_[4]);
    delete[] trace_;
    cudaSetDevice(device_);
    if (done_event_) cudaEventDestroy(done_event_);
    for (auto& kv : graphs_)
        if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
    if (stream_) {
        cudaStreamSynchronize(stream_);
        cudaStreamDestroy(stream_);
    }
}

static std::vector<float> padded_bias(const std::vector<float>& b, int n) {
    std::vector<float> out(n, 0.0f);
    std::copy(b.begin(), b.end(), out.begin());
    return out;
}

// the scalar-head conv and the optional extra policy conv read the same input: one launch, cout <= 16
static ConvParams merged_small_conv(const NetSpec& s) {
    ConvParams m = s.scalar_conv;
    if (s.has_extra) {
        m.w.insert(m.w.end(), s.extra_conv.w.begin(), s.extra_conv.w.end());
        m.b.insert(m.b.end(), s.extra_conv.b.begin(), s.extra_conv.b.end());
        m.cout += 1;
    }
    return m;
}

// the attention head's 1x1 convs (post_act.py:120-121) in launches of <= 256 output channels (UMMA N limit), each
// writing its channel range of the concatenated feature matrix E[rows][att_stride]
struct AttChunk {
    std::string name;
    ConvParams conv;
    int out_off;
};
static std::vector<AttChunk> att_chunks(const NetSpec& s) {
    std::vector<AttChunk> out;
    for (size_t k = 0; k < s.att_convs.size(); k++) {
        const ConvParams& c = s.att_convs[k];
        for (int c0 = 0; c0 < c.cout; c0 += 256) {
            AttChunk ch;
            ch.name = "att_conv" + std::to_string(k) + "_" + std::to_string(c0 / 256);
            ch.conv.cin = c.cin;
            ch.conv.ksize = c.ksize;
            ch.conv.cout = std::min(256, c.cout - c0);
            const size_t per = size_t(c.cin) * c.ksize * c.ksize;
            ch.conv.w.assign(c.w.begin() + size_t(c0) * per, c.w.begin() + size_t(c0 + ch.conv.cout) * per);
            ch.conv.b.assign(c.b.begin() + c0, c.b.begin() + c0 + ch.conv.cout);
            ch.out_off = s.att_chan_base[k] + c0;
            out.push_back(std::move(ch));
        }
    }
    return out;
}

// bf16 and TF32.  TF32 runs the row kernels on every board (no tower8k / heads8, no 8x8 embedding); its activations are f32 rows
// holding TF32-exact values, its weights f32 rounded to TF32 on the host, and a k-block is 32 channels instead of 64.
void Net::build_tc() {
    const bool tf32 = precision_ == 2;
    act_ = tf32 ? Act::kTf32 : Act::kBf16;
    const int esz = tf32 ? 4 : 2;   // bytes per activation / weight element
    const int kb = 128 / esz;       // channels per k-block (one 128-byte row of a SWIZZLE_128B tile)
    const CUtensorMapDataType dtype = tf32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    const int C = spec_.channels;
    const char* force = std::getenv("KZB_FORCE_LINEAR");
    // Boards smaller than 8x8 (ataxx 2..7, ttt) are embedded top-left in an 8x8 grid and run on the 8x8 whole-tower kernel:
    // the squares outside the board are forced to zero after every layer (tower8k's epilogue mask), so they act as the
    // convolution's zero padding.  Only when that kernel will really be used -- the per-layer kernels have no such mask.
    {
        auto off = [](const char* name) { const char* v = std::getenv(name); return v && v[0] == '1'; };
        const bool small = spec_.board_w <= 8 && spec_.board_h <= 8 && (spec_.board_w < 8 || spec_.board_h < 8);
        const int units = (((max_batch_ + 3) / 4 + 1) & ~1);
        embed8_ = !tf32 && small && !off("KZB_FORCE_LINEAR") && !off("KZB_NO_TOWER8") && !off("KZB_NO_EMBED8") && round_up(C, 64) <= 128 &&
                  (units + num_sms_ - 1) / num_sms_ <= tower8k_max_local_units();
    }
    const int W = embed8_ ? 8 : spec_.board_w, H = embed8_ ? 8 : spec_.board_h;  // the board as the kernels see it
    mode_ = (!tf32 && W == 8 && H == 8 && !(force && force[0] == '1')) ? 1 : 0;
    // DENSE rows, one per square: conv_i2c.cu gets a 3x3 layer's zero padding from the TMA engine's im2col mode
    lay_ = RowLayout{W, H};
    conv_i2c_prepare();
    if (mode_ == 1) {
        // 8x8: whole 4-board units; the cluster-pair tower kernel pads the batch to an even number of units
        boards_i2c_ = round_up(max_batch_, 8);  // a multiple of 8 boards: whole 256-pixel tiles
        rows_alloc_ = boards_i2c_ * 64;
    } else {  // whole 256-pixel pair tiles, and whole boards under every one of them
        const int pixels = round_up(max_batch_ * W * H, 256);
        boards_i2c_ = (pixels + W * H - 1) / (W * H);
        rows_alloc_ = round_up(std::max(pixels, boards_i2c_ * W * H), 128);
    }
    cin_pad_ = round_up(spec_.cin, kb);
    c_pad_ = i2c_width(C, kb);
    cp_pad_ = i2c_width(spec_.policy_conv1.cout, kb);
    pm_stride_ = round_up(spec_.policy_conv2.cout, 16);
    s1_stride_ = 16;

    act_in_.alloc(size_t(rows_alloc_) * cin_pad_ * esz);
    act_x_.alloc(size_t(rows_alloc_) * c_pad_ * esz);
    act_t_.alloc(size_t(rows_alloc_) * c_pad_ * esz);
    act_h1_.alloc(size_t(rows_alloc_) * cp_pad_ * esz);
    act_s1_.alloc(size_t(rows_alloc_) * s1_stride_ * 4);
    act_pm_.alloc(size_t(rows_alloc_) * pm_stride_ * 4);
    att_stride_ = spec_.has_attention ? spec_.att_chan_base.back() : 0;
    act_att_.alloc(size_t(rows_alloc_) * att_stride_ * 4);

    // `width` output channels stored per row of `out` (stride `out_stride`, from channel out_off on).  Tower form: the output is the
    // next layer's operand (bf16 / TF32), width a multiple of 32, relu_n 0 or width.  Head form (`head`, the 1x1 head convs): f32
    // output, not rounded; the MMA runs width rounded up to 32 channels and the output map clips the rest.
    auto add = [&](const std::string& name, const ConvParams& c, DeviceBuffer& in, int in_stride, const DeviceBuffer* res,
                   DeviceBuffer& out, int out_stride, bool head, int width, int relu_n, int out_off = 0) {
        auto st = std::make_unique<ConvStep>();
        st->name = name;
        st->taps = c.ksize * c.ksize;
        const int n = round_up(width, 32);
        const int cin_pad = in_stride;
        const int ktot = st->taps * cin_pad;
        std::vector<float> wf(size_t(n) * ktot, 0.0f);
        for (int co = 0; co < c.cout; co++)
            for (int ci = 0; ci < c.cin; ci++)
                for (int t = 0; t < st->taps; t++)
                    wf[size_t(co) * ktot + size_t(t) * cin_pad + ci] = c.w[(size_t(co) * c.cin + ci) * st->taps + t];
        if (tf32) {
            for (float& v : wf) v = tf32_round(v);
            upload(st->w_tc, wf);
        } else {
            std::vector<__nv_bfloat16> w(wf.size());
            for (size_t i = 0; i < wf.size(); i++) w[i] = __float2bfloat16_rn(wf[i]);
            upload(st->w_tc, w);
        }
        upload(st->bias, padded_bias(c.b, n));

        // weight map with a box of `rows` output channels x one k-block
        auto wmap = [&](int rows) {
            uint64_t dims[2] = {uint64_t(ktot), uint64_t(n)};
            uint64_t strides[1] = {uint64_t(ktot) * esz};
            uint32_t box[2] = {uint32_t(kb), uint32_t(rows)};
            return make_tmap(st->w_tc.ptr, 2, dims, strides, box, true, false, dtype);
        };
        st->tmap_i2c = make_tmap_im2col(in.ptr, in_stride, W, H, boards_i2c_, kb, 128, st->taps == 9 ? 1 : 0, dtype);
        // staging boxes of 32 rows x 32 channels: 64-byte (bf16) or 128-byte (f32) rows; `cols` channels of rows `stride` apart
        auto rows_map = [&](void* ptr, int cols, int stride, bool f32) {
            uint64_t dims[2] = {uint64_t(cols), uint64_t(rows_alloc_)};
            uint64_t strides[1] = {uint64_t(stride) * (f32 ? 4 : 2)};
            uint32_t box[2] = {32, 32};
            return make_tmap(ptr, 2, dims, strides, box, f32, !f32, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16);
        };
        const bool f32_out = tf32 || head;
        st->tmap_out = rows_map(static_cast<uint8_t*>(out.ptr) + size_t(out_off) * (f32_out ? 4 : 2), width, out_stride, f32_out);
        st->tmap_res = res ? rows_map(res->ptr, c_pad_, c_pad_, tf32) : st->tmap_out;
        // output channels in split0 slices (twice as many for small batches, run_network); each CTA of a pair stages half of
        // every weight tile of its slice
        st->split0 = base_split(n);
        if (st->split0 == 0) throw std::logic_error("internal: conv_i2c layer of " + std::to_string(n) + " channels has no slicing");
        const int slice = n / st->split0;
        st->split_double = slice % 64 == 0;  // the halved slice is still whole 32-channel chunks
        st->tmap_w[0] = wmap(slice / 2);
        st->tmap_w[1] = st->split_double ? wmap(slice / 4) : st->tmap_w[0];
        ConvTcParams& p = st->tc;
        p.taps = st->taps;
        p.cin_pad = cin_pad;
        p.kblocks = cin_pad / kb;
        p.tf32 = tf32 ? 1 : 0;
        p.head = head ? 1 : 0;
        p.n = n;
        p.lay = lay_;
        p.bias = st->bias.as<float>();
        p.relu_n = relu_n;
        p.has_res = res ? 1 : 0;
        p.stages = conv_i2c_pick_stages(f32_out ? 4 : 2);
        int cols = 32;  // two accumulators of the widest slice
        while (cols < 2 * slice) cols *= 2;
        p.tmem_cols = cols;
        p.n_split = 1;
        const char* pdl_env = std::getenv("KZB_PDL");  // programmatic dependent launch of consecutive conv_i2c layers (KZB_PDL=0: off)
        p.pdl = (pdl_env && pdl_env[0] == '0') ? 0 : 1;
        convs_.push_back(std::move(st));
    };

    add("conv_first", spec_.first, act_in_, cin_pad_, nullptr, act_x_, c_pad_, false, c_pad_, 0);
    for (int d = 0; d < spec_.depth; d++) {
        add("block" + std::to_string(d) + "_conv1", spec_.blocks[2 * d], act_x_, c_pad_, nullptr, act_t_, c_pad_, false, c_pad_, c_pad_);
        add("block" + std::to_string(d) + "_conv2", spec_.blocks[2 * d + 1], act_t_, c_pad_, &act_x_, act_x_, c_pad_, false, c_pad_, c_pad_);
    }
    head_first_ = convs_.size();
    if (spec_.has_attention) {
        add("scalar_conv", merged_small_conv(spec_), act_x_, c_pad_, nullptr, act_s1_, s1_stride_, true, s1_stride_, spec_.scalar_conv.cout);
        for (const AttChunk& ch : att_chunks(spec_))
            add(ch.name, ch.conv, act_x_, c_pad_, nullptr, act_att_, att_stride_, true, round_up(ch.conv.cout, 16), 0, ch.out_off);
    } else {
        add("policy_conv1", spec_.policy_conv1, act_x_, c_pad_, nullptr, act_h1_, cp_pad_, false, cp_pad_, cp_pad_);
        add("scalar_conv", merged_small_conv(spec_), act_x_, c_pad_, nullptr, act_s1_, s1_stride_, true, s1_stride_, spec_.scalar_conv.cout);
        add("policy_conv2", spec_.policy_conv2, act_h1_, cp_pad_, nullptr, act_pm_, pm_stride_, true, pm_stride_, 0);
    }

    // fused heads kernel: policy conv1 -> relu -> conv2, scalar conv -> relu -> fc -> relu -> fc, masked softmax (heads8.cu)
    const char* no_h8 = std::getenv("KZB_NO_HEADS8");
    if (mode_ == 1 && !spec_.has_attention && !spec_.has_extra && !(no_h8 && no_h8[0] == '1')) {
        Heads8Params hp{};
        hp.kblocks = c_pad_ / 64;
        hp.n1 = cp_pad_;
        hp.n2 = pm_stride_;
        hp.pc = spec_.policy_conv2.cout;
        hp.hc = spec_.scalar_conv.cout;
        hp.hs = spec_.fc1.out;
        bool src_ok = true;
        for (int32_t v : spec_.policy_src) src_ok = src_ok && v >= kPolicySrcZero;
        if (src_ok && heads8_supported(hp)) {
            heads8_prepare();
            ConvStep& c1 = *convs_[head_first_];
            ConvStep& cs = *convs_[head_first_ + 1];
            ConvStep& c2 = *convs_[head_first_ + 2];
            hp.b1 = c1.bias.as<float>();
            hp.bs = cs.bias.as<float>();
            hp.b2 = c2.bias.as<float>();
            // the first `rows` output channels of a 1x1 step's bf16 weights [n][cin_pad], all of them in one box
            auto wmap = [&](const ConvStep& st, int rows) {
                uint64_t dims[2] = {uint64_t(st.tc.cin_pad), uint64_t(rows)};
                uint64_t strides[1] = {uint64_t(st.tc.cin_pad) * 2};
                uint32_t box[2] = {64, uint32_t(rows)};
                return make_tmap(st.w_tc.ptr, 2, dims, strides, box);
            };
            heads_maps_.w1 = wmap(c1, hp.n1);
            heads_maps_.ws = wmap(cs, 16);
            heads_maps_.w2 = wmap(c2, hp.n2);
            uint64_t dims[2] = {uint64_t(c_pad_), uint64_t(rows_alloc_)};
            uint64_t strides[1] = {uint64_t(c_pad_) * 2};
            uint32_t box[2] = {64, 128};
            heads_maps_.x = make_tmap(act_x_.ptr, 2, dims, strides, box);
            heads_params_ = hp;
            use_heads8_ = true;
        }
    }

    // whole-tower persistent kernel: all 2*depth+1 conv3x3 layers in one launch (tower8k.cu)
    const char* no_t8 = std::getenv("KZB_NO_TOWER8");
    const int units_max = ((max_batch_ + 3) / 4 + 1) & ~1;
    if (mode_ == 1 && c_pad_ <= 128 && !(no_t8 && no_t8[0] == '1') &&
        (units_max + num_sms_ - 1) / num_sms_ <= tower8k_max_local_units()) {
        tower8k_prepare();
        tower_layers_ = 1 + 2 * spec_.depth;
        const int n = c_pad_;
        act_xt_.alloc(size_t(std::max(rows_alloc_ / 256 + 1, 2 * num_sms_ + 2)) * 128 * 256 * 2);  // one slot per (CTA, local unit)
        const int cluster = 2;  // CTA pairs: each loads half of every weight tile and multicasts it
        {
            ConvStep& f = *convs_[0];
            uint64_t dims[2] = {uint64_t(9 * cin_pad_), uint64_t(n)};
            uint64_t strides[1] = {uint64_t(9 * cin_pad_) * 2};
            uint32_t box[2] = {64, uint32_t(n / cluster)};
            tower_kmaps_.w[0] = make_tmap(f.w_tc.ptr, 2, dims, strides, box);
        }
        const size_t layer_w_bytes = size_t(n) * 9 * c_pad_ * 2;
        w_tower_.alloc(std::max<size_t>(layer_w_bytes * 2 * spec_.depth, 256), true);
        for (int i = 0; i < 2 * spec_.depth; i++)
            CK(cudaMemcpy(w_tower_.as<uint8_t>() + layer_w_bytes * i, convs_[1 + i]->w_tc.ptr, layer_w_bytes, cudaMemcpyDeviceToDevice));
        {
            uint64_t dims[2] = {uint64_t(9 * c_pad_), uint64_t(std::max(1, 2 * spec_.depth) * n)};
            uint64_t strides[1] = {uint64_t(9 * c_pad_) * 2};
            uint32_t box[2] = {64, uint32_t(n / cluster)};
            tower_kmaps_.w[1] = make_tmap(w_tower_.ptr, 2, dims, strides, box);
        }
        std::vector<TowerLayerDev> layers(tower_layers_);
        for (int i = 0; i < tower_layers_; i++) {
            TowerLayerDev& l = layers[i];
            const bool first = i == 0, conv2 = !first && (i % 2 == 0);
            l.a_map = first ? 0 : (conv2 ? 2 : 1);
            l.w_map = first ? 0 : 1;
            l.w_row0 = first ? 0 : (i - 1) * n;
            l.cin_pad = first ? cin_pad_ : c_pad_;
            l.kblocks = l.cin_pad / 64;
            l.relu_n = first ? 0 : n;
            l.has_res = conv2 ? 1 : 0;
            l.out_buf = (first || conv2) ? 1 : 2;
            l.bias = convs_[i]->bias.as<float>();
            // a narrow single-k-block first layer only stages / multiplies the chunks that exist
            l.ksteps = (first && l.kblocks == 1) ? std::max(1, (spec_.cin + 15) / 16) : 4;
            l.kchunks = 2 * l.ksteps;
            l.out_rowmajor = (i == tower_layers_ - 1) ? 1 : 0;
        }
        upload(d_tower_layers_, layers);
        Tower8Params& tp = tower_params_;
        tp.num_layers = tower_layers_;
        tp.layers = d_tower_layers_.as<TowerLayerDev>();
        tp.n = n;
        tp.n_store = n;
        tp.x = act_x_.as<__nv_bfloat16>();
        tp.t = act_t_.as<__nv_bfloat16>();
        tp.xt = act_xt_.as<__nv_bfloat16>();
        tp.stride = c_pad_;
        tp.cluster = cluster;
        tp.board_w = spec_.board_w;
        tp.board_h = spec_.board_h;
        int cols = 32;
        while (cols < 4 * n) cols *= 2;
        tp.tmem_cols = cols;
        // k-chunk-major activations, one staged copy per k-block
        const uint64_t boards_total = uint64_t(rows_alloc_ / 64);
        act_ink_.alloc(size_t(cin_pad_ / 8) * boards_total * 1024);
        act_xk_.alloc(size_t(c_pad_ / 8) * boards_total * 1024);
        act_tk_.alloc(size_t(c_pad_ / 8) * boards_total * 1024);
        auto kload = [&](DeviceBuffer& buf, int kc_total, int nb) {  // (x*8+c8, board, y, kc)
            uint64_t dims[4] = {64, boards_total, 8, uint64_t(kc_total)};
            uint64_t strides[3] = {1024, 128, boards_total * 1024};
            // 72 > 64: the engine zero-fills the pad row of every 8-position group; 9 > 8: and a zero rank behind the board
            uint32_t box[4] = {72, uint32_t(nb), 9, 1};
            return make_tmap(buf.ptr, 4, dims, strides, box, false);
        };
        auto kstore = [&](DeviceBuffer& buf, int kc_total, int nb) {  // (x*8+c8, kc, board, y)
            uint64_t dims[4] = {64, uint64_t(kc_total), boards_total, 8};
            uint64_t strides[3] = {boards_total * 1024, 1024, 128};
            uint32_t box[4] = {80, 4, uint32_t(nb), 1};  // staging rows are 160 bytes (bank spreading); elements 64..79 are clipped
            return make_tmap(buf.ptr, 4, dims, strides, box, false);
        };
        auto rstore = [&](DeviceBuffer& buf, int nb) {  // row-major rows, one rank of an nb-board unit: (c, x, board, y)
            uint64_t dims[4] = {uint64_t(c_pad_), 8, uint64_t(rows_alloc_ / 64), 8};
            uint64_t strides[3] = {uint64_t(c_pad_) * 2, uint64_t(c_pad_) * 2 * 64, uint64_t(c_pad_) * 2 * 8};
            uint32_t box[4] = {32, 8, uint32_t(nb), 1};
            return make_tmap(buf.ptr, 4, dims, strides, box, false);
        };
        for (int nb = 3; nb <= 4; nb++) {
            tower_kmaps_.a[0][nb - 3] = kload(act_ink_, cin_pad_ / 8, nb);
            tower_kmaps_.a[1][nb - 3] = kload(act_xk_, c_pad_ / 8, nb);
            tower_kmaps_.a[2][nb - 3] = kload(act_tk_, c_pad_ / 8, nb);
            tower_kmaps_.out[0][nb - 3] = kstore(act_xk_, c_pad_ / 8, nb);
            tower_kmaps_.out[1][nb - 3] = kstore(act_tk_, c_pad_ / 8, nb);
            tower_kmaps_.out[2][nb - 3] = rstore(act_x_, nb);
        }
        tp.b_slots = tower8k_pick_b_slots();
        const char* bs = std::getenv("KZB_B_SLOTS");
        if (bs && std::atoi(bs) >= 2 && std::atoi(bs) <= tp.b_slots) tp.b_slots = std::atoi(bs);
        tp.timeline = nullptr;
        {
            const char* pdl_env = std::getenv("KZB_PDL");  // KZB_PDL=0: plain stream order between encode, tower and heads
            tp.pdl = (pdl_env && pdl_env[0] == '0') ? 0 : 1;
        }
        const char* dbg = std::getenv("KZB_DEBUG");
        tp.debug = dbg ? std::atoi(dbg) : 0;
        use_tower8k_ = true;
    }
}

void Net::build_f32() {
    act_ = Act::kF32;
    const int W = spec_.board_w, H = spec_.board_h, C = spec_.channels;
    mode_ = -1;
    lay_ = RowLayout{W, H};
    rows_alloc_ = max_batch_ * W * H;
    cin_pad_ = round_up(spec_.cin, 8);
    c_pad_ = round_up(C, 8);
    cp_pad_ = round_up(spec_.policy_conv1.cout, 8);
    pm_stride_ = round_up(spec_.policy_conv2.cout, 4);
    s1_stride_ = 16;

    act_in_.alloc(size_t(rows_alloc_) * cin_pad_ * 4);
    act_x_.alloc(size_t(rows_alloc_) * c_pad_ * 4);
    act_t_.alloc(size_t(rows_alloc_) * c_pad_ * 4);
    act_h1_.alloc(size_t(rows_alloc_) * cp_pad_ * 4);
    act_s1_.alloc(size_t(rows_alloc_) * s1_stride_ * 4);
    act_pm_.alloc(size_t(rows_alloc_) * pm_stride_ * 4);

    att_stride_ = spec_.has_attention ? spec_.att_chan_base.back() : 0;
    act_att_.alloc(size_t(rows_alloc_) * att_stride_ * 4);

    auto add = [&](const std::string& name, const ConvParams& c, DeviceBuffer& in, int in_stride, const DeviceBuffer* res,
                   DeviceBuffer& out, int out_stride, int relu_n, int out_off = 0) {
        auto st = std::make_unique<ConvStep>();
        st->name = name;
        st->taps = c.ksize * c.ksize;
        std::vector<float> w(size_t(st->taps) * c.cin * c.cout);
        for (int co = 0; co < c.cout; co++)
            for (int ci = 0; ci < c.cin; ci++)
                for (int t = 0; t < st->taps; t++)
                    w[(size_t(t) * c.cin + ci) * c.cout + co] = c.w[(size_t(co) * c.cin + ci) * st->taps + t];
        upload(st->w_f32, w);
        upload(st->bias, c.b);
        ConvF32Params& p = st->f32;
        p.in = in.as<float>();
        p.in_stride = in_stride;
        p.w = st->w_f32.as<float>();
        p.bias = st->bias.as<float>();
        p.res = res ? res->as<float>() : nullptr;
        p.res_stride = c_pad_;
        p.out = out.as<float>() + out_off;
        p.out_stride = out_stride;
        p.cin = c.cin;
        p.cout = c.cout;
        p.taps = st->taps;
        p.relu_n = relu_n;
        p.lay = lay_;
        convs_.push_back(std::move(st));
    };
    add("conv_first", spec_.first, act_in_, cin_pad_, nullptr, act_x_, c_pad_, 0);
    for (int d = 0; d < spec_.depth; d++) {
        add("block" + std::to_string(d) + "_conv1", spec_.blocks[2 * d], act_x_, c_pad_, nullptr, act_t_, c_pad_, C);
        add("block" + std::to_string(d) + "_conv2", spec_.blocks[2 * d + 1], act_t_, c_pad_, &act_x_, act_x_, c_pad_, C);
    }
    if (spec_.has_attention) {
        add("scalar_conv", merged_small_conv(spec_), act_x_, c_pad_, nullptr, act_s1_, s1_stride_, spec_.scalar_conv.cout);
        for (const AttChunk& ch : att_chunks(spec_)) add(ch.name, ch.conv, act_x_, c_pad_, nullptr, act_att_, att_stride_, 0, ch.out_off);
    } else {
        add("policy_conv1", spec_.policy_conv1, act_x_, c_pad_, nullptr, act_h1_, cp_pad_, spec_.policy_conv1.cout);
        add("scalar_conv", merged_small_conv(spec_), act_x_, c_pad_, nullptr, act_s1_, s1_stride_, spec_.scalar_conv.cout);
        add("policy_conv2", spec_.policy_conv2, act_h1_, cp_pad_, nullptr, act_pm_, pm_stride_, 0);
    }
}

// offsets inside the contiguous input block [mv_off | scalars | bits | mv_idx] -> a single H2D copy per batch
struct InBlock {
    size_t off_scalars, off_bits, off_idx;
};
static InBlock in_block(int max_batch, int scalar_count, int bits_stride) {
    InBlock b;
    b.off_scalars = align16(size_t(max_batch + 1) * 4);
    b.off_bits = b.off_scalars + align16(size_t(max_batch) * scalar_count * 4);
    b.off_idx = b.off_bits + align16(size_t(max_batch) * bits_stride);
    return b;
}
// offsets inside the contiguous output block [err word (16 B) | values | probs] -> a single D2H copy per batch
struct OutBlock {
    size_t off_values, off_probs;
};
static OutBlock out_block(int max_batch) { return {16, 16 + align16(size_t(max_batch) * 5 * 4)}; }

void Net::bind_mapper(int scalar_count, int bool_channels, int h, int w, int policy_len) {
    // twin of check_graph_shapes, rust/kz-core/src/network/common.rs:165-198
    if (scalar_count < 0 || bool_channels < 0) throw std::runtime_error("negative channel count");
    if (scalar_count + bool_channels != spec_.cin || h != spec_.board_h || w != spec_.board_w)
        throw std::runtime_error("Input shape mismatch between graph and mapper: graph [BATCH, " + std::to_string(spec_.cin) + ", " +
                                 std::to_string(spec_.board_h) + ", " + std::to_string(spec_.board_w) + "] vs mapper [BATCH, " +
                                 std::to_string(scalar_count + bool_channels) + ", " + std::to_string(h) + ", " + std::to_string(w) + "]");
    if (policy_len != spec_.policy_len)
        throw std::runtime_error("Wrong policy shape: graph has " + std::to_string(spec_.policy_len) + " entries, mapper " + std::to_string(policy_len));
    CK(cudaSetDevice(device_));
    scalar_count_ = scalar_count;
    bool_channels_ = bool_channels;
    bits_stride_ = (bool_channels * h * w + 7) / 8;
    mv_cap_ = size_t(max_batch_) * spec_.policy_len;
    const size_t in_bytes = in_block(max_batch_, scalar_count_, bits_stride_).off_idx + mv_cap_ * 4;
    d_mv_off_.alloc(in_bytes, true);
    h_in_.alloc(in_bytes);
    const size_t out_bytes = out_block(max_batch_).off_probs + mv_cap_ * 4;
    d_err_.alloc(out_bytes, true);
    h_out_.alloc(out_bytes);
}

void Net::check_batch(int batch) const {
    // cudnn.rs:58 assert!(batch_size <= max_batch_size)
    if (batch < 0 || batch > max_batch_)
        throw std::runtime_error("batch size " + std::to_string(batch) + " exceeds max_batch_size " + std::to_string(max_batch_));
}
void Net::require_mapper() const {
    if (scalar_count_ < 0) throw std::runtime_error("kzb_net_bind_mapper must be called before packed evaluation");
}

void Net::upload_packed(const uint8_t* bits, const float* scalars, int batch, const uint32_t* mv_idx, const uint32_t* mv_off) {
    InBlock ib = in_block(max_batch_, scalar_count_, bits_stride_);
    uint8_t* h = h_in_.as<uint8_t>();
    size_t moves = 0;
    if (mv_off) {
        if (mv_off[0] != 0) throw std::runtime_error("mv_off[0] must be 0");
        for (int i = 0; i < batch; i++)
            if (mv_off[i + 1] < mv_off[i]) throw std::runtime_error("mv_off must be non-decreasing");
        moves = mv_off[batch];
        if (moves > mv_cap_) throw std::runtime_error("more legal moves than batch * policy_len");
        std::memcpy(h, mv_off, size_t(batch + 1) * 4);
        if (moves) std::memcpy(h + ib.off_idx, mv_idx, moves * 4);
    } else {
        std::memset(h, 0, size_t(batch + 1) * 4);
    }
    std::memcpy(h + ib.off_scalars, scalars, size_t(batch) * scalar_count_ * 4);
    std::memcpy(h + ib.off_bits, bits, size_t(batch) * bits_stride_);
    // the gaps between the segments are small; copy the used prefix in one go
    size_t used = ib.off_idx + moves * 4;
    CK(cudaMemcpyAsync(d_mv_off_.ptr, h, used, cudaMemcpyHostToDevice, stream_));
    staged_batch_ = batch;
    staged_moves_ = moves;
}

void Net::run_encode(int batch, const StepHook& hook) {
    InBlock ib = in_block(max_batch_, scalar_count_, bits_stride_);
    EncodeParams p{};
    p.rec_w = spec_.board_w;
    p.rec_h = spec_.board_h;
    p.sym = cur_sym_;
    p.square_src = d_sym_square_.as<int32_t>();
    p.bits = d_mv_off_.as<uint8_t>() + ib.off_bits;
    p.scalars = reinterpret_cast<const float*>(d_mv_off_.as<uint8_t>() + ib.off_scalars);
    p.batch = batch;
    p.bits_stride = bits_stride_;
    p.scalar_count = scalar_count_;
    p.bool_channels = bool_channels_;
    p.lay = lay_;
    p.c_pad = cin_pad_;
    p.out = act_in_.ptr;
    if (use_tower8k_) {
        p.out = act_ink_.ptr;
        launch_encode_kc(p, cin_pad_ / 8, rows_alloc_ / 64, stream_);
    } else {
        launch_encode_nhwc(p, act_, stream_);
    }
    if (hook) hook("encode");
}

void Net::run_network(int batch, const StepHook& hook) {
    size_t first_step = 0;
    if (use_tower8k_) {
        Tower8Params tp = tower_params_;
        tp.num_units = (((batch + 3) / 4) + 1) & ~1;  // cluster pairs: rows of the padding unit exist (boards_alloc) and are never read back
        tp.valid_rows = batch * 64;
        if (timeline_step_ == "tower8") tp.timeline = d_timeline_.as<unsigned long long>();
        // balanced assignment: every CTA owns 6..8 contiguous boards (two units of 4 / 3); otherwise 4-board units
        const int grid = num_sms_ & ~1;
        const char* nobal = std::getenv("KZB_NO_BALANCE");
        tp.balanced = 0;
        if (!(nobal && nobal[0] == '1') && batch / grid >= 6 && (batch + grid - 1) / grid <= 8) {
            tp.balanced = 1;
            tp.bal_grid = grid;
            tp.bal_base = batch / grid;
            tp.bal_rem = batch % grid;
        }
        launch_tower8k(tower_kmaps_, tp, num_sms_, stream_);
        if (hook) hook("tower8");
        first_step = size_t(tower_layers_);
    }
    const size_t last_step = (use_heads8_ && precision_ == 1) ? head_first_ : convs_.size();
    for (size_t si = first_step; si < last_step; si++) {
        auto& st = convs_[si];
        if (precision_ != 0) {
            ConvTcParams p = st->tc;
            p.num_tiles = (batch * lay_.W * lay_.H + 127) / 128;
            // the output channels in split0 slices of <= 256; small batches: twice the slices, so that twice as many SM pairs share
            // the layer, when the work items fill at most half of them (KZB_CONV_SPLIT=0: never)
            const char* split = std::getenv("KZB_CONV_SPLIT");
            const bool dbl = !(split && split[0] == '0') && st->split_double && 2 * ((p.num_tiles + 1) / 2) * st->split0 <= num_sms_ / 2;
            p.n_split = st->split0 * (dbl ? 2 : 1);
            launch_conv_i2c(st->tmap_i2c, st->tmap_w[dbl ? 1 : 0], st->tmap_out, st->tmap_res, p, num_sms_, stream_);
        } else {
            ConvF32Params p = st->f32;
            p.batch = batch;
            launch_conv_fp32(p, stream_);
        }
        if (hook) hook(st->name.c_str());
    }
}

HeadOutputs Net::head_outputs(int batch, bool packed, bool to_host) const {
    HeadOutputs o{};
    o.batch = batch;
    o.policy_len = spec_.policy_len;
    o.packed = packed ? 1 : 0;
    o.out_scalars = d_out_scalars_.as<float>();
    o.out_logits = d_out_logits_.as<float>();
    if (packed) {
        const InBlock ib = in_block(max_batch_, scalar_count_, bits_stride_);
        const OutBlock ob = out_block(max_batch_);
        o.mv_off = d_mv_off_.as<uint32_t>();
        o.mv_idx = reinterpret_cast<const uint32_t*>(d_mv_off_.as<uint8_t>() + ib.off_idx);
        o.sym = cur_sym_;
        o.policy_map = d_sym_policy_.as<int32_t>();
        // results either stay in HBM (staged timing) or are written straight into the pinned, device-mapped host block
        // (kzb_eval_packed: no separate D2H copies, the posted PCIe writes overlap the kernel)
        uint8_t* out = to_host ? h_out_.as<uint8_t>() : d_err_.as<uint8_t>();
        o.err_flag = reinterpret_cast<int*>(out);
        o.out_values = reinterpret_cast<float*>(out + ob.off_values);
        o.out_probs = reinterpret_cast<float*>(out + ob.off_probs);
    }
    return o;
}

void Net::run_tail(int batch, bool packed, const StepHook& hook, bool to_host) {
    const HeadOutputs out = head_outputs(batch, packed, to_host);
    if (use_heads8_ && precision_ == 1) {
        Heads8Params p = heads_params_;
        p.out = out;
        p.num_tiles = (batch + 1) / 2;
        p.fc1_t = d_fc1_t_.as<float>();
        p.fc1_b = d_fc1_b_.as<float>();
        p.fc2_w = d_fc2_w_.as<float>();
        p.fc2_b = d_fc2_b_.as<float>();
        p.policy_src = d_policy_src_.as<int32_t>();
        p.timeline = timeline_step_ == "heads8" ? d_timeline_.as<unsigned long long>() : nullptr;
        p.pdl = (use_tower8k_ && tower_params_.pdl) ? 1 : 0;  // only behind the tower kernel, which triggers the dependent launch
        launch_heads8(heads_maps_, p, num_sms_, stream_);
        if (hook) hook("heads8");
        return;
    }
    HeadsTailParams p{};
    p.out = out;
    p.lay = lay_;
    p.s1 = act_s1_.as<float>();
    p.s1_stride = s1_stride_;
    p.hc = spec_.scalar_conv.cout;
    p.pm = act_pm_.as<float>();
    p.pm_stride = pm_stride_;
    p.fc1_t = d_fc1_t_.as<float>();
    p.fc1_b = d_fc1_b_.as<float>();
    p.fc2_w = d_fc2_w_.as<float>();
    p.fc2_b = d_fc2_b_.as<float>();
    p.hs = spec_.fc1.out;
    p.extra_w = spec_.has_extra ? d_extra_w_.as<float>() : nullptr;
    p.extra_b = spec_.has_extra ? spec_.extra_fc.b[0] : 0.0f;
    p.policy_src = spec_.has_attention ? nullptr : d_policy_src_.as<int32_t>();
    p.att = act_att_.as<float>();
    p.att_stride = att_stride_;
    p.att_q = spec_.att_q;
    p.att_div = spec_.att_div;
    p.att_entries = spec_.has_attention ? d_att_entries_.as<AttEntryDev>() : nullptr;
    launch_heads_tail(p, stream_);
    if (hook) hook("heads_tail");
}

void Net::eval_planes(const float* nchw, int batch, float* out_scalars, float* out_logits) {
    check_batch(batch);
    if (batch == 0) return;
    CK(cudaSetDevice(device_));
    const int area = spec_.area();
    CK(cudaMemcpyAsync(d_nchw_.ptr, nchw, size_t(batch) * spec_.cin * area * 4, cudaMemcpyHostToDevice, stream_));
    if (use_tower8k_)
        launch_nchw_to_kc(d_nchw_.as<float>(), batch, spec_.cin, spec_.board_w, spec_.board_h, cin_pad_ / 8, rows_alloc_ / 64, act_ink_.ptr,
                          stream_);
    else
        launch_nchw_to_rows(d_nchw_.as<float>(), batch, spec_.cin, lay_, cin_pad_, act_in_.ptr, act_, stream_);
    run_network(batch, nullptr);
    run_tail(batch, false, nullptr);
    CK(cudaMemcpyAsync(out_scalars, d_out_scalars_.ptr, size_t(batch) * 5 * 4, cudaMemcpyDeviceToHost, stream_));
    CK(cudaMemcpyAsync(out_logits, d_out_logits_.ptr, size_t(batch) * spec_.policy_len * 4, cudaMemcpyDeviceToHost, stream_));
    CK(cudaStreamSynchronize(stream_));
    CK(cudaGetLastError());
}

void Net::set_symmetries(int n_sym, const int32_t* square_src, const int32_t* policy_map) {
    require_mapper();
    if (n_sym < 1 || n_sym > 255) throw std::runtime_error("symmetry count must be in 1..255");
    const int area = spec_.area(), plen = spec_.policy_len;
    for (int i = 0; i < n_sym * area; i++)
        if (square_src[i] < 0 || square_src[i] >= area) throw std::runtime_error("symmetry square table entry out of range");
    for (int i = 0; i < n_sym * plen; i++)
        if (policy_map[i] < -1 || policy_map[i] >= plen)  // -1: this index is not a move (the reference's tables use it, too)
            throw std::runtime_error("symmetry policy table entry out of range");
    CK(cudaSetDevice(device_));
    upload(d_sym_square_, std::vector<int32_t>(square_src, square_src + size_t(n_sym) * area));
    upload(d_sym_policy_, std::vector<int32_t>(policy_map, policy_map + size_t(n_sym) * plen));
    d_sym_.alloc(size_t(max_batch_), true);
    h_sym_.alloc(size_t(max_batch_));
    n_sym_ = n_sym;
}

void Net::eval_packed(const uint8_t* bits, const float* scalars, int batch, const uint32_t* mv_idx, const uint32_t* mv_off,
                      float* out_values, float* out_policy, const uint8_t* sym) {
    check_batch(batch);
    require_mapper();
    if (batch == 0) return;
    cur_sym_ = nullptr;
    if (sym) {
        if (n_sym_ == 0) throw std::runtime_error("kzb_net_set_symmetries must be called before an evaluation with symmetries");
        for (int i = 0; i < batch; i++)
            if (sym[i] >= n_sym_) throw std::runtime_error("symmetry index out of range");
        CK(cudaSetDevice(device_));
        std::memcpy(h_sym_.ptr, sym, size_t(batch));
        CK(cudaMemcpyAsync(d_sym_.ptr, h_sym_.ptr, size_t(batch), cudaMemcpyHostToDevice, stream_));
        cur_sym_ = d_sym_.as<uint8_t>();
    }
    struct ClearSym {  // the staged / planes paths never apply a symmetry
        const uint8_t*& ref;
        ~ClearSym() { ref = nullptr; }
    } clear_sym{cur_sym_};
    using clk = std::chrono::steady_clock;
    const bool trace = trace_ != nullptr;
    clk::time_point t0, t1, t2, t3, t4;
    if (trace) t0 = clk::now();
    CK(cudaSetDevice(device_));
    upload_packed(bits, scalars, batch, mv_idx, mv_off);
    if (trace) t1 = clk::now();
    *h_out_.as<volatile int>() = 0;  // error word; the tail kernel only ever writes non-zero into it
    // The kernel sequence of a batch size that keeps coming back (the full batch above all: self-play batches are full 99 % of the
    // time) is captured once into a CUDA graph and replayed: one launch call instead of one per kernel (46 for a 20-block go net).
    // Evaluations with symmetries and one-off sizes take the direct path.
    BatchGraph* bg = nullptr;
    if (use_graph_ && cur_sym_ == nullptr) {
        auto it = graphs_.find(batch);
        if (it != graphs_.end()) bg = &it->second;
        else if (graphs_.size() < kMaxGraphs) bg = &graphs_[batch];
    }
    if (bg && bg->exec) {
        CK(cudaGraphLaunch(bg->exec, stream_));
    } else if (bg && (++bg->seen >= 2 || batch == max_batch_)) {
        cudaGraph_t graph = nullptr;
        CK(cudaStreamBeginCapture(stream_, cudaStreamCaptureModeThreadLocal));
        run_encode(batch, nullptr);
        run_network(batch, nullptr);
        run_tail(batch, true, nullptr, /*to_host=*/true);
        CK(cudaStreamEndCapture(stream_, &graph));
        cudaError_t ge = cudaGraphInstantiate(&bg->exec, graph, 0);
        cudaGraphDestroy(graph);
        if (ge != cudaSuccess) {  // fall back to direct launches for good
            cudaGetLastError();
            bg->exec = nullptr;
            use_graph_ = false;
            run_encode(batch, nullptr);
            run_network(batch, nullptr);
            run_tail(batch, true, nullptr, /*to_host=*/true);
        } else {
            CK(cudaGraphLaunch(bg->exec, stream_));
        }
    } else {
        run_encode(batch, nullptr);
        run_network(batch, nullptr);
        run_tail(batch, true, nullptr, /*to_host=*/true);
    }
    if (trace) t2 = clk::now();
    if (blocking_sync_) {  // the calling thread sleeps while the GPU works (self-play: executor threads share cores with generators)
        if (!done_event_) CK(cudaEventCreateWithFlags(&done_event_, cudaEventBlockingSync | cudaEventDisableTiming));
        CK(cudaEventRecord(done_event_, stream_));
        CK(cudaEventSynchronize(done_event_));
    } else {
        CK(cudaStreamSynchronize(stream_));
    }
    CK(cudaGetLastError());
    if (trace) t3 = clk::now();
    int err = *h_out_.as<int>();
    if (err != 0)
        throw std::runtime_error("Softmax input sum must be strictly positive (board " + std::to_string(err - 1) +
                                 "): the network produced NaN/inf logits");
    const OutBlock ob = out_block(max_batch_);
    std::memcpy(out_values, h_out_.as<uint8_t>() + ob.off_values, size_t(batch) * 5 * 4);
    if (staged_moves_) std::memcpy(out_policy, h_out_.as<uint8_t>() + ob.off_probs, staged_moves_ * 4);
    if (trace) {
        t4 = clk::now();
        auto us = [](clk::time_point a, clk::time_point b) { return std::chrono::duration<double, std::micro>(b - a).count(); };
        trace_[0] += us(t0, t1);
        trace_[1] += us(t1, t2);
        trace_[2] += us(t2, t3);
        trace_[3] += us(t3, t4);
        trace_[4] += 1;
    }
}

void Net::encode_planes(const uint8_t* bits, const float* scalars, int batch, float* out_nchw) {
    check_batch(batch);
    require_mapper();
    if (batch == 0) return;
    CK(cudaSetDevice(device_));
    upload_packed(bits, scalars, batch, nullptr, nullptr);
    InBlock ib = in_block(max_batch_, scalar_count_, bits_stride_);
    launch_encode_nchw_f32(d_mv_off_.as<uint8_t>() + ib.off_bits, reinterpret_cast<const float*>(d_mv_off_.as<uint8_t>() + ib.off_scalars),
                           batch, bits_stride_, scalar_count_, bool_channels_, spec_.area(), d_nchw_.as<float>(), stream_);
    CK(cudaMemcpyAsync(out_nchw, d_nchw_.ptr, size_t(batch) * spec_.cin * spec_.area() * 4, cudaMemcpyDeviceToHost, stream_));
    CK(cudaStreamSynchronize(stream_));
    CK(cudaGetLastError());
}

void Net::stage_packed(const uint8_t* bits, const float* scalars, int batch, const uint32_t* mv_idx, const uint32_t* mv_off) {
    check_batch(batch);
    require_mapper();
    CK(cudaSetDevice(device_));
    upload_packed(bits, scalars, batch, mv_idx, mv_off);
    CK(cudaStreamSynchronize(stream_));
}

void Net::flush_l2() {
    const size_t bytes = size_t(256) << 20;  // > 126 MB L2
    if (!d_flush_.ptr) d_flush_.alloc(bytes, false);
    CK(cudaMemsetAsync(d_flush_.ptr, 1, bytes, stream_));
}

void Net::time_staged(int iters, bool flush, float* ms_out) {
    require_mapper();
    if (staged_batch_ <= 0) throw std::runtime_error("no staged batch: call kzb_stage_packed first");
    CK(cudaSetDevice(device_));
    std::vector<cudaEvent_t> ev(size_t(iters) * 2);
    for (auto& e : ev) CK(cudaEventCreate(&e));
    for (int i = 0; i < iters; i++) {
        if (flush) flush_l2();
        CK(cudaEventRecord(ev[2 * i], stream_));
        run_encode(staged_batch_, nullptr);
        run_network(staged_batch_, nullptr);
        run_tail(staged_batch_, true, nullptr);
        CK(cudaEventRecord(ev[2 * i + 1], stream_));
    }
    CK(cudaStreamSynchronize(stream_));
    CK(cudaGetLastError());
    for (int i = 0; i < iters; i++) CK(cudaEventElapsedTime(&ms_out[i], ev[2 * i], ev[2 * i + 1]));
    for (auto& e : ev) cudaEventDestroy(e);
}

void Net::profile_staged(bool flush, std::vector<std::string>& names, std::vector<float>& ms) {
    require_mapper();
    if (staged_batch_ <= 0) throw std::runtime_error("no staged batch: call kzb_stage_packed first");
    CK(cudaSetDevice(device_));
    const char* tl_env = std::getenv("KZB_TIMELINE");  // development aid: per-CTA clock stamps of the tower8 or heads8 step
    if (tl_env && tl_env[0]) {
        timeline_step_ = tl_env;
        d_timeline_.alloc(size_t(num_sms_) * 1024 * 8, true);
    }
    std::vector<cudaEvent_t> ev;
    names.clear();
    auto mark = [&]() {
        cudaEvent_t e;
        CK(cudaEventCreate(&e));
        CK(cudaEventRecord(e, stream_));
        ev.push_back(e);
    };
    StepHook hook = [&](const char* name) {
        names.push_back(name);
        mark();
    };
    if (flush) flush_l2();
    mark();
    run_encode(staged_batch_, hook);
    run_network(staged_batch_, hook);
    run_tail(staged_batch_, true, hook);
    CK(cudaStreamSynchronize(stream_));
    CK(cudaGetLastError());
    ms.resize(names.size());
    for (size_t i = 0; i < names.size(); i++) CK(cudaEventElapsedTime(&ms[i], ev[i], ev[i + 1]));
    for (auto& e : ev) cudaEventDestroy(e);
    if (!timeline_step_.empty()) {
        std::vector<unsigned long long> h(size_t(num_sms_) * 1024);
        CK(cudaMemcpy(h.data(), d_timeline_.ptr, h.size() * 8, cudaMemcpyDeviceToHost));
        if (FILE* f = std::fopen("gpurun_out/timeline.txt", "w")) {
            for (int c = 0; c < num_sms_; c++) {
                for (int j = 0; j < 1024; j++) std::fprintf(f, "%lld ", h[c * 1024 + j] ? (long long)(h[c * 1024 + j] - h[c * 1024]) : -1LL);
                std::fprintf(f, "\n");
            }
            std::fclose(f);
        }
        timeline_step_.clear();
    }
}

}  // namespace kzb
