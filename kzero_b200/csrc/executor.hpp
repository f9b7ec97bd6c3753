// The network object behind the C ABI: device buffers, packed weights, TMA tensor maps and the fixed
// launch schedule for one AlphaZero ResNet.  The B200 build's counterpart of kn-cuda-eval's
// `CudaExecutor` (planner + executor; call sites rust/kz-core/src/network/cudnn.rs:32,73).
#pragma once
#include <functional>
#include <memory>
#include <string>
#include <unordered_map>
#include <vector>

#include "kernels.cuh"
#include "net_spec.hpp"

namespace kzb {

struct DeviceBuffer {
    void* ptr = nullptr;
    size_t bytes = 0;
    DeviceBuffer() = default;
    DeviceBuffer(const DeviceBuffer&) = delete;
    DeviceBuffer& operator=(const DeviceBuffer&) = delete;
    ~DeviceBuffer();
    void alloc(size_t n, bool zero = true);
    template <typename T>
    T* as() const {
        return static_cast<T*>(ptr);
    }
};

struct PinnedBuffer {
    void* ptr = nullptr;
    size_t bytes = 0;
    PinnedBuffer() = default;
    PinnedBuffer(const PinnedBuffer&) = delete;
    PinnedBuffer& operator=(const PinnedBuffer&) = delete;
    ~PinnedBuffer();
    void alloc(size_t n);
    template <typename T>
    T* as() const {
        return static_cast<T*>(ptr);
    }
};

// one conv launch of the schedule
struct ConvStep {
    std::string name;
    int taps = 9;
    // tensor-core form (bf16, or f32 rounded to TF32): conv_i2c.cu
    CUtensorMap tmap_out{}, tmap_res{};  // output / residual rows, box (32 channels, 32 rows): SWIZZLE_64B bf16, SWIZZLE_128B f32
    CUtensorMap tmap_i2c{};  // im2col map of the input rows
    // output channel slices: split0 slices of n / split0 <= 256 channels, or (split_double, small batches) 2 * split0;
    // tmap_w[i]: weight box of half a slice (n / split0 / 2, n / split0 / 4 rows)
    int split0 = 1;
    bool split_double = false;
    CUtensorMap tmap_w[2]{};
    ConvTcParams tc{};
    DeviceBuffer w_tc;  // [n][taps*cin_pad] bf16, or f32 rounded to TF32
    // fp32 form
    ConvF32Params f32{};
    DeviceBuffer w_f32;  // [taps][cin][cout]
    DeviceBuffer bias;   // [n] f32
};

class Net {
public:
    Net(int device, const void* onnx, size_t len, int max_batch, int precision);
    Net(int device, NetSpec spec, int max_batch, int precision);
    ~Net();

    void bind_mapper(int scalar_count, int bool_channels, int h, int w, int policy_len);
    void eval_planes(const float* nchw, int batch, float* out_scalars, float* out_logits);
    void eval_packed(const uint8_t* bits, const float* scalars, int batch, const uint32_t* mv_idx, const uint32_t* mv_off,
                     float* out_values, float* out_policy, const uint8_t* sym = nullptr);
    void set_symmetries(int n_sym, const int32_t* square_src, const int32_t* policy_map);
    void encode_planes(const uint8_t* bits, const float* scalars, int batch, float* out_nchw);
    void stage_packed(const uint8_t* bits, const float* scalars, int batch, const uint32_t* mv_idx, const uint32_t* mv_off);
    void time_staged(int iters, bool flush_l2, float* ms_out);
    void profile_staged(bool flush_l2, std::vector<std::string>& names, std::vector<float>& ms);
    // kzb_eval_packed waits for the GPU by spinning (lowest latency, default) or by sleeping on a blocking event
    void set_blocking_sync(bool on) { blocking_sync_ = on; }
    int launches_per_eval() const {
        int n = int(convs_.size()) + 2 - (use_tower8k_ ? tower_layers_ - 1 : 0);
        if (use_heads8_) n -= int(convs_.size() - head_first_);  // head convs + tail become one launch
        return n;
    }

    const NetSpec& spec() const { return spec_; }
    int device() const { return device_; }
    int max_batch() const { return max_batch_; }
    int precision() const { return precision_; }
    int conv_mode() const { return precision_ != 0 ? mode_ : -1; }

private:
    using StepHook = std::function<void(const char*)>;
    void build_tc();  // bf16 and TF32: the tcgen05 kernels
    void build_f32();
    void check_batch(int batch) const;
    void require_mapper() const;
    void upload_packed(const uint8_t* bits, const float* scalars, int batch, const uint32_t* mv_idx, const uint32_t* mv_off);
    void run_encode(int batch, const StepHook& hook);
    void run_network(int batch, const StepHook& hook);
    HeadOutputs head_outputs(int batch, bool packed, bool to_host) const;
    void run_tail(int batch, bool packed, const StepHook& hook, bool to_host = false);
    void flush_l2();

    int device_, max_batch_, precision_;
    NetSpec spec_;
    cudaStream_t stream_ = nullptr;
    int num_sms_ = 148;

    int scalar_count_ = -1, bool_channels_ = -1, bits_stride_ = 0;
    RowLayout lay_{};
    int mode_ = 0;       // tensor-core paths, dense rows: 0 row kernels (any board; always in TF32), 1 8x8 boards (tower8k / heads8 where they apply)
    int rows_alloc_ = 0; // multiple of 128
    int cin_pad_ = 0, c_pad_ = 0, cp_pad_ = 0, s1_stride_ = 16, pm_stride_ = 0;
    Act act_ = Act::kBf16;
    bool embed8_ = false;  // a board smaller than 8x8 embedded in the 8x8 grid of the whole-tower kernel
    int boards_i2c_ = 0;   // boards covered by the im2col tensor maps (>= every 256-pixel tile of a full batch)

    DeviceBuffer d_bits_, d_scalars_, d_mv_idx_, d_mv_off_, d_nchw_;
    DeviceBuffer act_in_, act_x_, act_t_, act_h1_, act_s1_, act_pm_, act_att_;
    int att_stride_ = 0;
    DeviceBuffer d_fc1_t_, d_fc1_b_, d_fc2_w_, d_fc2_b_, d_extra_w_, d_policy_src_, d_att_entries_;
    DeviceBuffer d_out_scalars_, d_out_logits_, d_err_;
    DeviceBuffer d_flush_, d_timeline_;
    std::string timeline_step_;
    PinnedBuffer h_in_, h_out_;
    size_t mv_cap_ = 0;
    bool blocking_sync_ = false;
    // CUDA graphs of the kernel sequence, one per batch size that keeps coming back (KZB_NO_GRAPH=1 disables): the role of the
    // reference's MultiBatchNetwork (rust/kz-core/src/network/multibatch.rs:19-35), without its padding -- a graph computes exactly
    // its batch.  A size is captured the second time it is seen (the full batch: the first time); at most kMaxGraphs are kept.
    bool use_graph_ = true;
    static constexpr size_t kMaxGraphs = 48;
    struct BatchGraph {
        cudaGraphExec_t exec = nullptr;
        int seen = 0;
    };
    std::unordered_map<int, BatchGraph> graphs_;
    int n_sym_ = 0;
    const uint8_t* cur_sym_ = nullptr;  // device pointer while an evaluation with symmetries is in flight
    DeviceBuffer d_sym_square_, d_sym_policy_, d_sym_;
    PinnedBuffer h_sym_;
    cudaEvent_t done_event_ = nullptr;
    double* trace_ = nullptr;  // KZB_TRACE=1: accumulated host-side phase times of eval_packed
    int staged_batch_ = 0;
    size_t staged_moves_ = 0;

    std::vector<std::unique_ptr<ConvStep>> convs_;

    // fused heads kernel (8x8 boards, conv policy head): replaces the three head conv steps and the tail kernel
    bool use_heads8_ = false;
    size_t head_first_ = 0;  // index of the first head conv step in convs_
    Heads8Maps heads_maps_{};
    Heads8Params heads_params_{};

    // whole-tower persistent kernel (8x8 boards, tower8k.cu): covers convs_[0 .. tower_layers_); k-chunk-major activation
    // tensors A[kc][board][y][x][8]
    bool use_tower8k_ = false;
    int tower_layers_ = 0;
    Tower8Params tower_params_{};
    DeviceBuffer d_tower_layers_, w_tower_, act_xt_;
    Tower8kMaps tower_kmaps_{};
    int tower_k_b_slots_ = 0;
    DeviceBuffer act_ink_, act_xk_, act_tk_;
};

// thread-local error plumbing for the C ABI
void set_last_error(const std::string& msg);
const char* last_error();

}  // namespace kzb
