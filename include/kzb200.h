/*
 * kzb200.h -- C ABI of libkzb200.so: B200-native batched evaluation of kZero's AlphaZero ResNet.
 *
 * This is the drop-in boundary for ONE path of the reference: what `CudaNetwork` does between
 * `Network::evaluate_batch` and the GPU (rust/kz-core/src/network/cudnn.rs:18-88).  It replaces the
 * kn-cuda-eval / kn-cuda-sys / cuDNN dependency for that path; everything above the `Network` trait
 * (kz-selfplay executor threads, RandomSymmetryNetwork, MCTS) is an unchanged consumer.
 * Plain pointers and sizes only; all host pointers are owned by the caller and only used during the call.
 *
 * Threading (mirrors `evaluate_batch(&mut self)`, network/mod.rs:52-63): a kzb_net handle is NOT
 * thread-safe; different handles are independent (own stream, own buffers) and may be created, used and
 * destroyed concurrently from different threads, on the same or different devices.
 *
 * Errors: every int-returning function returns 0 on success and non-zero on failure; the message is
 * available (per thread) from kzb_last_error().  The reference panics in the same situations
 * (cudnn.rs:58 batch too large, common.rs:165-198 shape mismatch, common.rs:110 softmax sum not > 0);
 * the Rust shim turns a non-zero return into a panic to preserve that behaviour.
 * There is no CPU fallback: without a CUDA device every entry point that needs one fails.
 */
#ifndef KZB200_H
#define KZB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct kzb_net kzb_net;

#define KZB_PRECISION_FP32 0 /* CUDA-core fp32, <= 1e-4 max-abs vs the CPU executor            */
#define KZB_PRECISION_BF16 1 /* tcgen05 tensor cores: bf16 operands, fp32 accumulate (the fast path) */
/* tcgen05 kind::tf32 on the row kernels for every board: f32 activations rounded to TF32 (round to nearest, ties away), fp32
 * accumulate.  Logits and raw scalars within 4e-3 * max(1, max |logit|) of the f32 CPU executor, probabilities within 1e-3
 * (tests/test_tf32.py); about 7x closer than bf16 on deep towers. */
#define KZB_PRECISION_TF32 2

/* Replaces CudaDevice::all() (rust/kz-selfplay/src/server/server.rs:49-51). */
int kzb_device_count(void);

/* Thread-local message of the last failure on this thread ("" if none). */
const char* kzb_last_error(void);

/* Shapes of a loaded network, for the caller's own checks. */
typedef struct kzb_net_info {
    int32_t input_channels, board_h, board_w; /* graph input [BATCH, C, H, W]                 */
    int32_t policy_len;                       /* product of the policy output's non-batch dims */
    int32_t channels, depth;                  /* tower width / residual blocks                 */
    int32_t max_batch, precision, device;
    int32_t conv_mode;      /* 0: row kernels (dense rows; always in tf32), 1: 8x8-board kernels, -1: fp32 */
    double flops_per_position; /* algorithmic FLOPs (no padding/halo), SURVEY.md 8(d)          */
} kzb_net_info;

/* Replaces `CudaNetwork::new(mapper, &graph, max_batch_size, device)` (network/cudnn.rs:29-43) together
 * with `load_graph_from_onnx_path` + `optimize_graph` (rust/kz-selfplay/src/server/server_alphazero.rs:126-128):
 * parses the ONNX bytes, recognises the ResNet tower + heads, folds every BatchNorm, packs weights,
 * allocates device buffers for `max_batch` positions.  Fails with a message for graphs that are not the
 * reference architecture (python/lib/model/post_act.py).  Widths, in every precision: tower and policy conv1 up to 1024
 * channels, policy conv2 up to 256 output channels; a wider net fails with a message naming the layer and the limit.  Tensor-core
 * layers wider than 256 channels run in slices of at most 256 output channels, padded to a multiple of 64 (704 -> 768, 832 -> 896,
 * so that every slice keeps at least 128 channels). */
int kzb_net_create_from_onnx(int device, const void* onnx_bytes, size_t onnx_len, int max_batch, int precision,
                             kzb_net** out);

/* The same network from weights the caller already holds -- for a host that keeps the reference's `load_graph` untouched
 * (`load_graph_from_onnx_path` + `optimize_graph`, server_alphazero.rs:126-128) and hands the optimised Graph's constants over,
 * exactly what `CudaExecutor::new(device, &graph, batch)` receives today (network/cudnn.rs:32).  All pointers are read during the
 * call only.  Convolutions are [cout][cin][k][k] f32 + [cout] bias with their in-block BatchNorm already folded (optimize_graph
 * does that; kzb_net_create_from_onnx does it itself); the tower's trailing BatchNormalization (post_act.py:207) is passed as the
 * per-channel affine y = final_scale * x + final_shift and folded into the head convs here.  Conv-policy heads only (chess conv +
 * gather, ataxx, go); a network with the attention policy head goes through kzb_net_create_from_onnx. */
typedef struct kzb_conv_weights {
    int32_t cin, cout, ksize; /* ksize 3 (stride 1, zero padding 1) or 1 */
    const float* w;           /* [cout][cin][ksize][ksize] */
    const float* b;           /* [cout] */
} kzb_conv_weights;
typedef struct kzb_fc_weights {
    int32_t in, out;
    const float* w; /* [out][in] (Gemm with transB = 1) */
    const float* b; /* [out] */
} kzb_fc_weights;
/* channels and policy_conv1.cout: 1..1024; policy_conv2.cout: at most 256 (see kzb_net_create_from_onnx) */
typedef struct kzb_net_spec {
    int32_t input_channels, board_h, board_w, channels, depth;
    kzb_conv_weights first;         /* conv3x3 input_channels -> channels, bias, no ReLU (post_act.py:203)             */
    const kzb_conv_weights* blocks; /* 2 * depth conv3x3 channels -> channels, ReLU after each, residual add after every second */
    const float* final_scale;       /* [channels] or NULL (with final_shift): the trailing BatchNormalization as an affine */
    const float* final_shift;
    kzb_conv_weights scalar_conv;   /* conv1x1 channels -> hc, ReLU (post_act.py:10-23)                                */
    kzb_fc_weights fc1, fc2;        /* hc * H * W -> hs (ReLU) -> 5                                                    */
    kzb_conv_weights policy_conv1;  /* conv1x1 channels -> cp, ReLU (post_act.py:54-112)                               */
    kzb_conv_weights policy_conv2;  /* conv1x1 cp -> pc                                                                */
    int32_t has_extra;              /* go: extra pass-move logit = fc(flatten(conv1x1(channels -> 1)))  (post_act.py:63-84) */
    kzb_conv_weights extra_conv;
    kzb_fc_weights extra_fc;
    int32_t policy_len;
    const int32_t* policy_src;      /* [policy_len]: >= 0: element pc * H * W + sq of policy_conv2's output (what Flatten / Gather
                                       select); -1: constant zero (ataxx pass); -2 - e: output e of extra_fc (go pass)          */
} kzb_net_spec;
int kzb_net_create(int device, const kzb_net_spec* spec, int max_batch, int precision, kzb_net** out);

/* Twin of check_graph_shapes (network/common.rs:165-198): verifies the graph input is
 * [BATCH, scalar_count + bool_channels, board_h, board_w] and the policy has `policy_len` entries, and
 * tells the network how a packed record splits into scalar and bool planes (InputMapper::input_bool_shape /
 * input_scalar_count, rust/kz-core/src/mapping/mod.rs:20-22).  Required before the *_packed / encode calls. */
int kzb_net_bind_mapper(kzb_net* net, int scalar_count, int bool_channels, int board_h, int board_w, int policy_len);

int kzb_net_get_info(const kzb_net* net, kzb_net_info* out);

/* Host-only half of kzb_net_create_from_onnx: parse + recognise + fold, no device touched (max_batch,
 * precision, device, conv_mode are reported as -1).  Lets a caller validate a network file, and lets the
 * host logic be tested on a machine without a GPU. */
int kzb_onnx_inspect(const void* onnx_bytes, size_t onnx_len, kzb_net_info* out);

/* Replaces dropping the CudaNetwork (executor.rs:326-331 drops the old net before loading the next). */
void kzb_net_destroy(kzb_net* net);

/* Exact semantic twin of `CudaExecutor::evaluate(&[DTensor::F32(input)])` (network/cudnn.rs:73):
 * nchw_in [batch, C, H, W] f32 -> out_scalars [batch, 5] raw head outputs, out_policy_logits [batch, policy_len].
 * Computes exactly `batch` rows (1 <= batch <= max_batch); rows are independent of each other. */
int kzb_eval_planes(kzb_net* net, const float* nchw_in, int batch, float* out_scalars, float* out_policy_logits);

/* The fused fast path: everything `CudaNetwork::evaluate_batch` does (cudnn.rs:55-87) in one call.
 *   bits    [batch, ceil(bool_channels*H*W/8)]  BitBuffer::storage() per board (mapping/bit_buffer.rs:68-70)
 *   scalars [batch, scalar_count] f32           as pushed by InputMapper::encode_input (mapping/mod.rs:38)
 *   mv_idx / mv_off: CSR list of PolicyMapper::move_to_index over board.available_moves(), in iteration
 *                    order (same as collect_policy_indices, rust/kz-selfplay/src/binary_output.rs:299-315);
 *                    mv_off has batch+1 entries, mv_off[0] == 0; a terminal board has an empty range.
 *   out_values [batch, 5]: value = tanh(s0), wdl = softmax(s1..s3), moves_left = s4   (network/common.rs:59-74)
 *   out_policy [mv_off[batch]]: softmax over each board's legal moves only            (network/common.rs:76-86)
 * Returns non-zero (and writes no NaN probabilities silently) if any softmax sum is not > 0 (common.rs:110). */
int kzb_eval_packed(kzb_net* net, const uint8_t* bits, const float* scalars, int batch, const uint32_t* mv_idx,
                    const uint32_t* mv_off, float* out_values, float* out_policy);

/* Board symmetries on the GPU ("next" row N4; replaces RandomSymmetryNetwork's host-side work, network/symmetry.rs:41-67,
 * 126-148: `board.map(sym)` before the evaluation and `unmap_eval` after it).  The tables are supplied by the caller and are
 * game-agnostic here:
 *   square_src [n_sym][H*W]      plane square sq of the MAPPED board is square square_src[s][sq] of the original board
 *   policy_map [n_sym][policy_len]  policy index of map_move(sym, mv) for the move with index i (for ataxx: the `map_mv`
 *                                rows of python/lib/mapping/ataxx_symmetry.json)
 * kzb_eval_packed_sym takes the ORIGINAL boards' records and legal-move indices plus one symmetry id per board; the input
 * planes are transformed while they are expanded and every legal index is looked up through policy_map before the
 * masked softmax, so the result is what RandomSymmetryNetwork returns for that choice of symmetries. */
int kzb_net_set_symmetries(kzb_net* net, int n_sym, const int32_t* square_src, const int32_t* policy_map);
int kzb_eval_packed_sym(kzb_net* net, const uint8_t* bits, const float* scalars, const uint8_t* sym, int batch,
                        const uint32_t* mv_idx, const uint32_t* mv_off, float* out_values, float* out_policy);

/* K2 alone, for bit-exact parity checks: twin of InputMapper::encode_input_full (mapping/mod.rs:40-63),
 * out_nchw [batch, scalar_count + bool_channels, H, W] f32, produced on the GPU. */
int kzb_encode_planes(kzb_net* net, const uint8_t* bits, const float* scalars, int batch, float* out_nchw);

/* ---- measurement hooks (bench.py); not part of the reference's interface ------------------------- */

/* Upload one packed batch into the network's device buffers (inputs resident in HBM afterwards). */
int kzb_stage_packed(kzb_net* net, const uint8_t* bits, const float* scalars, int batch, const uint32_t* mv_idx,
                     const uint32_t* mv_off);
/* Run the device side of kzb_eval_packed on the staged batch `iters` times, each iteration timed with
 * CUDA events on the network's own stream; ms_out[iters].  If flush_l2 != 0 a 256 MiB scratch buffer is
 * overwritten before every iteration, outside the timed region. */
int kzb_time_staged(kzb_net* net, int iters, int flush_l2, float* ms_out);
/* Same, but per kernel launch of ONE iteration: names_out receives '\n'-separated step names,
 * ms_out[*n_steps] the CUDA-event duration of each launch.  Returns non-zero if the buffers are too small. */
int kzb_profile_staged(kzb_net* net, int flush_l2, char* names_out, size_t names_cap, float* ms_out, int ms_cap,
                       int* n_steps);
/* Number of kernel launches one kzb_eval_packed call issues. */
int kzb_launches_per_eval(const kzb_net* net);

/* ---- self-play driver ("next" row N1, SURVEY.md 8(f); BASELINE.json configs[3]) ---------------------------------
 * The producer side of the hot path: generator threads running concurrent AlphaZero tree searches and executor
 * threads batching their requests into the evaluator above.  Replaces, for measurement purposes, what
 * `selfplay_server_main` spawns per device (rust/kz-selfplay/src/server/server_alphazero.rs:32-124):
 * `generator_alphazero_main` (generator_alphazero.rs:23-260) + `batched_executor_loop` (executor.rs:27-146), with the
 * search of rust/kz-core/src/zero/{step,node,tree}.rs.  No TCP control plane, no game files. */

#define KZB_GAME_SYNTH_CHESS 0 /* chess-shaped synthetic game: 13x8x8 bools + 8 scalars, 1880-move policy, 20..45 legal moves */
#define KZB_GAME_ATAXX7 1      /* 7x7 ataxx, AtaxxStdMapper encoding (rust/kz-core/src/mapping/ataxx.rs)                      */
#define KZB_GAME_GO9 2         /* 9x9 go, GoStdMapper encoding without territory planes (rust/kz-core/src/mapping/go.rs)      */
#define KZB_GAME_CHESS 3       /* chess with legal move generation, ChessStdMapper encoding and the flat 1880-move policy      */
#define KZB_GAME_GO9_TERRITORY 4 /* 9x9 go with GoStdMapper::new(9, true): 7 bool planes, what server.rs:193 constructs              */

/* Field for field the reference's settings: StartupSettings (rust/kz-selfplay/src/server/protocol.rs:11-40:
 * cpu_threads_per_device, gpu_threads_per_device, gpu_batch_size, search_batch_size) and Settings (protocol.rs:58-110). */
typedef struct kzb_selfplay_config {
    int32_t game;
    int32_t visits;            /* full_iterations: root visits per move                                             */
    int32_t search_batch;      /* search_batch_size: requests gathered per tree per round (virtual loss)            */
    int32_t gpu_batch;         /* gpu_batch_size: max positions per evaluator call                                  */
    int32_t cpu_threads;       /* cpu_threads_per_device: generator threads                                         */
    int32_t gpu_threads;       /* gpu_threads_per_device: executor threads, one network instance each               */
    int32_t concurrent_games;  /* 0 = the reference's ceil((gpu_threads + 1) * gpu_batch / search_batch)             */
    int32_t max_game_length;
    int32_t cache_size;        /* per-game LRU evaluation cache                                                     */
    int32_t zero_temp_move_count;
    int32_t max_moves;         /* stop after this many played moves (0 = no limit)                                  */
    int32_t max_games;         /* stop after this many finished games (0 = no limit): one record file = games_per_gen games */
    int32_t part_iterations;   /* root visits of a non-full search (Settings::part_iterations)                      */
    float full_search_prob;    /* probability that a move gets the full `visits` (Settings::full_search_prob)       */
    float duration_s;
    float temperature;         /* move selection temperature                                                        */
    float dirichlet_alpha, dirichlet_eps;
    float policy_temperature_root, policy_temperature_child; /* search_policy_temperature_*                        */
    float exploration_weight, moves_left_weight, moves_left_clip, moves_left_sharpness; /* UctWeights              */
    float fpu_root;
    int32_t fpu_root_relative; /* FpuMode: 0 fixed, 1 relative                                                      */
    float fpu_child;
    int32_t fpu_child_relative;
    float virtual_loss;        /* search_virtual_loss_weight                                                        */
    int32_t q_mode_wdl;        /* QMode: 0 value head, 1 wdl head with draw_score                                   */
    float draw_score;
    int32_t executor_blocking_sync; /* 0: executor threads spin while the GPU works (lowest latency; needs a core each),
                                       1: they sleep on a blocking event (use when generators and executors share cores) */
    int32_t dummy_network;       /* 1: answer every request with uniform wdl / policy instead of evaluating a network -- the
                                    reference's DummyNetwork / UseDummyNetwork (network/dummy.rs:44-60); needs no GPU.
                                    2: a deterministic pseudo-network (sharp policies and values hashed from the encoded
                                    record) for host-side profiling and tests, also without a GPU                      */
    const char* output_prefix;   /* NULL / "": no records; else finished games are written to <prefix>.bin/.off/.json in the
                                    reference's format (rust/kz-selfplay/src/binary_output.rs:128-297)                      */
    uint64_t seed;
} kzb_selfplay_config;

/* The counters of the reference's collector line `evals/s: real / cached / potential` (collector.rs:172-191). */
typedef struct kzb_selfplay_stats {
    double seconds;
    uint64_t real_evals;      /* positions evaluated by the network                                                 */
    uint64_t cached_evals;    /* requests served from the per-game LRU caches                                       */
    uint64_t potential_evals; /* batches * gpu_batch                                                                */
    uint64_t batches;
    uint64_t max_batch;
    uint64_t games_finished, moves_played;
    uint64_t root_visits;     /* sum of root visits of the finished searches                                        */
    uint64_t concurrent_games;
    uint64_t games_written;   /* games in the record file (all of it, when the run continued a file left open by an interrupt)  */
    uint64_t interrupted;     /* 1: a session run returned on kzb_selfplay_request_interrupt before max_games games were in
                               * its record file; the file stays open in the session and the next run with the same
                               * output_prefix continues it                                                              */
} kzb_selfplay_stats;

/* The reference's typical production settings (python/main/loop_main_alpha.py:24-52, UctWeights::default). */
void kzb_selfplay_default_config(kzb_selfplay_config* config);

/* Run self-play on `device` with the network in `onnx_bytes` until duration_s / max_moves; MCTS nodes/sec =
 * (real_evals + cached_evals) / seconds, NN positions/sec = real_evals / seconds. */
int kzb_selfplay_run(int device, const void* onnx_bytes, size_t onnx_len, int precision, const kzb_selfplay_config* config,
                     kzb_selfplay_stats* stats);

/* Ask every kzb_selfplay_run in this process to return as soon as possible (the `Stop` command, protocol.rs:37);
 * callable from any thread.  The flag stays set -- a run that starts while it is set returns at once -- until
 * kzb_selfplay_clear_stop: a Stop that arrives while a network is still loading must not be lost. */
void kzb_selfplay_request_stop(void);
void kzb_selfplay_clear_stop(void);

/* Ask every kzb_selfplay_session_run in this process to return NOW without closing its record file, so that the caller can start
 * the next run -- with a new network or new settings -- under the same games and into the same file: how a network that arrives in
 * the middle of a generation is put to work at once, as the reference's executors do (rust/kz-selfplay/src/server/executor.rs:50-65,
 * 320-342) instead of at the next file boundary.  Sticky like the stop flag, until kzb_selfplay_clear_interrupt; ignored by
 * kzb_selfplay_run (which has no session to keep the file in). */
void kzb_selfplay_request_interrupt(void);
void kzb_selfplay_clear_interrupt(void);

/* A session keeps the concurrent games of one server connection alive BETWEEN runs: every kzb_selfplay_session_run plays until
 * config->max_games more games have finished (one record file = games_per_gen games), writes them to config->output_prefix and
 * returns; the games still in flight -- boards, search trees, per-game caches, the positions recorded so far -- continue in the
 * next run, with that run's network and settings.  This is what the reference's server does: its generators run across file
 * boundaries, the collector only rotates the output file (rust/kz-selfplay/src/server/collector.rs:59-116), and a new network is
 * swapped in under running games (executor.rs:320-342) -- so long games are not dropped and the data has no length bias.
 * config->max_games counts the games in the record file: a run that continues a file left open by an interrupt (same output_prefix)
 * returns when the file holds max_games games.  Destroying a session finishes a file it still holds open.
 * The game, cpu_threads and the derived number of concurrent games are fixed by the first run (StartupSettings, protocol.rs:11-28). */
typedef struct kzb_selfplay_session kzb_selfplay_session;
int kzb_selfplay_session_create(int game, kzb_selfplay_session** out);
int kzb_selfplay_session_run(kzb_selfplay_session* session, int device, const void* onnx_bytes, size_t onnx_len, int precision,
                             const kzb_selfplay_config* config, kzb_selfplay_stats* stats);
void kzb_selfplay_session_destroy(kzb_selfplay_session* session);

/* Host-only (no GPU): one tree search of `config->visits` visits from the position `plies` random moves into game
 * `game_seed`, gathered in rounds of `config->search_batch` (virtual loss) and answered by a deterministic stand-in
 * network (eval_kind 0: uniform, the reference's DummyNetwork, network/dummy.rs:44-60; 1: hashed pseudo-random).
 * Exists so that the search (zero_step_gather / zero_step_apply / uct) can be checked against the oracle's restatement. */
typedef struct kzb_mcts_trace_out {
    int32_t capacity;       /* in: length of the three arrays below                                                 */
    int32_t n_children;     /* out: root children = available moves, in available_moves order                       */
    uint64_t* child_visits; /* complete_visits per root child                                                       */
    uint32_t* child_moves;  /* the child's move (= its policy index in the bundled games)                           */
    float* child_policy;    /* net_policy per root child                                                            */
    float root_values[5];   /* Tree::values(): value, win, draw, loss, moves_left from the root player's view       */
    uint64_t root_visits, tree_nodes, evals;
} kzb_mcts_trace_out;
int kzb_mcts_trace(const kzb_selfplay_config* config, uint64_t game_seed, int plies, int eval_kind, kzb_mcts_trace_out* out);

#ifdef __cplusplus
}
#endif
#endif /* KZB200_H */
