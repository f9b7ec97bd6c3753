"""The TF32 precision (KZB_PRECISION_TF32): tcgen05 kind::tf32 on the row kernels for every board, f32 activations rounded to TF32.

Every value a TF32 MMA reads is stored TF32-exact (round to nearest, ties away from zero, low 13 mantissa bits cleared:
tf32_round in kzero_b200/csrc/kernels.cuh), so the results do not depend on what the tensor core does with the low bits.

CPU: the host rounding on known bit patterns; a CPU emulation of the TF32 arithmetic (every Conv operand and every residual Add
rounded to TF32, f32 accumulation) stays below half of the GPU bar on deep towers; the exact-arithmetic probe nets are TF32-exact;
precision values are checked.
GPU: the probe matrix bit for bit against the float64 reference (the rounding on store: test_rounding_probes.py); random-init
nets against the f32 oracle within 4e-3 * max(1, max |logit|) on logits and raw scalars and 1e-3 on probabilities; batch
independence, graph replay, the packed decode, NaN reporting, the launch count of an 8x8 net (it takes the row path), and self-play.
"""
import subprocess
from pathlib import Path

import numpy as np
import pytest

import oracle
import test_exact_probe_nets as probes
from oracle.graph_exec import OnnxOracle
from helpers import NET_NAMES, bf16_emulation, load_net_fixture
from kzero_b200 import netgen
from kzero_b200.build import CSRC, _nvcc
from kzero_b200.network import B200Network, KzbError, PRECISION_BF16, PRECISION_TF32, mapper_for

TF32 = PRECISION_TF32
TF32_TOL = 4e-3  # logits and raw scalars: TF32_TOL * max(1, max |logit|)
TF32_PROB_TOL = 1e-3
FIXTURE_GAMES = {"ataxx7_2x32": "ataxx-7", "chess_conv_2x32": "chess", "chess_att_2x32": "chess-att", "go9_2x32": "go-9",
                 "ataxx5_scripted_1x16": "ataxx-5"}


def tf32_round(a):
    """numpy twin of tf32_round (kernels.cuh)."""
    u = np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)
    finite = (u & np.uint32(0x7F800000)) != np.uint32(0x7F800000)
    nan = ~finite & ((u & np.uint32(0x007FFFFF)) != 0)
    u = np.where(finite, u + np.uint32(0x1000), u)
    u = np.where(nan, u | np.uint32(0x00400000), u)
    return (u & np.uint32(0xFFFFE000)).astype(np.uint32).view(np.float32)


def tf32_emulation(onnx_bytes):
    """The oracle's op-by-op interpreter with the arithmetic of the TF32 path: every Conv reads TF32-rounded activations and
    weights and accumulates in f32; every Add (the residual stream) is stored TF32-rounded.  Conv via torch's CPU kernels."""

    class Emulation(OnnxOracle):
        def _run_node(self, node, env):
            if node.op == "Conv":
                env = dict(env)
                env[node.inputs[0]] = tf32_round(env[node.inputs[0]])
                env[node.inputs[1]] = tf32_round(env[node.inputs[1]])
                return super()._run_node(node, env)
            out = super()._run_node(node, env)
            if node.op == "Add":
                out = [tf32_round(out[0])]
            return out

    return Emulation(onnx_bytes, conv_backend="torch")


def _planes(spec, bits, scalars):
    return oracle.expand_planes(bits, scalars, (spec.bool_channels, spec.board_size, spec.board_size), spec.scalar_channels)


# ----------------------------------------------------------------------------------------------------------- CPU: rounding
ROUNDING_CASES = [  # (input bits, expected bits)
    (0x3F800000, 0x3F800000),  # 1.0
    (0x3F800FFF, 0x3F800000),  # just below half a TF32 ulp
    (0x3F801000, 0x3F802000),  # a tie rounds away from zero (to even would keep 1.0)
    (0xBF801000, 0xBF802000),  # and so on the negative side
    (0x3F803000, 0x3F804000),  # a tie above an odd mantissa
    (0x3FFFF000, 0x40000000),  # the carry reaches the exponent
    (0x7F7FE000, 0x7F7FE000),  # the largest TF32 value
    (0x7F7FEFFF, 0x7F7FE000),
    (0x7F7FF000, 0x7F800000),  # the midpoint above it, and the largest finite f32: Inf
    (0x7F7FFFFF, 0x7F800000),
    (0xFF7FFFFF, 0xFF800000),
    (0x7F800000, 0x7F800000),  # +-Inf stay
    (0xFF800000, 0xFF800000),
    (0x7FC00000, 0x7FC00000),  # NaN stays NaN, also when its payload sits in the low 13 bits
    (0x7F800001, 0x7FC00000),
    (0xFF801FFF, 0xFFC00000),
    (0x7F802000, 0x7FC02000),
    (0x00000000, 0x00000000),  # zeros and subnormals
    (0x80000000, 0x80000000),
    (0x00000001, 0x00000000),
    (0x00000FFF, 0x00000000),
    (0x00001000, 0x00002000),
    (0x807FF000, 0x80800000),  # the largest subnormal's neighbourhood rounds up to the smallest normal
    (0x007FE000, 0x007FE000),
]

HOST_PROGRAM = r"""
#include <cstdio>
#include "kernels.cuh"
int main() {
    unsigned u;
    while (std::scanf("%x", &u) == 1) {
        float x, y;
        std::memcpy(&x, &u, 4);
        y = kzb::tf32_round(x);
        std::memcpy(&u, &y, 4);
        std::printf("%08x\n", u);
    }
}
"""


def _host_tf32_round(tmp_path, bits):
    """The host rounding the executor applies to the weights, compiled from kernels.cuh."""
    src = tmp_path / "tf32_round.cpp"
    src.write_text(HOST_PROGRAM)
    exe = tmp_path / "tf32_round"
    cuda_include = str(Path(_nvcc()).resolve().parent.parent / "include")
    subprocess.run(["g++", "-O2", "-std=c++17", "-I", str(CSRC), "-I", cuda_include, "-o", str(exe), str(src)], check=True)
    out = subprocess.run([str(exe)], input="\n".join(f"{b:08x}" for b in bits), capture_output=True, text=True, check=True).stdout
    return np.array([int(v, 16) for v in out.split()], dtype=np.uint32)


def test_tf32_round_known_bit_patterns(tmp_path):
    inp = np.array([c[0] for c in ROUNDING_CASES], dtype=np.uint32)
    want = np.array([c[1] for c in ROUNDING_CASES], dtype=np.uint32)
    got_np = tf32_round(inp.view(np.float32)).view(np.uint32)
    got_host = _host_tf32_round(tmp_path, inp)
    for i, (a, b) in enumerate(ROUNDING_CASES):
        assert got_np[i] == b, f"numpy: {a:08x} -> {got_np[i]:08x}, want {b:08x}"
        assert got_host[i] == b, f"kernels.cuh: {a:08x} -> {got_host[i]:08x}, want {b:08x}"
    # random bit patterns (every class of float): the host code and the numpy twin agree; finite results are the nearest TF32 value
    rnd = np.random.default_rng(5).integers(0, 1 << 32, size=20000, dtype=np.uint64).astype(np.uint32)
    host = _host_tf32_round(tmp_path, rnd)
    assert np.array_equal(host, tf32_round(rnd.view(np.float32)).view(np.uint32))
    with np.errstate(invalid="ignore"):  # NaN payloads
        x = rnd.view(np.float32).astype(np.float64)
        r = host.view(np.float32).astype(np.float64)
    ok = np.isfinite(r) & np.isfinite(x)
    assert np.array_equal(np.isnan(x), np.isnan(r))
    assert (host[ok] & 0x1FFF == 0).all()
    ulp = np.exp2(np.floor(np.log2(np.maximum(np.abs(x[ok]), 2.0 ** -126))) - 10)
    assert (np.abs(r[ok] - x[ok]) <= ulp / 2).all()


# ----------------------------------------------------------------------------------------------------------- CPU: emulation
@pytest.mark.parametrize("game,depth,ch,n", [("chess", 16, 128, 16), ("go-9", 20, 256, 4), ("go-19", 40, 256, 1)])
def test_tf32_emulation_of_deep_towers_is_within_half_the_bar(game, depth, ch, n, capsys):
    spec = netgen.game_spec(game)
    onnx_bytes = netgen.build_onnx(spec, depth, ch, seed=0)
    bits, scalars, _, _ = netgen.synthetic_positions(spec, n, seed=1)
    x = _planes(spec, bits, scalars)
    ref_s, ref_p = OnnxOracle(onnx_bytes, conv_backend="torch").run(x)
    s, p = tf32_emulation(onnx_bytes).run(x)
    _, bp = bf16_emulation(onnx_bytes).run(x)
    scale = max(1.0, float(np.abs(ref_p).max()))
    err, err_s, err_bf16 = float(np.abs(p - ref_p).max()), float(np.abs(s - ref_s).max()), float(np.abs(bp - ref_p).max())
    with capsys.disabled():
        print(f"\n[{game} {depth}x{ch} n={n}] emulated vs f32 oracle: TF32 max |dlogit| {err:.5f}, bf16 {err_bf16:.5f}; TF32 max |dscalar| "
              f"{err_s:.5f}; logit scale {scale:.2f}, GPU bar {TF32_TOL * scale:.5f}")
    assert err <= 0.5 * TF32_TOL * scale
    assert err_s <= 0.5 * TF32_TOL * scale
    assert err < 0.5 * err_bf16


# ----------------------------------------------------------------------------------------------------------- CPU: probe nets
@pytest.mark.parametrize("case_id", probes.CASE_IDS)
def test_probe_nets_are_tf32_exact(case_id, monkeypatch):
    """What the bf16 path stores bf16-exact the TF32 path stores TF32-exact: rerun the reference's checks with TF32 instead."""
    checked = []

    def assert_tf32_exact(name, a):
        f = np.asarray(a, dtype=np.float32)
        assert np.array_equal(f.astype(np.float64), a), f"{name}: not representable in f32"
        assert np.array_equal(tf32_round(f), f), f"{name}: not representable in TF32"
        checked.append(name)

    monkeypatch.setattr(probes, "assert_bf16_exact", assert_tf32_exact)
    b = probes.build(probes.BY_ID[case_id])
    probes.reference(b.net, b.planes, check=True)
    assert "input planes" in checked and "first conv output" in checked
    for wt, _ in [b.net.fc1, b.net.fc2] + ([b.net.policy_conv2] if b.net.policy_conv2 is not None else []):
        assert_tf32_exact("head weights", wt)


def test_precision_3_is_rejected_with_a_message():
    spec = netgen.game_spec("go-9")
    onnx_bytes = netgen.build_onnx(spec, 1, 16, seed=2)
    with pytest.raises(KzbError, match=r"precision must be 0 \(fp32\), 1 \(bf16\) or 2 \(tf32\)"):
        B200Network(mapper_for(spec), onnx_bytes, 4, precision=3)


def test_tf32_without_a_device_fails_like_the_others():
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    spec = netgen.game_spec("go-9")
    onnx_bytes = netgen.build_onnx(spec, 1, 16, seed=2)
    for precision in (0, 1, TF32):
        with pytest.raises(KzbError, match="no CUDA device"):
            B200Network(mapper_for(spec), onnx_bytes, 4, precision=precision)


# ----------------------------------------------------------------------------------------------------------- GPU: probe nets
TF32_CASES = [c.id for c in probes.CASES if PRECISION_BF16 in c.precisions]
SWITCHES = ((), probes.V(KZB_PDL="0"), probes.V(KZB_CONV_SPLIT="0"))


@pytest.mark.gpu
@pytest.mark.parametrize("case_id", TF32_CASES)
def test_tf32_equals_float64_reference(case_id, monkeypatch, capsys):
    """Scalars, logits and moves_left bit-identical to the float64 reference, with and without PDL and the channel split; the
    packed decode within the bounds of test_exact_probe_nets."""
    case = probes.BY_ID[case_id]
    stats = []
    for env in SWITCHES:
        probes.run_gpu(case, TF32, env, monkeypatch, stats)
    with capsys.disabled():
        print(f"\n{case_id} tf32: largest decode error / bound {max(stats):.3f}")


@pytest.mark.gpu
def test_tf32_rejects_boards_wider_than_255_squares():
    spec = netgen.game_spec("go-256")
    onnx_bytes = netgen.build_onnx(spec, 1, 8, seed=3)
    with pytest.raises(KzbError, match="precision=fp32"):
        B200Network(mapper_for(spec), onnx_bytes, 1, precision=TF32)


@pytest.mark.gpu
@pytest.mark.parametrize("case_id", ["chess-c40-d1-b3", "ataxx-5", "go-9-hs33"])
def test_tf32_raw_weights_equal_the_onnx_net(case_id):
    case = probes.BY_ID[case_id]
    b = probes.build(case)
    model = probes.onnx_bytes(b.net, b.spec, case.depth, case.channels, case.hc, case.hs, case.q)
    outs = []
    for weights in (probes.raw_weights(b.net), model):
        with B200Network(b.mapper, weights, case.batch, precision=TF32) as net:
            outs.append(net.evaluate_planes(b.planes) + net.evaluate_packed(b.bits, b.scalars, b.mv_idx, b.mv_off))
    for x, y in zip(*outs):
        assert np.array_equal(x, y)


# ----------------------------------------------------------------------------------------------------------- GPU: random-init parity
def _check(tag, s, p, ref_s, ref_p, capsys, probs=None, ref_probs=None):
    scale = max(1.0, float(np.abs(ref_p).max()))
    err_p, err_s = float(np.abs(p - ref_p).max()), float(np.abs(s - ref_s).max())
    err_prob = float(np.abs(probs - ref_probs).max()) if probs is not None and probs.size else 0.0
    with capsys.disabled():
        print(f"\n[{tag} tf32] max |dlogit| {err_p:.5f}, max |dscalar| {err_s:.5f} (bar {TF32_TOL * scale:.5f}, logit scale {scale:.2f}); "
              f"max |dprob| {err_prob:.6f}")
    assert err_p <= TF32_TOL * scale
    assert err_s <= TF32_TOL * scale
    assert err_prob <= TF32_PROB_TOL
    return err_p


@pytest.mark.gpu
@pytest.mark.parametrize("name", NET_NAMES)
def test_tf32_golden_nets_vs_reference_pytorch(name, capsys):
    onnx_bytes, x, scalars, policy = load_net_fixture(name)
    spec = netgen.game_spec(FIXTURE_GAMES[name])
    with B200Network(mapper_for(spec), onnx_bytes, 8, precision=TF32) as net:
        info = net.info()
        assert info.precision == TF32 and info.conv_mode == 0
        s, p = net.evaluate_planes(x)
    _check(name, s, p, scalars, policy, capsys)


@pytest.mark.gpu
def test_tf32_chess_16x128_full_batch_1024(capsys):
    spec = netgen.game_spec("chess")
    onnx_bytes = netgen.build_onnx(spec, 16, 128, seed=0)
    n = 1024
    bits, scalars, mv_idx, mv_off = netgen.synthetic_positions(spec, n, seed=31)
    planes = _planes(spec, bits, scalars)
    ref_s, ref_p = OnnxOracle(onnx_bytes, conv_backend="torch").run(planes)
    ref_values, ref_probs = oracle.decode_output(ref_s, ref_p, mv_idx, mv_off)
    with B200Network(mapper_for(spec), onnx_bytes, n, precision=TF32) as net:
        # an 8x8 net takes the row path: encode, 2 * depth + 1 tower convs, policy conv1, scalar conv, policy conv2, tail
        assert net.info().conv_mode == 0 and net.launches_per_eval() == 1 + (2 * 16 + 1) + 3 + 1
        v1, p1 = net.evaluate_packed(bits, scalars, mv_idx, mv_off)  # captures the full-batch graph
        v2, p2 = net.evaluate_packed(bits, scalars, mv_idx, mv_off)  # replays it
        s, p = net.evaluate_planes(planes)
    assert np.array_equal(v1, v2) and np.array_equal(p1, p2)
    _check("chess 16x128 n=1024", s, p, ref_s, ref_p, capsys, p1, ref_probs)
    assert np.abs(v1[:, 1:] - ref_values[:, 1:]).max() <= TF32_PROB_TOL


def _go_case(game, depth, ch, n_small, n_full, capsys):
    spec = netgen.game_spec(game)
    bits, scalars, mv_idx, mv_off = netgen.synthetic_positions(spec, n_small, seed=33)
    planes = _planes(spec, bits, scalars)
    onnx_bytes = netgen.build_onnx(spec, depth, ch, seed=0)
    ref_s, ref_p = OnnxOracle(onnx_bytes, conv_backend="torch").run(planes)
    ref_values, ref_probs = oracle.decode_output(ref_s, ref_p, mv_idx, mv_off)
    with B200Network(mapper_for(spec), onnx_bytes, n_small, precision=TF32) as net:
        assert net.info().conv_mode == 0
        values, probs = net.evaluate_packed(bits, scalars, mv_idx, mv_off)
        s, p = net.evaluate_planes(planes)
    err = _check(f"{game} {depth}x{ch} n={n_small}", s, p, ref_s, ref_p, capsys, probs, ref_probs)
    # the same boards repeated up to a full batch: every copy reproduces the oracle-checked rows bit for bit
    reps = n_full // n_small
    counts = np.diff(mv_off.astype(np.int64))
    big_off = np.zeros(n_full + 1, np.uint32)
    big_off[1:] = np.cumsum(np.tile(counts, reps))
    with B200Network(mapper_for(spec), onnx_bytes, n_full, precision=TF32) as net:
        bv, bp = net.evaluate_packed(np.tile(bits, (reps, 1)), np.tile(scalars, (reps, 1)), np.tile(mv_idx, reps), big_off)
    assert np.array_equal(bv, np.tile(values, (reps, 1)))
    assert np.array_equal(bp, np.tile(probs, reps))
    return onnx_bytes, planes, ref_p, err


@pytest.mark.gpu
def test_tf32_go9_20x256_vs_oracle_and_batch_4096(capsys):
    _go_case("go-9", 20, 256, 64, 4096, capsys)


@pytest.mark.gpu
def test_tf32_go19_40x256_vs_oracle_and_batch_8192(capsys):
    onnx_bytes, planes, ref_p, err = _go_case("go-19", 40, 256, 4, 8192, capsys)
    spec = netgen.game_spec("go-19")
    with B200Network(mapper_for(spec), onnx_bytes, 4, precision=PRECISION_BF16) as net:
        _, p = net.evaluate_planes(planes)
    err_bf16 = float(np.abs(p - ref_p).max())
    with capsys.disabled():
        print(f"\n[go-19 40x256] max |dlogit| TF32 {err:.5f}, bf16 {err_bf16:.5f}")
    assert err < 0.5 * err_bf16  # a "TF32" path that really rounds to bf16 would not get there


# ----------------------------------------------------------------------------------------------------------- GPU: path properties
@pytest.mark.gpu
@pytest.mark.parametrize("game", ["chess", "go-9"])
def test_tf32_rows_independent_of_batch(game):
    spec = netgen.game_spec(game)
    onnx_bytes = netgen.build_onnx(spec, 2, 32, seed=12)
    bits, scalars, mv_idx, mv_off = netgen.synthetic_positions(spec, 37, seed=13)
    with B200Network(mapper_for(spec), onnx_bytes, 64, precision=TF32) as net:
        v_all, p_all = net.evaluate_packed(bits, scalars, mv_idx, mv_off)
        for i in [0, 5, 36]:
            sl = slice(int(mv_off[i]), int(mv_off[i + 1]))
            v1, p1 = net.evaluate_packed(bits[i:i + 1], scalars[i:i + 1], mv_idx[sl], np.array([0, sl.stop - sl.start], np.uint32))
            assert np.array_equal(v1[0], v_all[i])
            assert np.array_equal(p1, p_all[sl])


@pytest.mark.gpu
@pytest.mark.parametrize("game", ["chess", "ataxx-7", "go-9"])
def test_tf32_packed_equals_planes_plus_decode(game):
    """evaluate_packed (fused decode, CUDA graph) agrees with evaluate_planes followed by the reference decode."""
    spec = netgen.game_spec(game)
    onnx_bytes = netgen.build_onnx(spec, 3, 64, seed=21)
    bits, scalars, mv_idx, mv_off = netgen.synthetic_positions(spec, 24, seed=22)
    with B200Network(mapper_for(spec), onnx_bytes, 24, precision=TF32) as net:
        values, probs = net.evaluate_packed(bits, scalars, mv_idx, mv_off)
        s, p = net.evaluate_planes(_planes(spec, bits, scalars))
    ref_values, ref_probs = oracle.decode_output(s, p, mv_idx, mv_off)
    assert np.array_equal(values[:, 4], s[:, 4])
    assert np.abs(values - ref_values).max() <= 1e-6
    assert np.abs(probs - ref_probs).max() <= 1e-6


@pytest.mark.gpu
@pytest.mark.parametrize("game", ["chess", "go-9"])
def test_tf32_nan_inputs_are_reported_not_emitted(game):
    spec = netgen.game_spec(game)
    onnx_bytes = netgen.build_onnx(spec, 2, 64, seed=61)
    bits, scalars, mv_idx, mv_off = netgen.synthetic_positions(spec, 9, seed=62)
    bad = scalars.copy()
    bad[4, 0] = np.nan
    with B200Network(mapper_for(spec), onnx_bytes, 16, precision=TF32) as net:
        with pytest.raises(KzbError, match="strictly positive"):
            net.evaluate_packed(bits, bad, mv_idx, mv_off)
        v, p = net.evaluate_packed(bits, scalars, mv_idx, mv_off)  # the handle stays usable
        assert np.isfinite(v).all() and np.isfinite(p).all()


# ----------------------------------------------------------------------------------------------------------- GPU: self-play
@pytest.mark.gpu
def test_tf32_selfplay_go9_games_replay_under_the_oracle_rules(tmp_path):
    from kzero_b200 import selfplay
    from test_selfplay_records import replay_under_oracle_rules

    onnx_bytes = netgen.build_onnx(netgen.game_spec("go-9"), 2, 32, seed=41)
    prefix = str(tmp_path / "games_0")
    cfg = selfplay.default_config(game=selfplay.GAME_GO9, visits=40, search_batch=8, gpu_batch=64, cpu_threads=2, gpu_threads=2, max_games=6,
                                  max_game_length=30, duration_s=60.0, output_prefix=prefix, seed=9)
    r = selfplay.run(onnx_bytes, cfg, precision=TF32)
    assert r.games_written > 0 and r.real_evals > 0 and r.batches > 0
    assert replay_under_oracle_rules(prefix, "go-9", "Go9") >= 40


@pytest.mark.gpu
def test_tf32_selfplay_session_go9_passes_the_precision_through(tmp_path):
    """kzb_selfplay_session_run with precision TF32: two generations, each file replays under the oracle rules."""
    from kzero_b200 import selfplay
    from test_selfplay_records import replay_under_oracle_rules

    onnx_bytes = netgen.build_onnx(netgen.game_spec("go-9"), 2, 32, seed=42)
    with selfplay.Session(selfplay.GAME_GO9) as session:
        for gen in range(2):
            prefix = str(tmp_path / f"games_{gen}")
            cfg = selfplay.default_config(game=selfplay.GAME_GO9, visits=40, search_batch=8, gpu_batch=64, cpu_threads=2, gpu_threads=1,
                                          max_games=4, max_game_length=30, duration_s=60.0, output_prefix=prefix, seed=11)
            r = session.run(onnx_bytes, cfg, precision=TF32)
            assert r.games_written > 0 and r.real_evals > 0
            assert replay_under_oracle_rules(prefix, "go-9", "Go9") > 0
