"""Towers and policy conv1 wider than 256 channels (up to 1024), in bf16, TF32 and fp32.

On the tensor cores a layer wider than 256 channels runs in slices of at most 256 output channels (conv_i2c.cu), padded to a
multiple of 64, and small batches double the number of slices when the halved slices are still whole 32-channel chunks
(executor.cu).  The exact-arithmetic probe nets of test_exact_probe_nets.py prove each slicing bit for bit:

  go-9-c320-d1-b7      base split 2 (slices of 160); a small batch, but 4 x 80 is not allowed
  go-9-c512-d1-b7      base split 2, doubled to 4 slices of 128 at this batch
  go-19-c384-d1-b40    slices of 192 on a non-8x8 board
  chess-c512-d1-b5     the 8x8 row path (no tower8k / heads8 at this width) plus the tail kernel at 512 channels
  chess-c384-d2-b1024  more pair tiles than SM pairs: base split only, several waves
  raw-19x9-c288        a width that is not a multiple of 64 (padded to 320)
  chess-c128-n1-384    policy conv1 wider than 256 behind a narrow tower (tower8k, then conv_i2c for policy conv1)
  att-q64-c384         the attention head's f32-output convs reading a 384-channel input (a longer K loop only)
  go-9-c1024-d1-b3     the widest net: base split 4, doubled to 8 slices of 128

CPU: the probe preconditions (bf16- and TF32-exact, exact f32 sums) and the f32 oracle against the float64 reference.
GPU: the probe nets bit for bit in every precision and under KZB_PDL=0 / KZB_CONV_SPLIT=0, the launch count of the 256-wide net,
raw-weight and ONNX creation, rows independent of batch and split, random-init parity at size, and the limits' messages.
"""
import numpy as np
import pytest

import oracle
import test_exact_probe_nets as probes
from oracle.graph_exec import OnnxOracle
from test_tf32 import TF32_TOL, tf32_round
from kzero_b200 import netgen
from kzero_b200.network import B200Network, KzbError, PRECISION_BF16, PRECISION_FP32, PRECISION_TF32, mapper_for

BF16, TF32, FP32 = PRECISION_BF16, PRECISION_TF32, PRECISION_FP32
BF16_TOL = 2e-2  # logits: BF16_TOL * max(1, max |logit|)
Case = probes.Case
GO = probes.GO

# `launches`: bf16 launches_per_eval, the count of the same net at 256 channels
WIDE = [
    Case("go-9-c320-d1-b7", game="go-9", channels=320, depth=1, batch=7, launches=GO(1)),
    Case("go-9-c512-d1-b7", game="go-9", channels=512, depth=1, batch=7, launches=GO(1)),
    Case("go-19-c384-d1-b40", game="go-19", channels=384, depth=1, batch=40, launches=GO(1)),
    Case("chess-c512-d1-b5", channels=512, depth=1, batch=5, launches=GO(1)),
    Case("chess-c384-d2-b1024", channels=384, depth=2, batch=1024, launches=GO(2)),
    Case("raw-19x9-c288", game=None, board=(19, 9), channels=288, depth=1, batch=5, launches=GO(1)),
    Case("chess-c128-n1-384", channels=128, n1=384, batch=5, launches=probes.TAIL_8X8),
    Case("att-q64-c384", game="chess-att", channels=384, q=64, batch=5, launches=1 + 3 + 1 + 2 + 1),  # + scalar conv, 2 attention convs
    Case("go-9-c1024-d1-b3", game="go-9", channels=1024, depth=1, batch=3, launches=GO(1)),
]
WIDE_IDS = [c.id for c in WIDE]
BY_ID = {c.id: c for c in WIDE}
assert not set(WIDE_IDS) & set(probes.CASE_IDS)
SWITCHES = ((), probes.V(KZB_PDL="0"), probes.V(KZB_CONV_SPLIT="0"))


# ----------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("case_id", WIDE_IDS)
def test_wide_probe_preconditions_hold(case_id, monkeypatch):
    """Every wide probe net is exact in bf16 and in TF32 (reference(check=True)), and informative."""
    case = BY_ID[case_id]
    b = probes.build(case)
    probes.reference(b.net, b.planes, check=True)
    x = probes.conv64(b.planes, *b.net.first)
    assert (x != 0).mean() > 0.2

    def assert_tf32_exact(name, a):
        f = np.asarray(a, dtype=np.float32)
        assert np.array_equal(f.astype(np.float64), a), f"{name}: not representable in f32"
        assert np.array_equal(tf32_round(f), f), f"{name}: not representable in TF32"

    monkeypatch.setattr(probes, "assert_bf16_exact", assert_tf32_exact)
    probes.reference(b.net, b.planes, check=True)


@pytest.mark.parametrize("case_id", ["go-9-c320-d1-b7", "att-q64-c384"])
def test_wide_oracle_equals_float64_reference(case_id):
    case = BY_ID[case_id]
    b = probes.build(case)
    ref_s, ref_p = probes.reference(b.net, b.planes, check=True)
    model = probes.onnx_bytes(b.net, b.spec, case.depth, case.channels, case.hc, case.hs, case.q)
    s, p = OnnxOracle(model).run(b.planes)
    assert np.array_equal(s, ref_s.astype(np.float32))
    assert np.array_equal(p, ref_p.astype(np.float32))


# ----------------------------------------------------------------------------------------------------------- GPU: probe nets
@pytest.mark.gpu
@pytest.mark.parametrize("case_id", WIDE_IDS)
def test_wide_equals_float64_reference(case_id, monkeypatch, capsys):
    """Scalars, logits and moves_left bit-identical to the float64 reference in bf16, TF32 (default, KZB_PDL=0, KZB_CONV_SPLIT=0)
    and fp32; the packed decode within the bounds of test_exact_probe_nets; the bf16 launch count that of the 256-wide net."""
    case = BY_ID[case_id]
    stats = []
    for precision in (BF16, TF32):
        for env in SWITCHES:
            probes.run_gpu(case, precision, env, monkeypatch, stats)
    probes.run_gpu(case, FP32, (), monkeypatch, stats)
    with capsys.disabled():
        print(f"\n{case_id}: largest decode error / bound {max(stats):.3f}")


@pytest.mark.gpu
@pytest.mark.parametrize("case_id", ["go-9-c320-d1-b7", "chess-c512-d1-b5"])
def test_wide_raw_weights_equal_the_onnx_net(case_id):
    """kzb_net_create and kzb_net_create_from_onnx build bit-identical wide networks, in every precision."""
    case = BY_ID[case_id]
    b = probes.build(case)
    model = probes.onnx_bytes(b.net, b.spec, case.depth, case.channels, case.hc, case.hs, case.q)
    for precision in (BF16, TF32, FP32):
        outs = []
        for weights in (probes.raw_weights(b.net), model):
            with B200Network(b.mapper, weights, case.batch, precision=precision) as net:
                outs.append(net.evaluate_planes(b.planes) + net.evaluate_packed(b.bits, b.scalars, b.mv_idx, b.mv_off))
        for x, y in zip(*outs):
            assert np.array_equal(x, y)


# ----------------------------------------------------------------------------------------------------------- GPU: random-init nets
def _tiled(bits, scalars, mv_idx, mv_off, reps):
    counts = np.diff(mv_off.astype(np.int64))
    off = np.zeros(len(counts) * reps + 1, np.uint32)
    off[1:] = np.cumsum(np.tile(counts, reps))
    return np.tile(bits, (reps, 1)), np.tile(scalars, (reps, 1)), np.tile(mv_idx, reps), off


@pytest.mark.gpu
@pytest.mark.parametrize("precision", [BF16, TF32])
def test_wide_rows_independent_of_batch_and_split(precision, monkeypatch):
    """go-19 at 384 channels: batch 4 runs 4 slices of 96, batches 40 and 1500 two slices of 192 (KZB_CONV_SPLIT=0: two at every
    batch); every copy of a board's row is bit-identical across all of them."""
    spec = netgen.game_spec("go-19")
    onnx_bytes = netgen.build_onnx(spec, 2, 384, seed=71)
    base = netgen.synthetic_positions(spec, 4, seed=72)
    results = []
    for env in ((), probes.V(KZB_CONV_SPLIT="0")):
        for key, val in env:
            monkeypatch.setenv(key, val)
        try:
            with B200Network(mapper_for(spec), onnx_bytes, 1500, precision=precision) as net:
                for n in (4, 40, 1500):
                    values, probs = net.evaluate_packed(*_tiled(*base, n // 4))
                    results.append((f"{dict(env) or 'default'} batch {n}", values, probs))
        finally:
            for key, _ in env:
                monkeypatch.delenv(key)
    ref_tag, ref_v, ref_p = results[0]
    for tag, values, probs in results:
        reps = values.shape[0] // 4
        assert np.array_equal(values, np.tile(ref_v, (reps, 1))), f"{tag} differs from {ref_tag}"
        assert np.array_equal(probs, np.tile(ref_p, reps)), f"{tag} differs from {ref_tag}"


@pytest.mark.gpu
@pytest.mark.parametrize("game,depth,ch,n", [("go-19", 20, 384, 4), ("chess", 10, 512, 16)])
def test_wide_random_init_vs_oracle(game, depth, ch, n, capsys):
    """Random-init nets at size against the f32 oracle: bf16 logits within 2e-2 * max(1, max |logit|), TF32 logits and raw scalars
    within 4e-3 * max(1, max |logit|)."""
    spec = netgen.game_spec(game)
    onnx_bytes = netgen.build_onnx(spec, depth, ch, seed=0)
    bits, scalars, _, _ = netgen.synthetic_positions(spec, n, seed=73)
    planes = oracle.expand_planes(bits, scalars, (spec.bool_channels, spec.board_size, spec.board_size), spec.scalar_channels)
    ref_s, ref_p = OnnxOracle(onnx_bytes, conv_backend="torch").run(planes)
    scale = max(1.0, float(np.abs(ref_p).max()))
    for precision, tol, tag in ((BF16, BF16_TOL, "bf16"), (TF32, TF32_TOL, "tf32")):
        with B200Network(mapper_for(spec), onnx_bytes, n, precision=precision) as net:
            assert net.info().channels == ch
            s, p = net.evaluate_planes(planes)
        err_p, err_s = float(np.abs(p - ref_p).max()), float(np.abs(s - ref_s).max())
        with capsys.disabled():
            print(f"\n[{game} {depth}x{ch} n={n} {tag}] max |dlogit| {err_p:.5f}, max |dscalar| {err_s:.5f} (bar {tol * scale:.5f})")
        assert err_p <= tol * scale
        if precision == TF32:
            assert err_s <= tol * scale


# ----------------------------------------------------------------------------------------------------------- GPU: the limits
@pytest.mark.gpu
@pytest.mark.parametrize("case,message", [
    (Case("go-9-c1025", game="go-9", channels=1025, depth=0, batch=1), r"a tower of 1025 channels is not supported \(at most 1024\)"),
    (Case("go-9-n1-1025", game="go-9", channels=32, n1=1025, batch=1),
     r"policy conv1 with 1025 output channels is not supported \(at most 1024\)"),
    (Case("raw-9x9-n2-257", game=None, board=(9, 9), channels=32, n2=257, batch=1),
     r"policy conv2 with 257 output channels is not supported \(at most 256\)"),
], ids=lambda v: v.id if isinstance(v, Case) else "")
def test_wider_than_the_limits_is_rejected(case, message):
    b = probes.build(case)
    for precision in (BF16, TF32, FP32):
        with pytest.raises(KzbError, match=message):
            B200Network(b.mapper, probes.raw_weights(b.net), 1, precision=precision)
