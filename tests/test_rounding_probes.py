"""Rounding on store, bf16 and TF32: probe nets whose stored values are mostly not representable, bit for bit against a float64
reference that rounds exactly what the path stores rounded.

The probe nets of test_exact_probe_nets.py store only values that are exact in bf16 and TF32, so no rounding ever changes one
there.  These nets are the same probe nets with the first conv's weights on the board planes and every tower and head bias
scaled by the precision's scale (bf16 255, TF32 257: both exact in their format, so the host keeps the scaled weights), and the
first conv's weights on the scalar planes scaled by 256.  Every value stays an integer (or on the 2^-5 / 2^-6 grid of the heads)
and every f32 sum stays exact, but the tower outputs reach 2^16, where most integers are neither bf16 nor TF32 values.

Every other board of a batch gets scalars 4 + u 2^-12 (u not a multiple of 16): off the bf16 grid (2^-5 in [4, 8)) and the TF32
grid (2^-8), so the encode kernels (encode_kc, encode_nhwc, nchw_to_kc, nchw_to_rows) must round them; once rounded they sit on
the 2^-8 grid, and times 256 the first conv's products are integers again.

The reference rounds, in the precision's format and with its rounding (bf16: to nearest even, as __float2bfloat16_rn;
TF32: to nearest, ties away from zero, as tf32_round in kernels.cuh):
  - the input planes;
  - the first conv's output and block conv1's output after the ReLU;
  - each block's output, once, from the f32 value x + relu(y);
  - policy conv1's output.
Biases, the scalar conv's output, policy conv2, the extra conv, the attention convs and the FC layers stay in f32.

CPU: the preconditions, a sizeable share of changed stores, exact ties in the tower stores (so that rounding to even, rounding
ties away and truncating all give different results), and a fault table: every wrong rounding changes the probe outputs.
GPU: scalars and logits bit for bit, the decode within its bounds, through evaluate_planes and evaluate_packed.
"""
import functools
from dataclasses import dataclass, replace
from typing import Callable

import numpy as np
import pytest

import test_exact_probe_nets as probes
import test_wide_towers as wide
from helpers import bf16_round
from test_tf32 import tf32_round
from kzero_b200.network import PRECISION_BF16, PRECISION_TF32

V = probes.V
NO_EMBED8, PDL0, SPLIT0 = V(KZB_NO_EMBED8="1"), V(KZB_PDL="0"), V(KZB_CONV_SPLIT="0")
SCALAR_SCALE = 256.0


@dataclass(frozen=True)
class Format:
    name: str
    precision: int
    round: Callable  # f32 array -> f32 array: what the path's stores do
    drop: int  # low f32 mantissa bits the format lacks
    tie: str  # "even" or "away": what the rounding does at an exact tie
    scale: float


FORMATS = {
    "bf16": Format("bf16", PRECISION_BF16, bf16_round, 16, "even", 255.0),
    "tf32": Format("tf32", PRECISION_TF32, tf32_round, 13, "away", 257.0),
}

# case id -> the switches run besides the default.  Together the bf16 cases cover every bf16 path: tower8k with heads8 (chess,
# ataxx-5 embedded, 9472 boards), the tail kernel with conv_i2c for the 1x1 convs (KZB_NO_HEADS8), conv_i2c for the 8x8
# tower (KZB_NO_TOWER8) and for a small board (KZB_NO_EMBED8), go with and without the doubled channel split, a non-square board,
# a layer in slices, and the attention head created through ONNX.
CASES = {
    "bf16": {
        "chess-c40-d1-b3": (probes.NO_HEADS8, probes.NO_TOWER8),
        "ataxx-5": (NO_EMBED8,),
        "chess-c32-d2-b9472": (),
        "go-9-c192-b7": (SPLIT0,),
        "raw-19x9": (),
        "raw-19x9-c288": (),
        "att-q16": (),
    },
    "tf32": {case_id: (PDL0, SPLIT0) for case_id in ("chess-c40-d1-b3", "go-9-c192-b7", "raw-19x9", "ataxx-5")},
}
PARAMS = [(f, c) for f in CASES for c in CASES[f]]
ALL_CASES = {**probes.BY_ID, **wide.BY_ID}

FAULTS = ["truncated", "other_tie", "rounded_before_residual_add", "unrounded_policy_conv1", "unrounded_input_scalars"]


def round_bits(a, drop, mode):
    """Finite f32 values cut to 24 - drop significant bits: "even" and "away" round to nearest (ties to even / away from zero),
    "truncate" rounds toward zero."""
    u = np.ascontiguousarray(a, dtype=np.float32).view(np.uint32).astype(np.uint64)
    half = np.uint64(1 << (drop - 1))
    if mode == "even":
        u = u + (half - np.uint64(1)) + ((u >> np.uint64(drop)) & np.uint64(1))
    elif mode == "away":
        u = u + half
    else:
        assert mode == "truncate"
    return (u & np.uint64(0xFFFFFFFF ^ ((1 << drop) - 1))).astype(np.uint32).view(np.float32)


def is_tie(f, drop):
    """f32 values exactly halfway between two neighbours of the format."""
    u = np.ascontiguousarray(f, dtype=np.float32).view(np.uint32)
    return (u & np.uint32((1 << drop) - 1)) == np.uint32(1 << (drop - 1))


@functools.lru_cache(maxsize=None)
def rounding_probe(fmt_name, case_id) -> probes.Built:
    """The probe net of case_id scaled for the format (module docstring) and its inputs, every other board with off-grid scalars."""
    fmt = FORMATS[fmt_name]
    b = probes.build(ALL_CASES[case_id])
    net, k, cs = b.net, fmt.scale, b.mapper.input_scalar_count

    def bias(wb):
        return None if wb is None else (wb[0], wb[1] * k)

    w0 = net.first[0] * k
    w0[:, :cs] = net.first[0][:, :cs] * SCALAR_SCALE
    att = None
    if net.att is not None:
        # The attention dot product multiplies two conv outputs: over a tower of 2^16 integers it cannot stay exact in f32.  Its
        # convs keep their biases only; the tower's rounding reaches the outputs through the scalar head.
        (bw, bb), (uw, ub), q = net.att
        att = ((0 * bw, bb), (0 * uw, ub), q)
    scaled = replace(net, first=(w0, net.first[1] * k), blocks=[bias(wb) for wb in net.blocks], scalar_conv=bias(net.scalar_conv),
                     fc1=bias(net.fc1), fc2=bias(net.fc2), policy_conv1=bias(net.policy_conv1), policy_conv2=bias(net.policy_conv2),
                     extra_conv=bias(net.extra_conv), extra_fc=bias(net.extra_fc), att=att)
    rng = np.random.default_rng([ord(ch) for ch in case_id + fmt_name])
    scalars = b.scalars.copy()
    off = scalars[::2]
    u = 16 * rng.integers(0, 1 << 10, size=off.shape) + rng.integers(1, 16, size=off.shape)
    scalars[::2] = (4 + u * 2.0 ** -12).astype(np.float32)
    planes = b.planes.copy()
    planes[:, :cs] = scalars[:, :, None, None]
    return replace(b, net=scaled, scalars=scalars, planes=planes)


def reference_stores(net, planes, fmt: Format, fault=None):
    """float64 forward pass with the stores of the path in fmt -> (scalars, logits, [stores, changed by the rounding, exact ties]
    over the tower and policy conv1 stores).  Without a fault it asserts that every stored value is f32-exact before it is rounded
    and that every sum is exact in f32.  fault: one of FAULTS, the wrong rounding to emulate."""
    n = planes.shape[0]
    check = fault is None
    rnd = fmt.round
    if fault == "truncated":
        rnd = functools.partial(round_bits, drop=fmt.drop, mode="truncate")
    elif fault == "other_tie":
        rnd = functools.partial(round_bits, drop=fmt.drop, mode="away" if fmt.tie == "even" else "even")
    counts = np.zeros(3, np.int64)

    def store(name, a, counted=True):
        f = a.astype(np.float32)
        if check:
            assert np.array_equal(f.astype(np.float64), a), f"{name}: not f32-exact before rounding"
        r = rnd(f).astype(np.float64)
        if counted:
            counts[:] += (a.size, int((r != a).sum()), int(is_tie(f, fmt.drop).sum()))
        return r

    def conv(name, xin, wb):
        w, b = wb
        if check:
            probes.assert_exact_sum(name, xin, w, b, probes.conv64(np.abs(xin), np.abs(w), np.abs(b)))
        return probes.conv64(xin, w, b)

    def fc(name, xin, wb):
        w, b = wb
        if check:
            probes.assert_exact_sum(name, xin, w, b, np.abs(xin) @ np.abs(w).T + np.abs(b))
        return xin @ w.T + b

    x = planes.astype(np.float64)
    if fault != "unrounded_input_scalars":
        x = store("input planes", x, counted=False)
    x = store("first conv", conv("first conv", x, net.first))
    for d in range(len(net.blocks) // 2):
        t = store(f"block{d} conv1", probes.relu(conv(f"block{d} conv1", x, net.blocks[2 * d])))
        y = probes.relu(conv(f"block{d} conv2", t, net.blocks[2 * d + 1]))
        if fault == "rounded_before_residual_add":
            y = store(f"block{d} conv2", y, counted=False)
        x = store(f"block{d} output", x + y)
    s1 = probes.relu(conv("scalar conv", x, net.scalar_conv))
    scalars = fc("fc2", probes.relu(fc("fc1", s1.reshape(n, -1), net.fc1)), net.fc2)
    if net.att is not None:
        (bulk_w, under_w, q) = net.att
        logits = probes.attention_logits(conv("attention bulk conv", x, bulk_w), conv("attention under conv", x[:, :, 7:8, :], under_w),
                                         q, check)
    else:
        h1 = probes.relu(conv("policy conv1", x, net.policy_conv1))
        h1 = h1 if fault == "unrounded_policy_conv1" else store("policy conv1", h1)
        pm = conv("policy conv2", h1, net.policy_conv2).reshape(n, -1)
        src = net.policy_src
        logits = np.where(src >= 0, pm[:, np.maximum(src, 0)], 0.0)
        if net.extra_conv is not None:
            e = conv("extra conv", x, net.extra_conv)
            logits = np.where(src == -2, fc("extra fc", e.reshape(n, -1), net.extra_fc), logits)
    if check:
        assert np.array_equal(scalars.astype(np.float32), scalars) and np.array_equal(logits.astype(np.float32), logits)
    return scalars, logits, counts


@functools.lru_cache(maxsize=4)
def expected(fmt_name, case_id):
    b = rounding_probe(fmt_name, case_id)
    s, p, _ = reference_stores(b.net, b.planes, FORMATS[fmt_name])
    return probes.expected(s, p, b.mv_idx, b.mv_off)


# ----------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("fmt_name", FORMATS)
def test_round_bits_is_the_rounding_of_the_format(fmt_name):
    """round_bits with the format's tie rule is the rounding the reference applies, on every finite bit pattern class."""
    fmt = FORMATS[fmt_name]
    u = np.random.default_rng(7).integers(0, 1 << 32, size=100000, dtype=np.uint64).astype(np.uint32)
    u = u[(u & 0x7F800000) < 0x7F000000]  # finite and clear of the overflow to Inf
    u = np.concatenate([u, (u & ~np.uint32((1 << fmt.drop) - 1)) | np.uint32(1 << (fmt.drop - 1))])  # and as many exact ties
    f = u.view(np.float32)
    assert np.array_equal(round_bits(f, fmt.drop, fmt.tie).view(np.uint32), fmt.round(f).view(np.uint32))
    ties = is_tie(f, fmt.drop)
    assert ties.sum() >= u.size // 2
    results = [round_bits(f[ties], fmt.drop, m).view(np.uint32) for m in ("even", "away", "truncate")]
    assert all((a != b).any() for i, a in enumerate(results) for b in results[i + 1:])


@pytest.mark.parametrize("fmt_name,case_id", PARAMS)
def test_rounding_probe_nets_are_exact_and_exercise_the_rounding(fmt_name, case_id):
    fmt = FORMATS[fmt_name]
    b = rounding_probe(fmt_name, case_id)
    _, _, (stores, changed, ties) = reference_stores(b.net, b.planes, fmt)
    assert changed > 0.1 * stores, f"the rounding changes only {changed} of {stores} stores"
    assert ties > 0, "no exact ties among the stores: rounding to even and ties away would agree"
    # the host rounding keeps the conv weights (the biases are added in f32 by the epilogues and are not rounded)
    net = b.net
    w = [net.first[0], net.scalar_conv[0]] + [wb[0] for wb in net.blocks]
    w += [net.policy_conv1[0], net.policy_conv2[0]] if net.att is None else [net.att[0][0], net.att[1][0]]
    assert all(np.array_equal(fmt.round(np.float32(a)), np.float32(a)) for a in w)
    # the scalars of every other board are off the grid of both formats
    off = b.scalars[::2]
    assert (bf16_round(off) != off).all() and (tf32_round(off) != off).all()


@pytest.mark.parametrize("fmt_name", FORMATS)
def test_rounding_faults_change_the_probe_outputs(fmt_name, capsys):
    """Each wrong rounding changes at least one logit or scalar of chess-c40-d1-b3: truncation, the other tie rule, rounding
    relu(conv2) before the residual add, leaving policy conv1 or the input scalars unrounded."""
    fmt = FORMATS[fmt_name]
    b = rounding_probe(fmt_name, "chess-c40-d1-b3")
    s0, p0, _ = reference_stores(b.net, b.planes, fmt)
    rows = []
    for fault in FAULTS:
        s1, p1, _ = reference_stores(b.net, b.planes, fmt, fault=fault)
        changed = int((s0 != s1).sum() + (p0 != p1).sum())
        assert changed > 0, f"{fmt_name} {fault} leaves the outputs unchanged"
        rows.append(f"{fmt_name} {fault:28s} {changed:6d} outputs changed")
    with capsys.disabled():
        print("\n" + "\n".join(rows))


# ----------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("fmt_name,case_id", PARAMS)
def test_stores_are_rounded_like_the_reference(fmt_name, case_id, monkeypatch):
    """Scalars, logits and moves_left bit-identical to the reference that rounds every store of the path, through
    evaluate_planes and evaluate_packed, by default and under the case's switches; the decode within its bounds."""
    fmt = FORMATS[fmt_name]
    case = ALL_CASES[case_id]
    b = rounding_probe(fmt_name, case_id)
    ref = expected(fmt_name, case_id)
    for env in ((),) + CASES[fmt_name][case_id]:
        probes.run_gpu(case, fmt.precision, env, monkeypatch, [], b=b, ref=ref)
