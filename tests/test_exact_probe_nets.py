"""Every kernel path against a float64 reference, bit for bit, on probe networks whose arithmetic is exact.

The parity tests in test_gpu_parity.py compare random-init networks with the f32 oracle within a tolerance (2e-2 on bf16 logits).
A kernel that reads one tap from the wrong place or one board's residual from its neighbour can stay inside that bar
(test_faults_change_the_probe_outputs prints by how much each such fault moves a default net).  The probe networks here are built
so that every correct implementation returns the same numbers whatever its summation order, rounding points or MMA scheme:

  - tower convs have weights in {-1, 0, +1}, k nonzeros per output channel, spread so that every (tap, input channel) slot of a
    layer is used; biases are integers, calibrated on the test batch (median pre-activation, lowered so that nothing stored
    exceeds 256; the residual branch is capped at (256 - max of the input layer) / depth);
  - the head layers that produce logits and scalars have weights +-2^-5 (policy conv2) and +-2^-6 (fc2, extra fc);
  - the final BN is the identity; inputs are 0/1 bits and small integer scalars, half of each batch dense random bits.

`reference(..., check=True)` asserts the two preconditions that make this exact, in float64: (a) every tensor any path may store
in bf16 satisfies x == bf16(x); (b) every accumulation is exact in f32 (all terms on a grid 2^-q with sum |terms| < 2^(24-q)).
A net that violates them fails there; it never quietly weakens the comparison.

Then evaluate_planes must return the reference's scalars and logits exactly, in bf16 and fp32 and under every kernel switch.
evaluate_packed returns moves_left exactly; value, WDL and probabilities go through expf / tanhf and are held to a bound built
from CUDA's documented errors (2 ulp for expf and tanhf, IEEE division, n 2^-24 relative for an n-term sum of positive terms).

The batches reach the sizes where the persistent kernels loop: tower8k up to 16 units per CTA (9,472 boards), heads8 up to 32
tiles per CTA, conv_i2c over many waves of pair tiles; test_rows_past_the_batch_do_not_leak leaves NaN rows behind the batch.
The values these nets store are exact in bf16 and TF32, so the rounding on store is checked by test_rounding_probes.py.
"""
import functools
from dataclasses import dataclass
from typing import Optional, Tuple

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import oracle
from helpers import bf16_round
from oracle.graph_exec import OnnxOracle
from kzero_b200 import mapping, netgen
from kzero_b200.network import B200Network, KzbError, Mapper, PRECISION_BF16, PRECISION_FP32, PRECISION_TF32, RawWeights

BF16, FP32, TF32 = PRECISION_BF16, PRECISION_FP32, PRECISION_TF32
PRECISION_NAMES = {BF16: "bf16", TF32: "tf32", FP32: "fp32"}
U = 2.0 ** -24  # unit roundoff of f32
BN_EPS = np.float32(1e-5)
IDENTITY_VAR = np.float32(1 - 1e-5)  # with eps: an f32 BatchNormalization that is exactly the identity


# ----------------------------------------------------------------------------------------------------------- the cases
@dataclass(frozen=True)
class Case:
    id: str
    game: Optional[str] = "chess"  # netgen game for inputs and policy layout; None: a raw board of `board`
    board: Optional[Tuple[int, int]] = None  # (h, w) of a raw board: 3 bool planes, 2 scalars
    channels: int = 32
    depth: int = 1
    batch: int = 3
    max_batch: int = 0  # 0: batch
    hc: int = 4
    hs: int = 32
    n1: int = 0  # policy conv1 width; 0: channels
    n2: int = 0  # policy conv2 width; 0: the game's
    q: int = 0  # attention query channels (chess-att, created from ONNX)
    variants: Tuple[Tuple[Tuple[str, str], ...], ...] = ()  # environment settings run besides the default
    precisions: Tuple[int, ...] = (BF16, FP32)
    launches: int = 0  # bf16 launches_per_eval with default settings; 0: not checked
    k: int = 9


V = lambda **env: tuple(sorted(env.items()))  # noqa: E731
NO_HEADS8, NO_TOWER8 = V(KZB_NO_HEADS8="1"), V(KZB_NO_TOWER8="1")
TAIL_8X8 = 6  # encode, tower8k, policy conv1, scalar conv, policy conv2, tail kernel
GO = lambda depth: 2 * depth + 6  # noqa: E731  encode, 2 depth + 1 tower convs, policy conv1, scalar conv, policy conv2, tail
PDL0, B_SLOTS2 = V(KZB_PDL="0"), V(KZB_B_SLOTS="2")

# The large batches below are chosen for a B200's 148 SMs (74 SM pairs), as are the unit and tile counts of the older cases.
# tower8k, uniform scheme (outside the balanced band of 6..8 boards per CTA): 4-board units, their count rounded up to even.
#   1186: 298 units, 2 to 3 per CTA;  4001: 1002 units, 6 to 7 per CTA, the last real unit holds 1 board, then a padding unit;
#   9469: 2368 units, 16 per CTA (kMaxLocalUnits), the last unit holds 1 board;  9472: the same, every unit full.
#   Depth 2: five layers, so every ready[] barrier changes phase at least 4 times.  heads8 at 9472: 4736 tiles, 32 per CTA.
# conv_i2c, 128-row tiles in pairs: go-19 b400 1129 tiles (565 pair tiles over 74 clusters); raw-19x9 b120 161 tiles, so the last
# pair's second CTA lies wholly past the batch; go-9 b116 74 tiles (37 pair tiles: the split doubles), b117 75 tiles (38: it does not).
LARGE = [
    Case("chess-c32-d2-b1186", channels=32, depth=2, batch=1186, max_batch=9472, launches=3),
    Case("chess-c32-d2-b4001", channels=32, depth=2, batch=4001, max_batch=9472, launches=3, variants=(PDL0, B_SLOTS2)),
    Case("chess-c32-d2-b9469", channels=32, depth=2, batch=9469, max_batch=9472, launches=3),
    Case("chess-c32-d2-b9472", channels=32, depth=2, batch=9472, launches=3, variants=(NO_HEADS8, PDL0, B_SLOTS2)),
    Case("chess-c96-d2-b3000", channels=96, depth=2, batch=3000, max_batch=9472, launches=3, variants=(NO_HEADS8,)),
    Case("ataxx-5-b4001", game="ataxx-5", channels=32, depth=2, batch=4001, launches=3, variants=(PDL0,)),
    Case("go-19-c64-b400", game="go-19", channels=64, depth=1, batch=400, launches=GO(1), variants=(PDL0,)),
    Case("raw-19x9-b120", game=None, board=(19, 9), channels=64, depth=1, batch=120, launches=GO(1)),
    *[Case(f"go-9-c192-b{n}", game="go-9", channels=192, depth=1, batch=n, launches=GO(1)) for n in (116, 117)],
]

CASES = [
    # ---- tower8k + heads8 (encode, tower8k, heads8: 3 launches)
    Case("chess-c8-d0-b1", channels=8, depth=0, batch=1, launches=3),
    Case("chess-c40-d1-b3", channels=40, depth=1, batch=3, launches=3, variants=(NO_HEADS8, NO_TOWER8)),
    Case("chess-c72-d3-b5", channels=72, depth=3, batch=5, launches=3),
    Case("chess-c128-d1-b9", channels=128, depth=1, batch=9, launches=3, variants=(NO_HEADS8,)),
    Case("chess-c8-d3-b9", channels=8, depth=3, batch=9, launches=3),
    Case("chess-c128-d0-b5", channels=128, depth=0, batch=5, launches=3),
    Case("chess-c40-d3-b1", channels=40, depth=3, batch=1, launches=3),
    Case("chess-c72-d0-b3", channels=72, depth=0, batch=3, launches=3, variants=(NO_TOWER8,)),
    Case("chess-16x128-b1024", channels=128, depth=16, batch=1024, launches=3, variants=(V(KZB_NO_BALANCE="1"),)),
    *[Case(f"chess-c64-b{n}", channels=64, depth=1, batch=n, launches=3) for n in (887, 888, 1184, 1185)],
    Case("chess-c64-max9472", channels=64, depth=1, batch=16, max_batch=9472, launches=3),
    Case("chess-c64-max9473", channels=64, depth=1, batch=16, max_batch=9473, launches=2 * 1 + 3),  # conv_i2c per layer, heads8
    Case("chess-hist-2", game="chess-hist-2", channels=64, depth=1, batch=5, launches=3),
    Case("chess-hist-4", game="chess-hist-4", channels=64, depth=1, batch=5, launches=3),
    *[Case(f"ataxx-{s}", game=f"ataxx-{s}", channels=32, depth=1, batch=5, launches=3) for s in (2, 3, 4, 5, 6)],
    Case("ataxx-7", game="ataxx-7", channels=32, depth=2, batch=5, launches=3, variants=(V(KZB_NO_EMBED8="1"), NO_HEADS8)),
    *[Case(f"raw-{h}x{w}", game=None, board=(h, w), channels=32, depth=2, batch=5, launches=3) for h, w in ((8, 5), (6, 8), (3, 7))],
    Case("heads8-hc1-hs1", channels=32, hc=1, hs=1, batch=5, launches=3),
    Case("heads8-hc15-hs32", channels=32, hc=15, hs=32, batch=5, launches=3),
    Case("heads8-n1-64-c128", channels=128, n1=64, batch=5, launches=3),
    Case("heads8-n2-128", channels=64, n2=128, batch=5, launches=3),
    Case("tail8-hs33", channels=32, hs=33, batch=5, launches=TAIL_8X8),
    Case("tail8-n1-192", channels=64, n1=192, batch=5, launches=TAIL_8X8),
    # ---- conv_i2c (tower and head form) + tail kernel (go: encode, 2 depth + 1 convs, 3 head convs, tail)
    Case("go-3-c64-b1", game="go-3", channels=64, depth=1, batch=1),
    Case("go-5-c96-b2", game="go-5", channels=96, depth=1, batch=2, variants=(V(KZB_PDL="0"),)),
    Case("go-9-c192-b7", game="go-9", channels=192, depth=1, batch=7, variants=(V(KZB_CONV_SPLIT="0"),)),
    Case("go-13-c256-b40", game="go-13", channels=256, depth=1, batch=40, launches=2 * 1 + 1 + 5),
    Case("go-19-c64-b40", game="go-19", channels=64, depth=2, batch=40, variants=(V(KZB_PDL="0"), V(KZB_CONV_SPLIT="0"))),
    *[Case(f"raw-{h}x{w}", game=None, board=(h, w), channels=64, depth=1, batch=5) for h, w in ((9, 7), (19, 9), (8, 10))],
    Case("chess-linear", channels=64, depth=2, batch=5, variants=(V(KZB_FORCE_LINEAR="1"),)),
    Case("chess-c136", channels=136, depth=1, batch=5),
    Case("chess-c256", channels=256, depth=1, batch=5),
    *[Case(f"go-9-hs{hs}", game="go-9", channels=64, hs=hs, batch=5) for hs in (33, 64, 128)],
    *[Case(f"go-19-hc{hc}", game="go-19", channels=64, hc=hc, batch=5) for hc in (1, 9, 15)],
    *[Case(f"att-q{q}", game="chess-att", channels=128 if q == 128 else 32, q=q, batch=5) for q in (16, 64, 128)],
    Case("go-256-fp32", game="go-256", channels=8, depth=1, batch=1, precisions=(FP32,)),
    *LARGE,
]
CASE_IDS = [c.id for c in CASES]
assert len(set(CASE_IDS)) == len(CASE_IDS)
BY_ID = {c.id: c for c in CASES}


# ----------------------------------------------------------------------------------------------------------- the nets
@dataclass
class Net:
    board: Tuple[int, int]
    first: tuple
    blocks: list
    scalar_conv: tuple
    fc1: tuple
    fc2: tuple
    policy_conv1: Optional[tuple]
    policy_conv2: Optional[tuple]
    policy_src: Optional[np.ndarray]  # [P]: channel * area + square, -1: zero logit, -2: the extra fc
    extra_conv: Optional[tuple] = None
    extra_fc: Optional[tuple] = None
    att: Optional[tuple] = None  # (bulk conv, under conv, q)
    final_affine: Optional[tuple] = None  # only the default (random-init) nets have one


def conv64(x, w, b=None, pad=None, circular=False):
    pad = w.shape[-1] // 2 if pad is None else pad
    t = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float64))
    if circular and pad:
        t, pad = F.pad(t, (pad,) * 4, mode="circular"), 0
    return F.conv2d(t, torch.from_numpy(np.ascontiguousarray(w, dtype=np.float64)),
                    None if b is None else torch.from_numpy(np.asarray(b, dtype=np.float64)), padding=pad).numpy()


def sparse_pm1(rng, cout, cin, ks, k, scale=1.0):
    """Weights in {-scale, 0, +scale}: k nonzeros per output channel (more when cout * k would leave a (tap, channel) slot
    unused), every slot used by some output channel."""
    slots = cin * max(ks, 1) ** 2  # ks 0: an FC layer [cout, cin]
    kk = min(slots, max(k, -(-slots // cout)))
    w = np.zeros((cout, slots))
    perm = rng.permutation(slots)
    for co in range(cout):
        w[co, perm[(co * kk + np.arange(kk)) % slots]] = rng.choice([-1.0, 1.0], kk) * scale
    return w.reshape(cout, cin, ks, ks) if ks else w


def calibrate(pre, cap, grid=1.0):
    """Per output channel: minus the median pre-activation on the grid, lowered so that the largest output stays <= cap."""
    v = np.moveaxis(pre, 1, 0).reshape(pre.shape[1], -1)
    b = -np.floor(np.median(v, axis=1) / grid) * grid
    return np.minimum(b, np.floor((cap - v.max(axis=1)) / grid) * grid)


def relu(x):
    return np.maximum(x, 0.0)


def policy_layout(case, spec, area, n2):
    """-> (policy_src or None for attention, policy length)."""
    if case.game and not case.n2:
        if spec.head == "chess_conv":
            return mapping.chess_flat_to_conv().astype(np.int32), spec.policy_size
        if spec.head == "ataxx":
            return np.concatenate([np.arange(spec.policy_size - 1), [-1]]).astype(np.int32), spec.policy_size
        if spec.head == "go":
            return np.concatenate([np.arange(area), [-2]]).astype(np.int32), spec.policy_size
        return None, spec.policy_size
    # every conv output, shuffled, and one zero logit
    src = np.concatenate([np.random.default_rng(area * n2).permutation(n2 * area), [-1]]).astype(np.int32)
    return src, src.size


@dataclass
class Built:
    net: Net
    planes: np.ndarray
    bits: np.ndarray
    scalars: np.ndarray
    mv_idx: np.ndarray
    mv_off: np.ndarray
    mapper: Mapper
    spec: Optional[netgen.GameSpec]


def inputs(case, rng):
    """(spec, bits, scalars, (cb, h, w), cs): netgen's synthetic positions with integer scalars, half the batch dense bits."""
    n = case.batch
    if case.game:
        spec = netgen.game_spec(case.game)
        bits, scalars, _, _ = netgen.synthetic_positions(spec, n, seed=rng.integers(1 << 30))
        shape, cs = (spec.bool_channels, spec.board_size, spec.board_size), spec.scalar_channels
    else:
        spec, (h, w), cs = None, case.board, 2
        shape = (3, h, w)
        cell = rng.choice(4, size=(n, h * w), p=[0.3, 0.3, 0.05, 0.35])
        planes = np.stack([cell == p for p in range(3)], axis=1).reshape(n, -1)
        bits = np.packbits(planes, axis=1, bitorder="little")
        scalars = rng.integers(0, 2, size=(n, cs)).astype(np.float32)
    integral = scalars == np.round(scalars)
    scalars = np.where(integral, np.mod(scalars, 8), rng.integers(0, 4, size=scalars.shape)).astype(np.float32)
    dense = (n + 1) // 2
    bits[:dense] = rng.integers(0, 256, size=bits[:dense].shape, dtype=np.uint8)
    return spec, bits, scalars, shape, cs


@functools.lru_cache(maxsize=None)
def build(case: Case) -> Built:
    rng = np.random.default_rng([ord(ch) for ch in case.id])
    spec, bits, scalars, (cb, h, w), cs = inputs(case, rng)
    n, area, C, k = case.batch, h * w, case.channels, case.k
    planes = oracle.expand_planes(bits, scalars, (cb, h, w), cs)
    x = planes.astype(np.float64)

    w0 = sparse_pm1(rng, C, cb + cs, 3, k)
    pre = conv64(x, w0)
    b0 = calibrate(pre, 256 if case.depth == 0 else 128)
    x = pre + b0[:, None, None]
    res_cap = np.floor((256 - x.max()) / case.depth) if case.depth else 0.0
    blocks = []
    for _ in range(case.depth):
        w1 = sparse_pm1(rng, C, C, 3, k)
        pre = conv64(x, w1)
        b1 = calibrate(pre, 256)
        t = relu(pre + b1[:, None, None])
        w2 = sparse_pm1(rng, C, C, 3, k)
        pre = conv64(t, w2)
        b2 = calibrate(pre, res_cap)
        x = x + relu(pre + b2[:, None, None])
        blocks += [(w1, b1), (w2, b2)]

    def head_conv(cout, cap, scale=1.0, grid=1.0, act=True, xin=x):
        wc = sparse_pm1(rng, cout, C, 1, k, scale)
        pre = conv64(xin, wc)
        bc = calibrate(pre, cap, grid)
        out = pre + bc[:, None, None]
        return (wc, bc), (relu(out) if act else out)

    def fc(xin, cout, cap, scale=1.0, grid=1.0, act=True):
        wf = sparse_pm1(rng, cout, xin.shape[1], 0, k, scale)
        pre = xin @ wf.T
        bf = calibrate(pre, cap, grid)
        out = pre + bf
        return (wf, bf), (relu(out) if act else out)

    scalar_conv, s1 = head_conv(case.hc, 256)
    fc1, hid = fc(s1.reshape(n, -1), case.hs, 256)
    fc2, _ = fc(hid, 5, np.inf, 2.0 ** -6, 2.0 ** -6, act=False)
    n2 = case.n2 or (spec.policy_conv_channels if spec else 17)
    src, plen = policy_layout(case, spec, area, n2)
    extra_conv = extra_fc = att = pc1 = pc2 = None
    if case.q:
        bulk, _ = head_conv(2 * case.q, 256, act=False)
        under, _ = head_conv(3 * case.q, 256, act=False, xin=x[:, :, 7:8, :])
        att = (bulk, under, case.q)
    else:
        pc1, h1 = head_conv(case.n1 or C, 256)
        wp2 = sparse_pm1(rng, n2, h1.shape[1], 1, k, 2.0 ** -5)
        pre = conv64(h1, wp2)
        pc2 = (wp2, calibrate(pre, np.inf, 2.0 ** -5))
        if (src == -2).any():
            extra_conv, e = head_conv(1, 256, act=False)
            extra_fc, _ = fc(e.reshape(n, -1), 1, np.inf, 2.0 ** -6, 2.0 ** -6, act=False)
    net = Net((h, w), (w0, b0), blocks, scalar_conv, fc1, fc2, pc1, pc2, src, extra_conv, extra_fc, att)

    mv_rng = np.random.default_rng(1 + n)
    counts = mv_rng.integers(1, min(plen, 60) + 1, size=n)
    mv_off = np.concatenate([[0], np.cumsum(counts)]).astype(np.uint32)
    mv_idx = np.concatenate([mv_rng.choice(plen, size=c, replace=False) for c in counts]).astype(np.uint32)
    return Built(net, planes, bits, scalars, mv_idx, mv_off, Mapper((cb, w, h), cs, (plen,)), spec)


# ----------------------------------------------------------------------------------------------------------- the reference
def grid_exp(a):
    """Smallest q >= 0 with a * 2^q integral everywhere."""
    a = np.asarray(a, dtype=np.float64)
    for q in range(40):
        if np.array_equal(np.round(a * 2.0 ** q), a * 2.0 ** q):
            return q
    raise AssertionError("values are not on a binary grid")


def assert_exact_sum(name, x, w, b, absum):
    q = grid_exp(x) + grid_exp(w)
    assert grid_exp(b) <= q, f"{name}: bias is off the 2^-{q} grid of the products"
    assert absum.max() < 2.0 ** (24 - q), f"{name}: sum |terms| {absum.max()} reaches 2^{24 - q}, f32 accumulation is not exact"


def assert_bf16_exact(name, a):
    f = np.asarray(a, dtype=np.float32)
    assert np.array_equal(f.astype(np.float64), a), f"{name}: not representable in f32"
    assert np.array_equal(bf16_round(f), f), f"{name}: not representable in bf16 (max |x| {np.abs(a).max()})"


FAULTS = ["mirrored_tap", "circular_padding", "dropped_kblock_channel", "residual_from_next_board", "dropped_last_bias",
          "relu_after_residual_add", "stale_layer_read", "unmasked_embedded_board", "swapped_h_w"]


def reference(net: Net, planes, check=False, fault=None):
    """float64 forward pass -> (scalars [n, 5], logits [n, P]).  check: assert the exactness preconditions (module docstring).
    fault: one of FAULTS, the deliberate bug to emulate."""
    n = planes.shape[0]
    h, w = net.board
    x = np.asarray(planes, dtype=np.float64)
    layers = [net.first] + net.blocks
    if check:
        for name, (wt, _) in [("first", net.first)] + [(f"block{i}", b) for i, b in enumerate(net.blocks)]:
            assert_bf16_exact(f"{name} weights", wt)
        assert_bf16_exact("input planes", x)

    embed = fault == "unmasked_embedded_board"
    if embed:  # the tower as tower8k runs a small board: embedded top-left in 8x8 and masked after every layer but the first
        assert h < 8 or w < 8
        x = np.pad(x, ((0, 0), (0, 0), (0, 8 - h), (0, 8 - w)))
        mask = np.zeros((8, 8))
        mask[:h, :w] = 1
    hit = 0 if not net.blocks else 1  # the layer the single-layer faults hit

    def conv(i, xin, name):
        wt, b = layers[i]
        if fault == "mirrored_tap" and i == hit:
            wt = wt.copy()
            wt[..., 2, 2] += wt[..., 0, 0]
            wt[..., 0, 0] = 0
        if fault == "dropped_kblock_channel" and i == hit:
            wt = wt.copy()
            wt[:, min(wt.shape[1], 64) - 1] = 0
        if fault == "dropped_last_bias":
            b = b.copy()
            b[-1] = 0
        if fault == "swapped_h_w":
            xin = xin.reshape(n, -1, w, h)
        y = conv64(xin, wt, b, circular=fault == "circular_padding")
        if fault == "swapped_h_w":
            y = y.reshape(n, -1, h, w)
        if check:
            assert_exact_sum(name, xin, wt, b, conv64(np.abs(xin), np.abs(wt), np.abs(b)))
        if embed and i != 0:
            y = y * mask
        return y

    x = conv(0, x, "first conv")
    if check:
        assert_bf16_exact("first conv output", x)
    x0 = x
    for d in range(len(net.blocks) // 2):
        t = relu(conv(1 + 2 * d, x, f"block{d} conv1"))
        if check:
            assert_bf16_exact(f"block{d} conv1 output", t)
        y = conv(2 + 2 * d, x0 if (fault == "stale_layer_read" and d == 0) else t, f"block{d} conv2")
        res = np.roll(x, -1, axis=0) if (fault == "residual_from_next_board" and d == 0) else x
        x = relu(res + y) if (fault == "relu_after_residual_add" and d == 0) else res + relu(y)
        if check:
            assert_bf16_exact(f"block{d} conv2 output", relu(y))
            assert_bf16_exact(f"block{d} output", x)
    if embed:
        x = x[:, :, :h, :w]
    if net.final_affine is not None:
        x = x * net.final_affine[0][:, None, None] + net.final_affine[1][:, None, None]

    def head_conv(wb, xin, name, act, stored_bf16=True):
        wt, b = wb
        y = conv64(xin, wt, b)
        if check:
            assert_bf16_exact(f"{name} weights", wt)
            assert_exact_sum(name, xin, wt, b, conv64(np.abs(xin), np.abs(wt), np.abs(b)))
        y = relu(y) if act else y
        if check and stored_bf16:
            assert_bf16_exact(f"{name} output", y)
        return y

    def fc(wb, xin, name, act):
        wt, b = wb
        if check:
            assert_bf16_exact(f"{name} weights", wt)
            assert_exact_sum(name, xin, wt, b, np.abs(xin) @ np.abs(wt).T + np.abs(b))
        y = xin @ wt.T + b
        return relu(y) if act else y

    s1 = head_conv(net.scalar_conv, x, "scalar conv", True)
    hid = fc(net.fc1, s1.reshape(n, -1), "fc1", True)
    scalars = fc(net.fc2, hid, "fc2", False)

    if net.att is not None:
        bulk_w, under_w, q = net.att
        bulk = head_conv(bulk_w, x, "attention bulk conv", False, stored_bf16=False)
        under = head_conv(under_w, x[:, :, 7:8, :], "attention under conv", False, stored_bf16=False)
        logits = attention_logits(bulk, under, q, check)
    else:
        h1 = head_conv(net.policy_conv1, x, "policy conv1", True)
        pm = head_conv(net.policy_conv2, h1, "policy conv2", False, stored_bf16=False).reshape(n, -1)
        src = net.policy_src
        logits = np.where(src >= 0, pm[:, np.maximum(src, 0)], 0.0)
        if net.extra_conv is not None:
            e = head_conv(net.extra_conv, x, "extra conv", False, stored_bf16=False)  # f32 in every path
            extra = fc(net.extra_fc, e.reshape(n, -1), "extra fc", False)
            logits = np.where(src == -2, extra, logits)
    if check:
        assert np.array_equal(scalars.astype(np.float32), scalars) and np.array_equal(logits.astype(np.float32), logits)
    return scalars, logits


def attention_logits(bulk, under, q, check):
    """The chess attention head's logits from the f32 outputs of its two convs."""
    n = bulk.shape[0]
    qf = bulk[:, :q].reshape(n, q, 64)
    qto = np.concatenate([bulk[:, q:].reshape(n, q, 64), under.reshape(n, q, 24)], axis=2)
    mm = np.einsum("nqf,nqt->nft", qf, qto)
    if check:
        assert_exact_sum("attention dot", qf, qto, 0.0, np.einsum("nqf,nqt->nft", np.abs(qf), np.abs(qto)))
    # one IEEE f32 division by the f32 constant the graph holds, as the oracle's Div and the tail kernel do
    att = mm.astype(np.float32) / np.array(float(q) ** 0.5, dtype=np.float32)
    return att.reshape(n, -1)[:, mapping.chess_flat_to_att()].astype(np.float64)


def decode64(scalars, logits, mv_idx, mv_off):
    """The packed decode in float64 -> (values [n, 5], probs, bound on |values - ref| [n, 5], bound on |probs - ref|): CUDA's
    expf / tanhf are within 2 ulp, division is IEEE, an n-term sum of positive f32 terms is within n 2^-24 relative, and the
    exponent's argument x - max is rounded once (|x - max| 2^-24 absolute)."""
    n = scalars.shape[0]
    values, bound_v = np.zeros((n, 5)), np.zeros((n, 5))
    values[:, 0] = np.tanh(scalars[:, 0])
    bound_v[:, 0] = 4 * U * np.abs(values[:, 0]) + 2.0 ** -140

    def softmax(z):
        z = z.astype(np.float32).astype(np.float64)
        d = z - z.max()
        p = np.exp(d)
        p /= p.sum()
        rel = 4 * U + 4 * U + len(z) * U + U + 2 * np.abs(d).max() * U
        return p, rel * p + 2.0 ** -140

    values[:, 1:4], bound_v[:, 1:4] = zip(*(softmax(scalars[i, 1:4]) for i in range(n)))
    values[:, 4] = scalars[:, 4]
    probs, bound_p = np.zeros(int(mv_off[-1])), np.zeros(int(mv_off[-1]))
    for i in range(n):
        sl = slice(int(mv_off[i]), int(mv_off[i + 1]))
        probs[sl], bound_p[sl] = softmax(logits[i, mv_idx[sl]])
    return values, probs, bound_v, bound_p


# ----------------------------------------------------------------------------------------------------------- creation paths
def raw_weights(net: Net) -> RawWeights:
    assert net.att is None
    return RawWeights(net.board, net.first, net.blocks, net.final_affine, net.scalar_conv, net.fc1, net.fc2, net.policy_conv1,
                      net.policy_conv2, net.policy_src, extra_conv=net.extra_conv, extra_fc=net.extra_fc)


def onnx_bytes(net: Net, spec, depth, channels, hc, hs, q):
    """The net as netgen's ONNX export, the final BN set to the identity (gamma 1, beta = mean = 0, var = f32(1 - 1e-5))."""
    names = {}
    netgen.build_onnx(spec, depth, channels, scalar_hidden_channels=hc, scalar_hidden_size=hs, query_channels=max(q, 1),
                      weights_out=names)
    convs = [net.first] + net.blocks + [net.scalar_conv]
    fcs = [net.fc1, net.fc2]
    if net.att is not None:
        convs += [net.att[0], net.att[1]]
    else:
        convs += [net.policy_conv1, net.policy_conv2] + ([net.extra_conv] if net.extra_conv else [])
        fcs += [net.extra_fc] if net.extra_fc else []
    conv_keys = sorted((int(k[1:]) for k in names if k[0] == "w"))
    fc_keys = sorted(int(k[4:]) for k in names if k.startswith("fc_w"))
    assert len(conv_keys) == len(convs) and len(fc_keys) == len(fcs)
    weights = {}
    for i, (wt, b) in zip(conv_keys, convs):
        weights[f"w{i}"], weights[f"b{i}"] = wt, b
    for i, (wt, b) in zip(fc_keys, fcs):
        weights[f"fc_w{i}"], weights[f"fc_b{i}"] = wt, b
    c = channels
    weights.update({"final_bn.weight": np.ones(c), "final_bn.bias": np.zeros(c), "final_bn.running_mean": np.zeros(c),
                    "final_bn.running_var": np.full(c, IDENTITY_VAR)})
    return netgen.build_onnx(spec, depth, channels, scalar_hidden_channels=hc, scalar_hidden_size=hs, query_channels=max(q, 1),
                             weights_in=weights)


def creation(case: Case, b: Built):
    if case.q:
        return onnx_bytes(b.net, b.spec, case.depth, case.channels, case.hc, case.hs, case.q)
    return raw_weights(b.net)


# ----------------------------------------------------------------------------------------------------------- CPU tests
def test_identity_bn_is_exact():
    """The identity final BN of the ONNX probe nets: the oracle's f32 BatchNormalization divides by sqrt(var + eps) == 1
    exactly, and the matcher's float64 fold scales by a with |a - 1| <= 2^-26, which rounds every head weight (0 or +-2^-j)
    back to itself."""
    assert np.float32(IDENTITY_VAR + BN_EPS) == np.float32(1)
    a = 1.0 / np.sqrt(np.float64(IDENTITY_VAR) + np.float64(BN_EPS))
    assert abs(a - 1) <= 2.0 ** -26
    for j in range(0, 12):
        for wt in (2.0 ** -j, -(2.0 ** -j)):
            assert np.float32(a * wt) == np.float32(wt)


@pytest.mark.parametrize("case_id", CASE_IDS)
def test_probe_preconditions_hold(case_id):
    """Every net of the GPU matrix is exact (reference(check=True) asserts it), and the generation is deterministic."""
    case = BY_ID[case_id]
    b = build(case)
    reference(b.net, b.planes, check=True)
    if case.batch > 64:
        return  # the large batches take long to generate twice; their recipe is the one the small cases repeat
    again = build.__wrapped__(case)
    assert np.array_equal(again.planes, b.planes) and np.array_equal(again.mv_idx, b.mv_idx)
    for (w1, b1), (w2, b2) in zip([b.net.first] + b.net.blocks, [again.net.first] + again.net.blocks):
        assert np.array_equal(w1, w2) and np.array_equal(b1, b2)
    # the calibration keeps the probes informative: a fair share of every stored tower tensor is nonzero
    x = conv64(b.planes, *b.net.first)
    assert (x != 0).mean() > 0.2


@pytest.mark.parametrize("case_id", ["chess-c40-d1-b3", "go-9-hs33", "ataxx-5", "att-q16", "att-q128"])
def test_oracle_equals_float64_reference(case_id):
    """The f32 oracle (plain C loops) returns exactly the float64 reference on the ONNX form of the probe nets."""
    case = BY_ID[case_id]
    b = build(case)
    ref_s, ref_p = reference(b.net, b.planes, check=True)
    model = onnx_bytes(b.net, b.spec, case.depth, case.channels, case.hc, case.hs, case.q)
    s, p = OnnxOracle(model).run(b.planes)
    assert np.array_equal(s, ref_s.astype(np.float32))
    assert np.array_equal(p, ref_p.astype(np.float32))


def default_net(game, depth, channels, seed=0):
    """A random-init netgen net (torch-default weights, a non-trivial final BN) as a Net."""
    spec = netgen.game_spec(game)
    wts = {}
    netgen.build_onnx(spec, depth, channels, seed=seed, weights_out=wts)
    g = {k: v.astype(np.float64) for k, v in wts.items()}
    conv = lambda i: (g[f"w{i}"], g[f"b{i}"])  # noqa: E731
    fcw = lambda i: (g[f"fc_w{i}"], g[f"fc_b{i}"])  # noqa: E731
    k = 2 * depth + 1
    scale = g["final_bn.weight"] / np.sqrt(g["final_bn.running_var"] + np.float64(BN_EPS))
    affine = (scale, g["final_bn.bias"] - scale * g["final_bn.running_mean"])
    src, _ = policy_layout(Case("default", game=game), spec, spec.area, spec.policy_conv_channels)
    return Net((spec.board_size,) * 2, conv(1), [conv(i) for i in range(2, k + 1)], conv(k + 1), fcw(k + 2), fcw(k + 3),
               conv(k + 4), conv(k + 5), src, final_affine=affine)


def torch_init(net: Net, seed):
    """The same shapes with torch-default weights U(-1/sqrt(fan_in), 1/sqrt(fan_in)) (netgen builds square boards only)."""
    rng = np.random.default_rng(seed)

    def re(wb):
        wt, b = wb
        bound = 1 / np.sqrt(np.prod(wt.shape[1:]))
        return rng.uniform(-bound, bound, wt.shape), rng.uniform(-bound, bound, b.shape)

    return Net(net.board, re(net.first), [re(b) for b in net.blocks], re(net.scalar_conv), re(net.fc1), re(net.fc2),
               re(net.policy_conv1), re(net.policy_conv2), net.policy_src)


def test_faults_change_the_probe_outputs(capsys):
    """Each deliberate fault changes at least one logit or scalar of a probe net.  Printed beside it: how far the same fault
    moves the logits of a default random-init net, which is why the tolerance tests cannot be relied on to see it."""
    where = {f: "chess-c40-d1-b3" for f in FAULTS}
    where.update(unmasked_embedded_board="ataxx-5", swapped_h_w="raw-9x7")
    rows = []
    for fault in FAULTS:
        b = build(BY_ID[where[fault]])
        s0, p0 = reference(b.net, b.planes)
        s1, p1 = reference(b.net, b.planes, fault=fault)
        changed = int((s0 != s1).sum() + (p0 != p1).sum())
        assert changed > 0, f"{fault} leaves the probe net {where[fault]} unchanged"
        if fault == "unmasked_embedded_board":
            dnet = default_net("ataxx-5", 2, 32)
        elif fault == "swapped_h_w":
            dnet = torch_init(b.net, 0)
        else:
            dnet = default_net("chess", 1, 40)
        planes = b.planes
        d0 = reference(dnet, planes)
        d1 = reference(dnet, planes, fault=fault)
        shift = max(np.abs(d0[0] - d1[0]).max(), np.abs(d0[1] - d1[1]).max())
        rows.append(f"{fault:26s} probe: {changed:6d} outputs changed   default net: max |shift| {shift:.3g}")
    with capsys.disabled():
        print("\n" + "\n".join(rows))


# ----------------------------------------------------------------------------------------------------------- GPU matrix
def expected(ref_s, ref_p, mv_idx, mv_off):
    """-> (scalars, logits, values, probabilities, bound on values, bound on probabilities) the GPU must meet."""
    return (ref_s, ref_p) + decode64(ref_s, ref_p, mv_idx, mv_off)


@functools.lru_cache(maxsize=8)
def case_reference(case: Case):
    """expected() of a case, computed once and shared by every precision and switch."""
    b = build(case)
    return expected(*reference(b.net, b.planes), b.mv_idx, b.mv_off)


def compare(tag, ref, s, p, values, probs, stats):
    """Scalars, logits and moves_left bit for bit, the decoded values and probabilities within their bounds."""
    ref_s, ref_p, ref_v, ref_probs, bound_v, bound_p = ref
    assert np.array_equal(s, ref_s.astype(np.float32)), f"{tag}: scalars differ in {np.count_nonzero(s != ref_s)} places"
    bad = np.argwhere(p != ref_p)
    assert bad.size == 0, f"{tag}: {len(bad)} logits differ, first (board, index) {bad[:4].tolist()}"
    assert np.array_equal(values[:, 4], ref_s[:, 4].astype(np.float32)), tag
    err_v = np.abs(values - ref_v)
    err_p = np.abs(probs - ref_probs)
    assert (err_v <= bound_v).all(), f"{tag}: values off by {err_v.max()}"
    assert (err_p <= bound_p).all(), f"{tag}: probabilities off by {err_p.max()}"
    stats.append(max((err_v[:, :4] / bound_v[:, :4]).max(), (err_p / bound_p).max() if err_p.size else 0.0))


def run_gpu(case: Case, precision, env, monkeypatch, stats, b=None, ref=None):
    """One network of the case in one precision under the switches env, against the reference (by default the case's net and
    inputs and their float64 reference; b and ref replace both)."""
    if b is None:
        b, ref = build(case), case_reference(case)
    for key, val in env:
        monkeypatch.setenv(key, val)
    try:
        with B200Network(b.mapper, creation(case, b), case.max_batch or case.batch, precision=precision) as net:
            if case.launches and precision == BF16 and not env:
                assert net.launches_per_eval() == case.launches
            s, p = net.evaluate_planes(b.planes)
            values, probs = net.evaluate_packed(b.bits, b.scalars, b.mv_idx, b.mv_off)
    finally:
        for key, _ in env:
            monkeypatch.delenv(key)
    compare(f"{case.id} {PRECISION_NAMES[precision]} {dict(env) or 'default'}", ref, s, p, values, probs, stats)
    return p


@pytest.mark.gpu
@pytest.mark.parametrize("case_id", CASE_IDS)
def test_gpu_equals_float64_reference(case_id, monkeypatch, capsys):
    """scalars and logits bit-identical to the reference on every path, in bf16 and fp32, with and without the kernel switches;
    the packed decode within its bound (the largest ratio of error to bound is printed)."""
    case = BY_ID[case_id]
    stats = []
    for precision in case.precisions:
        for env in ((),) + case.variants:
            run_gpu(case, precision, env, monkeypatch, stats)
    with capsys.disabled():
        print(f"\n{case_id}: largest decode error / bound {max(stats):.3f}")


@pytest.mark.gpu
@pytest.mark.parametrize("case_id", ["chess-c40-d1-b3", "ataxx-5", "go-9-hs33"])
def test_raw_weights_equal_the_onnx_net(case_id):
    """kzb_net_create and kzb_net_create_from_onnx build bit-identical networks from the same probe weights."""
    case = BY_ID[case_id]
    b = build(case)
    model = onnx_bytes(b.net, b.spec, case.depth, case.channels, case.hc, case.hs, case.q)
    for precision in (BF16, FP32):
        outs = []
        for weights in (raw_weights(b.net), model):
            with B200Network(b.mapper, weights, case.batch, precision=precision) as net:
                outs.append(net.evaluate_planes(b.planes) + net.evaluate_packed(b.bits, b.scalars, b.mv_idx, b.mv_off))
        for x, y in zip(*outs):
            assert np.array_equal(x, y)


@pytest.mark.gpu
@pytest.mark.parametrize("case_id", ["chess-c32-d2-b9469", "go-19-c64-b400"])
@pytest.mark.parametrize("precision", [BF16, TF32], ids=["bf16", "tf32"])
def test_rows_past_the_batch_do_not_leak(case_id, precision):
    """Row i is independent of the other rows and of batch (DESIGN §1), also of rows an earlier call left behind.  A call on
    three more boards, whose scalars are NaN, fails and leaves NaN in every activation buffer behind the batch; the next call's
    last tower8k unit, heads8 tile or conv pair tile holds those rows, and its results must still equal the reference."""
    case = BY_ID[case_id]
    b = build(case)
    n = case.batch
    assert case.max_batch in (0, n + 3)
    counts = np.diff(b.mv_off.astype(np.int64))
    last = slice(int(b.mv_off[n - 3]), int(b.mv_off[n]))
    mv_off = np.concatenate([b.mv_off, b.mv_off[n] + np.cumsum(counts[-3:])]).astype(np.uint32)
    nan_scalars = np.full((3, b.scalars.shape[1]), np.nan, np.float32)
    with B200Network(b.mapper, creation(case, b), n + 3, precision=precision) as net:
        with pytest.raises(KzbError, match="strictly positive"):
            net.evaluate_packed(np.concatenate([b.bits, b.bits[-3:]]), np.concatenate([b.scalars, nan_scalars]),
                                np.concatenate([b.mv_idx, b.mv_idx[last]]), mv_off)
        s, p = net.evaluate_planes(b.planes)
        values, probs = net.evaluate_packed(b.bits, b.scalars, b.mv_idx, b.mv_off)
    compare(f"{case_id} {PRECISION_NAMES[precision]} after NaN rows", case_reference(case), s, p, values, probs, [])
