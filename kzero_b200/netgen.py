"""Synthetic random-init nets in the reference's ONNX export structure (no torch, no `onnx` package).

The reference's networks reach the self-play server as ONNX files written by
python/lib/save_onnx.py:111-119 (opset 10, input `input`, outputs `scalars`,`policy`, dynamic batch).
There is no network access for real checkpoints, so the bench and the full-size GPU tests need
random-init nets of the named architectures.  This module writes ONNX bytes whose node sequence is
identical to what the reference's own classes export (python/lib/model/post_act.py:187-239 tower,
:10-23 scalar head, :54-112 conv policy heads, :115-141 attention head) -- pinned by
tests/test_netgen.py against tests/golden/export_structure.json, which was recorded from real
exports of the reference classes.

Initialisation follows torch defaults (Conv2d/Linear: U(-1/sqrt(fan_in), +1/sqrt(fan_in)) for weight
and bias) and SURVEY.md 8(d) for BatchNorm statistics (running_mean~N(0,0.1), running_var~U(0.5,1.5),
weight~U(0.5,1.5), bias~N(0,0.1)); in-block BNs are folded into the preceding Conv exactly like the
torch exporter does in eval mode, the final BN stays a BatchNormalization node.
"""
from __future__ import annotations

import struct
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import numpy as np

from .mapping import chess_flat_to_att, chess_flat_to_conv


# ------------------------------------------------------------------------------------ protobuf writer
def _varint(v: int) -> bytes:
    if v < 0:
        v += 1 << 64
    out = bytearray()
    while True:
        b = v & 0x7F
        v >>= 7
        if v:
            out.append(b | 0x80)
        else:
            out.append(b)
            return bytes(out)


def _key(fno: int, wt: int) -> bytes:
    return _varint((fno << 3) | wt)


def _ld(fno: int, payload: bytes) -> bytes:
    return _key(fno, 2) + _varint(len(payload)) + payload


def _vi(fno: int, v: int) -> bytes:
    return _key(fno, 0) + _varint(v)


def _tensor(name: str, arr: np.ndarray) -> bytes:
    arr = np.asarray(arr)
    dt = {np.dtype(np.float32): 1, np.dtype(np.int64): 7}[arr.dtype]
    out = b"".join(_vi(1, int(d)) for d in arr.shape)
    out += _vi(2, dt)
    if name:
        out += _ld(8, name.encode())
    out += _ld(9, np.ascontiguousarray(arr).astype(arr.dtype.newbyteorder("<")).tobytes())
    return out


def _attr(name: str, value) -> bytes:
    out = _ld(1, name.encode())
    if isinstance(value, float):
        out += _key(2, 5) + struct.pack("<f", value) + _vi(20, 1)
    elif isinstance(value, int):
        out += _vi(3, value) + _vi(20, 2)
    elif isinstance(value, np.ndarray):
        out += _ld(5, _tensor("", value)) + _vi(20, 4)
    elif isinstance(value, (list, tuple)):
        out += b"".join(_vi(8, int(v)) for v in value) + _vi(20, 7)
    else:
        raise TypeError(type(value))
    return out


def _value_info(name: str, shape: Sequence) -> bytes:
    dims = b""
    for d in shape:
        dims += _ld(1, _ld(2, d.encode()) if isinstance(d, str) else _vi(1, int(d)))
    tensor_type = _vi(1, 1) + _ld(2, dims)
    return _ld(1, name.encode()) + _ld(2, _ld(1, tensor_type))


class _GraphBuilder:
    def __init__(self, replace: Optional[dict] = None):
        self.replace = replace or {}
        self.nodes: List[bytes] = []
        self.inits: List[bytes] = []
        self.ops: List[str] = []
        self.arrays: dict = {}
        self._n = 0

    def init(self, name: str, arr: np.ndarray) -> str:
        if name in self.replace:
            new = np.asarray(self.replace[name], dtype=arr.dtype)
            if new.shape != arr.shape:
                raise ValueError(f"weights_in[{name!r}] has shape {new.shape}, the graph needs {arr.shape}")
            arr = new
        self.inits.append(_tensor(name, arr))
        self.arrays[name] = arr
        return name

    def node(self, op: str, inputs: Sequence[str], out: Optional[str] = None, **attrs) -> str:
        self._n += 1
        out = out or f"/{op}_{self._n}"
        payload = b"".join(_ld(1, i.encode()) for i in inputs) + _ld(2, out.encode())
        payload += _ld(3, f"{op}_{self._n}".encode()) + _ld(4, op.encode())
        payload += b"".join(_ld(5, _attr(k, v)) for k, v in attrs.items())
        self.nodes.append(payload)
        self.ops.append(op)
        return out

    def finish(self, inputs, outputs) -> bytes:
        g = b"".join(_ld(1, n) for n in self.nodes) + _ld(2, b"main_graph")
        g += b"".join(_ld(5, t) for t in self.inits)
        g += b"".join(_ld(11, _value_info(n, s)) for n, s in inputs)
        g += b"".join(_ld(12, _value_info(n, s)) for n, s in outputs)
        model = _vi(1, 5) + _ld(2, b"kzero_b200.netgen") + _ld(7, g) + _ld(8, _ld(1, b"") + _vi(2, 10))
        return model


# ------------------------------------------------------------------------------------ architecture
@dataclass(frozen=True)
class GameSpec:
    """Per-game tensor shapes, mirroring python/lib/games.py:22-58 (Game) and the Rust mappers."""
    name: str
    board_size: int
    bool_channels: int
    scalar_channels: int
    policy_size: int
    policy_conv_channels: int
    head: str  # "chess_conv" | "chess_att" | "ataxx" | "go"

    @property
    def input_channels(self) -> int:
        return self.bool_channels + self.scalar_channels

    @property
    def area(self) -> int:
        return self.board_size * self.board_size

    @property
    def bits_bytes(self) -> int:
        return (self.bool_channels * self.area + 7) // 8


def game_spec(name: str) -> GameSpec:
    if name == "chess":  # games.py:232-244, chess.rs:126-134,185
        return GameSpec("chess", 8, 13, 8, 1880, 73, "chess_conv")
    if name == "chess-att":
        return GameSpec("chess", 8, 13, 8, 1880, 73, "chess_att")
    if name.startswith("chess-hist-"):  # ChessHistoryMapper, rust/kz-core/src/mapping/chess.rs:25-40
        n = int(name.split("-")[2])
        return GameSpec(name, 8, 1 + 12 * (n + 1), 7 + (n + 1), 1880, 73, "chess_conv")
    if name.startswith("ataxx-"):  # games.py:144-159, ataxx.rs:21,94-104
        s = int(name.split("-")[1])
        return GameSpec(name, s, 3, 1, 17 * s * s + 1, 17, "ataxx")
    if name.startswith("go-"):  # games.py:178-194 (4 bool + 6 scalar, the Python-exportable form); "go-N-territory": GoStdMapper::new(size,
        # true), what the self-play server constructs (server.rs:193): three more bool planes (territory of us / them / nobody, go.rs:46-59)
        s = int(name.split("-")[1])
        return GameSpec(name, s, 7 if name.endswith("-territory") else 4, 6, s * s + 1, 1, "go")
    raise KeyError(name)


def _uniform(rng, shape, fan_in):
    b = 1.0 / np.sqrt(fan_in)
    return rng.uniform(-b, b, size=shape).astype(np.float32)


def _conv_params(rng, co, ci, k):
    fan_in = ci * k * k
    return _uniform(rng, (co, ci, k, k), fan_in), _uniform(rng, (co,), fan_in)


def _bn_params(rng, c):
    weight = rng.uniform(0.5, 1.5, c).astype(np.float32)
    bias = (rng.standard_normal(c) * 0.1).astype(np.float32)
    mean = (rng.standard_normal(c) * 0.1).astype(np.float32)
    var = rng.uniform(0.5, 1.5, c).astype(np.float32)
    return weight, bias, mean, var


_CONV3 = dict(dilations=[1, 1], group=1, kernel_shape=[3, 3], pads=[1, 1, 1, 1], strides=[1, 1])
_CONV1 = dict(dilations=[1, 1], group=1, kernel_shape=[1, 1], pads=[0, 0, 0, 0], strides=[1, 1])
_GEMM = dict(alpha=1.0, beta=1.0, transB=1)
_BN = dict(epsilon=float(np.float32(1e-5)), momentum=float(np.float32(0.9)))


def build_onnx(game: GameSpec, depth: int, channels: int, seed: int = 0, scalar_hidden_channels: int = 4,
               scalar_hidden_size: int = 32, query_channels: int = 32, fold_bn: bool = True,
               weights_out: Optional[dict] = None, legacy_three_outputs: bool = False,
               weights_in: Optional[dict] = None) -> bytes:
    """ONNX bytes for PredictionHeads(ResTower(depth, C_in, channels), ScalarHead, <policy head>).

    fold_bn=False keeps Conv -> BatchNormalization -> Relu un-folded inside blocks (what older torch
    versions / train-mode exports produce; Kyanite's optimiser folds those itself, SURVEY.md App. A).

    legacy_three_outputs: declare the outputs as (value [B], wdl [B, 3], policy), the legacy form network/common.rs:43-50 still accepts
    and this library rejects at load time (only used to test that rejection).

    weights_out: optional dict that receives every initializer (name -> array; tower convs are w1/b1 = input conv,
    w2.. = block convs in order) -- what bench.py's library comparator builds the same tower from.

    weights_in: optional dict (same names as weights_out) whose arrays replace those initializers; the random draws are made
    all the same, so the initializers it does not name keep their values.  Without it the bytes are unchanged."""
    rng = np.random.default_rng(seed)
    g = _GraphBuilder(weights_in)
    c, a, s = channels, game.area, game.board_size
    eps = np.float32(1e-5)
    k = 0

    def conv(x, w, b, attrs, out=None):
        nonlocal k
        k += 1
        return g.node("Conv", [x, g.init(f"w{k}", w), g.init(f"b{k}", b)], out, **attrs)

    def gemm(x, w, b, out=None):
        nonlocal k
        k += 1
        return g.node("Gemm", [x, g.init(f"fc_w{k}", w), g.init(f"fc_b{k}", b)], out, **_GEMM)

    def bn_node(x, params, tag):
        names = [g.init(f"{tag}.{n}", p) for n, p in zip(["weight", "bias", "running_mean", "running_var"], params)]
        return g.node("BatchNormalization", [x] + names, **_BN)

    # tower: post_act.py:201-228
    w0, b0 = _conv_params(rng, c, game.input_channels, 3)
    if game.name == "chess":  # (not chess-hist: its scalar order differs)
        # the two raw-count scalar planes (repetitions 0..2, halfmove clock 0..99, chess.rs:158-160) would
        # dominate a random-init net; a trained net has learned weights ~1/range for them, so scale likewise
        w0[:, 6] *= np.float32(1 / 2)
        w0[:, 7] *= np.float32(1 / 100)
    x = conv("input", w0, b0, _CONV3)
    for d in range(depth):
        y = x
        for j in range(2):
            w, b = _conv_params(rng, c, c, 3)
            bn = _bn_params(rng, c)
            if fold_bn:
                scale = bn[0] / np.sqrt(bn[3] + eps)
                w = (w * scale[:, None, None, None]).astype(np.float32)
                b = (b * scale + (bn[1] - scale * bn[2])).astype(np.float32)
                y = conv(y, w, b, _CONV3)
            else:
                y = conv(y, w, b, _CONV3)
                y = bn_node(y, bn, f"block{d}.bn{j}")
            y = g.node("Relu", [y])
        x = g.node("Add", [x, y])
    common = bn_node(x, _bn_params(rng, c), "final_bn")

    # scalar head: post_act.py:10-23
    hc, hs = scalar_hidden_channels, scalar_hidden_size
    y = conv(common, *_conv_params(rng, hc, c, 1), _CONV1)
    y = g.node("Relu", [y])
    y = g.node("Flatten", [y], axis=1)
    y = gemm(y, _uniform(rng, (hs, hc * a), hc * a), _uniform(rng, (hs,), hc * a))
    y = g.node("Relu", [y])
    gemm(y, _uniform(rng, (5, hs), hs), _uniform(rng, (5,), hs), out="scalars")

    # policy head
    policy_dim: object = game.policy_size
    if game.head in ("chess_conv", "ataxx", "go"):
        y = conv(common, *_conv_params(rng, c, c, 1), _CONV1)
        y = g.node("Relu", [y])
        pol = conv(y, *_conv_params(rng, game.policy_conv_channels, c, 1), _CONV1)
        if game.head == "chess_conv":  # post_act.py:86-88
            flat = g.node("Flatten", [pol], axis=1)
            idx = g.node("Constant", [], value=chess_flat_to_conv())
            g.node("Gather", [flat, idx], out="policy", axis=1)
        elif game.head == "ataxx":  # post_act.py:102-112: concat a zero "pass" logit
            shp = g.node("Shape", [pol])
            zero = g.node("Constant", [], value=np.array(0, dtype=np.int64))
            bs = g.node("Gather", [shp, zero], axis=0)
            flat = g.node("Flatten", [pol], axis=1)
            bs1 = g.node("Unsqueeze", [bs], axes=[0])
            one = g.node("Constant", [], value=np.array([1], dtype=np.int64))
            zshape = g.node("Concat", [bs1, one], axis=0)
            zeros = g.node("ConstantOfShape", [zshape], value=np.array([0], dtype=np.float32))
            g.node("Concat", [flat, zeros], out="policy", axis=1)
            policy_dim = "policy_dim_1"
        else:  # go: post_act.py:63-84 with extra_moves=1
            e = conv(common, *_conv_params(rng, 1, c, 1), _CONV1)
            e = g.node("Flatten", [e], axis=1)
            e = gemm(e, _uniform(rng, (1, a), a), _uniform(rng, (1,), a))
            flat = g.node("Flatten", [pol], axis=1)
            g.node("Concat", [flat, e], out="policy", axis=1)
    elif game.head == "chess_att":  # post_act.py:115-141
        q = query_channels
        i64 = lambda *v: np.array(v, dtype=np.int64)  # noqa: E731
        cst = lambda v: g.node("Constant", [], value=v)  # noqa: E731
        wb, bb = _conv_params(rng, 2 * q, c, 1)
        wu, bu = _conv_params(rng, 3 * q, c, 1)
        bulk = conv(common, wb, bb, _CONV1)
        row = g.node("Slice", [common, cst(i64(7)), cst(i64(8)), cst(i64(2)), cst(i64(1))])
        under = conv(row, wu, bu, _CONV1)
        qf = g.node("Slice", [bulk, cst(i64(0)), cst(i64(q)), cst(i64(1)), cst(i64(1))])
        qf = g.node("Reshape", [qf, cst(i64(0, q, 64))])
        qt = g.node("Slice", [bulk, cst(i64(q)), cst(i64(2 * q)), cst(i64(1)), cst(i64(1))])
        qt = g.node("Reshape", [qt, cst(i64(0, q, 64))])
        un = g.node("Reshape", [under, cst(i64(-1, q, 24))])
        qto = g.node("Concat", [qt, un], axis=2)
        qft = g.node("Transpose", [qf], perm=[0, 2, 1])
        mm = g.node("MatMul", [qft, qto])
        sc = g.node("Div", [mm, cst(np.array(float(q) ** 0.5, dtype=np.float32))])
        flat = g.node("Flatten", [sc], axis=1)
        g.node("Gather", [flat, cst(chess_flat_to_att())], out="policy", axis=1)
    else:
        raise KeyError(game.head)

    if weights_out is not None:
        weights_out.update(g.arrays)
    if legacy_three_outputs:
        i64 = lambda *v: g.node("Constant", [], value=np.array(v, dtype=np.int64))  # noqa: E731
        v = g.node("Slice", ["scalars", i64(0), i64(1), i64(1), i64(1)])
        g.node("Flatten", [v], out="value", axis=0)
        g.node("Slice", ["scalars", i64(1), i64(4), i64(1), i64(1)], out="wdl")
        return g.finish([("input", ["batch_size", game.input_channels, s, s])],
                        [("value", ["batch_size"]), ("wdl", ["batch_size", 3]), ("policy", ["batch_size", policy_dim])])
    return g.finish([("input", ["batch_size", game.input_channels, s, s])],
                    [("scalars", ["batch_size", 5]), ("policy", ["batch_size", policy_dim])])


# ------------------------------------------------------------------------------------ synthetic positions
def synthetic_positions(game: GameSpec, n: int, seed: int = 0, min_moves: int = 1,
                        max_moves: Optional[int] = None) -> Tuple[np.ndarray, np.ndarray, np.ndarray, np.ndarray]:
    """Seeded packed records in the layout `InputMapper::encode_input` produces
    (rust/kz-core/src/mapping/mod.rs:38, the record BinaryOutput::append_position writes,
    rust/kz-selfplay/src/binary_output.rs:218-247) plus a CSR legal-move index list like
    collect_policy_indices (binary_output.rs:299-315).

    -> bits [n, ceil(Cb*A/8)] u8, scalars [n, Cs] f32, mv_idx [total] u32, mv_off [n+1] u32.
    Distributions follow SURVEY.md 8(d) in spirit: sparse disjoint piece planes for chess, cell
    categories for ataxx/go, small-integer / one-hot scalars; legal moves are distinct uniform
    draws from the policy index range."""
    rng = np.random.default_rng(seed)
    a, cb = game.area, game.bool_channels
    planes = np.zeros((n, cb, a), dtype=np.uint8)
    scalars = np.zeros((n, game.scalar_channels), dtype=np.float32)
    if game.name == "chess":
        occ = rng.random((n, a))
        piece = rng.integers(0, 12, size=(n, a))
        for p in range(12):
            planes[:, p, :] = (occ < 0.35) & (piece == p)
        ep = rng.random(n) < 0.05
        planes[np.nonzero(ep)[0], 12, 40 + rng.integers(0, 8, size=int(ep.sum()))] = 1
        stm = rng.integers(0, 2, n)
        scalars[:, 0] = stm
        scalars[:, 1] = 1 - stm
        scalars[:, 2:6] = rng.integers(0, 2, size=(n, 4))
        scalars[:, 6] = rng.integers(0, 3, n)
        scalars[:, 7] = rng.integers(0, 100, n)
        lo, hi = 20, 45
    elif game.name.startswith("chess-hist"):  # chess.rs:42-95: en passant plane, then 12 piece planes per board
        boards = (cb - 1) // 12
        ep = rng.random(n) < 0.05
        planes[np.nonzero(ep)[0], 0, 40 + rng.integers(0, 8, size=int(ep.sum()))] = 1
        for h in range(boards):
            occ = rng.random((n, a))
            piece = rng.integers(0, 12, size=(n, a))
            for p in range(12):
                planes[:, 1 + 12 * h + p, :] = (occ < 0.35) & (piece == p)
        stm = rng.integers(0, 2, n)
        scalars[:, 0] = stm
        scalars[:, 1] = 1 - stm
        scalars[:, 2:6] = rng.integers(0, 2, size=(n, 4))
        scalars[:, 6] = rng.integers(0, 100, n) / np.float32(100)  # scaled like a trained net would see it
        scalars[:, 7:] = 1 + rng.integers(0, 3, size=(n, boards))  # 1 + repetitions (0 would be a padded board)
        lo, hi = 20, 45
    elif game.name.startswith("ataxx"):
        cell = rng.choice(4, size=(n, a), p=[0.3, 0.3, 0.05, 0.35])
        for p in range(3):
            planes[:, p, :] = cell == p
        scalars[:, 0] = rng.integers(0, 101, n) / np.float32(100)
        lo, hi = 1, min(100, game.policy_size)
    else:  # go
        cell = rng.choice(3, size=(n, a), p=[0.3, 0.3, 0.4])
        planes[:, 0, :] = cell == 0
        planes[:, 1, :] = cell == 1
        planes[:, 2, :] = 1
        ko = rng.random(n) < 0.1
        planes[np.nonzero(ko)[0], 3, rng.integers(0, a, size=int(ko.sum()))] = 1
        if cb == 7:  # territory planes: every point belongs to exactly one of us / them / nobody
            owner = rng.integers(0, 3, size=(n, a))
            for p in range(3):
                planes[:, 4 + p, :] = owner == p
        stm = rng.integers(0, 2, n)
        scalars[:, 0] = stm
        scalars[:, 1] = 1 - stm
        scalars[:, 4] = (rng.integers(-15, 16, n) / np.float32(2)) / np.float32(15)
        scalars[:, 5] = rng.integers(0, 2, n)
        lo, hi = 1, game.policy_size
    bits = np.packbits(planes.reshape(n, cb * a), axis=1, bitorder="little")
    assert bits.shape[1] == game.bits_bytes
    lo = max(lo, min_moves)
    hi = min(max_moves if max_moves is not None else hi, game.policy_size)
    counts = rng.integers(lo, hi + 1, size=n) if hi >= lo else np.full(n, hi)
    mv_off = np.zeros(n + 1, dtype=np.uint32)
    mv_off[1:] = np.cumsum(counts)
    mv_idx = np.empty(int(mv_off[-1]), dtype=np.uint32)
    for i in range(n):
        mv_idx[mv_off[i]:mv_off[i + 1]] = rng.choice(game.policy_size, size=int(counts[i]), replace=False)
    return bits, scalars, mv_idx, mv_off
