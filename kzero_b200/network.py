"""Python host mirror of the reference's `Network` interface over the C ABI (include/kzb200.h).

Mirrors, name for name where Python allows:
  trait Network<B>        rust/kz-core/src/network/mod.rs:52-63    -> B200Network.max_batch_size / evaluate_batch / evaluate
  ZeroEvaluation          network/mod.rs:26-32                     -> ZeroEvaluation(values, policy)
  ZeroValuesPov           rust/kz-core/src/zero/values.rs:14-18    -> ZeroValuesPov(value, wdl, moves_left)
  CudaNetwork::new        network/cudnn.rs:29-43                   -> B200Network(mapper, onnx_bytes, max_batch_size, device)
  BoardMapper shape half  mapping/mod.rs:19-36, 66-72              -> Mapper(input_bool_shape, input_scalar_count, policy_shape)

Board state itself (board-game crate) stays on the host in the reference and is out of scope here: a
"board" on this side is the record `InputMapper::encode_input` produces plus the legal-move index list
`PolicyMapper::move_to_index` yields (EncodedBoard), exactly what the Rust shim in INTEGRATION.md passes.

There is no CPU path: constructing a network without libkzb200.so or without a CUDA device raises.
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass
from typing import List, Sequence, Tuple

import numpy as np

from . import _abi
from ._abi import KzbError, NetInfo  # noqa: F401

PRECISION_FP32 = 0
PRECISION_BF16 = 1
PRECISION_TF32 = 2  # tcgen05 kind::tf32 on the row kernels, f32 activations rounded to TF32 (include/kzb200.h)


@dataclass(frozen=True)
class Mapper:
    """Shape half of `BoardMapper` (InputMapper + PolicyMapper), mapping/mod.rs:19-36,66-72."""
    input_bool_shape: Tuple[int, int, int]  # [bool channels, w, h]
    input_scalar_count: int
    policy_shape: Tuple[int, ...]

    def input_full_shape(self) -> Tuple[int, int, int]:
        b, w, h = self.input_bool_shape
        return (b + self.input_scalar_count, w, h)

    def input_bool_len(self) -> int:
        return int(np.prod(self.input_bool_shape))

    def policy_len(self) -> int:
        return int(np.prod(self.policy_shape))

    def bits_bytes(self) -> int:
        return (self.input_bool_len() + 7) // 8  # BitBuffer::new, bit_buffer.rs:11-17


@dataclass
class EncodedBoard:
    """What the host side knows about one board: encode_input's output + move_to_index of every legal move."""
    bits: np.ndarray  # uint8 [ceil(bool_len/8)]   BitBuffer::storage()
    scalars: np.ndarray  # float32 [scalar_count]
    policy_indices: np.ndarray  # uint32 [n_legal]; empty for a terminal board


@dataclass
class ZeroValuesPov:
    value: float
    wdl: Tuple[float, float, float]
    moves_left: float


@dataclass
class ZeroEvaluation:
    values: ZeroValuesPov
    policy: np.ndarray  # float32, only the available moves, in `available_moves` order; sums to 1


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(ctypes.c_void_p)


def _arr(a, dtype) -> np.ndarray:
    """`a` itself when it already is a C-contiguous array of `dtype` (the hot call stays copy-free), else a converted copy."""
    if type(a) is np.ndarray and a.dtype == dtype and a.flags.c_contiguous:
        return a
    return np.ascontiguousarray(a, dtype=dtype)


def device_count() -> int:
    return int(_abi.lib().kzb_device_count())


def inspect_onnx(onnx_bytes: bytes) -> NetInfo:
    info = NetInfo()
    _abi.check(_abi.lib().kzb_onnx_inspect(onnx_bytes, len(onnx_bytes), ctypes.byref(info)))
    return info


class RawWeights:
    """A kzb_net_spec built from numpy arrays (kept alive here): the input of kzb_net_create.

    first / blocks[i] / scalar_conv / policy_conv1 / policy_conv2 / extra_conv: (w [cout, cin, k, k], b [cout]);
    fc1 / fc2 / extra_fc: (w [out, in], b [out]); final_affine: (scale [C], shift [C]) or None; policy_src: int32 [policy_len]."""

    def __init__(self, board, first, blocks, final_affine, scalar_conv, fc1, fc2, policy_conv1, policy_conv2, policy_src,
                 extra_conv=None, extra_fc=None):
        self._keep = []

        def f32(a):
            a = np.ascontiguousarray(a, dtype=np.float32)
            self._keep.append(a)
            return a.ctypes.data_as(_abi._fp)

        def conv(wb):
            w, b = wb
            return _abi.ConvWeights(int(w.shape[1]), int(w.shape[0]), int(w.shape[2]), f32(w), f32(b))

        def fc(wb):
            w, b = wb
            return _abi.FcWeights(int(w.shape[1]), int(w.shape[0]), f32(w), f32(b))

        s = _abi.NetSpecC()
        s.board_h, s.board_w = (board, board) if isinstance(board, int) else board
        s.input_channels, s.channels, s.depth = int(first[0].shape[1]), int(first[0].shape[0]), len(blocks) // 2
        s.first = conv(first)
        self._blocks = (_abi.ConvWeights * max(len(blocks), 1))(*[conv(b) for b in blocks])
        s.blocks = ctypes.cast(self._blocks, ctypes.POINTER(_abi.ConvWeights))
        if final_affine is not None:
            s.final_scale, s.final_shift = f32(final_affine[0]), f32(final_affine[1])
        s.scalar_conv, s.fc1, s.fc2 = conv(scalar_conv), fc(fc1), fc(fc2)
        s.policy_conv1, s.policy_conv2 = conv(policy_conv1), conv(policy_conv2)
        s.has_extra = int(extra_conv is not None)
        if extra_conv is not None:
            s.extra_conv, s.extra_fc = conv(extra_conv), fc(extra_fc)
        src = np.ascontiguousarray(policy_src, dtype=np.int32)
        self._keep.append(src)
        s.policy_len, s.policy_src = int(src.size), src.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))
        self.spec = s


class B200Network:
    """Drop-in for `CudaNetwork<B, M>` (network/cudnn.rs:18-88) behind the same evaluate_batch contract."""

    def __init__(self, mapper: Mapper, onnx_bytes, max_batch_size: int, device: int = 0,
                 precision: int = PRECISION_BF16):
        """onnx_bytes: the ONNX file's bytes (kzb_net_create_from_onnx), or a `RawWeights` (kzb_net_create: weights the caller
        already holds, e.g. the constants of a Graph the reference's own `load_graph` produced)."""
        self._lib = _abi.lib()
        self._handle = ctypes.c_void_p()
        self.mapper = mapper
        if isinstance(onnx_bytes, RawWeights):
            _abi.check(self._lib.kzb_net_create(device, ctypes.byref(onnx_bytes.spec), int(max_batch_size), int(precision),
                                                ctypes.byref(self._handle)))
        else:
            _abi.check(self._lib.kzb_net_create_from_onnx(device, onnx_bytes, len(onnx_bytes), int(max_batch_size),
                                                          int(precision), ctypes.byref(self._handle)))
        try:
            _, w, h = mapper.input_bool_shape
            # check_graph_shapes(mapper, graph), network/common.rs:165-198
            _abi.check(self._lib.kzb_net_bind_mapper(self._handle, mapper.input_scalar_count, mapper.input_bool_shape[0],
                                                     h, w, mapper.policy_len()))
        except Exception:
            self.close()
            raise
        self._max_batch_size = int(max_batch_size)
        self._bits_bytes = mapper.bits_bytes()

    # -- lifetime ---------------------------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_handle", None):
            self._lib.kzb_net_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- Network trait ----------------------------------------------------------------------------
    def max_batch_size(self) -> int:
        return self._max_batch_size

    def evaluate_batch(self, boards: Sequence[EncodedBoard]) -> List[ZeroEvaluation]:
        """One result per board, same order (network/mod.rs:55-56)."""
        n = len(boards)
        assert n <= self._max_batch_size  # cudnn.rs:58
        if n == 0:
            return []
        bits = np.stack([np.asarray(b.bits, dtype=np.uint8) for b in boards])
        scalars = np.stack([np.asarray(b.scalars, dtype=np.float32) for b in boards]).reshape(n, -1)
        counts = [len(b.policy_indices) for b in boards]
        mv_off = np.zeros(n + 1, dtype=np.uint32)
        mv_off[1:] = np.cumsum(counts)
        mv_idx = (np.concatenate([np.asarray(b.policy_indices, dtype=np.uint32) for b in boards])
                  if mv_off[-1] else np.zeros(0, np.uint32))
        values, probs = self.evaluate_packed(bits, scalars, mv_idx, mv_off)
        out = []
        for i in range(n):
            v = values[i]
            out.append(ZeroEvaluation(ZeroValuesPov(float(v[0]), (float(v[1]), float(v[2]), float(v[3])), float(v[4])),
                                      probs[mv_off[i]:mv_off[i + 1]].copy()))
        return out

    def evaluate(self, board: EncodedBoard) -> ZeroEvaluation:
        result = self.evaluate_batch([board])
        assert len(result) == 1  # network/mod.rs:59-62
        return result[0]

    # -- array forms of the same call ---------------------------------------------------------------
    def evaluate_packed(self, bits: np.ndarray, scalars: np.ndarray, mv_idx: np.ndarray, mv_off: np.ndarray):
        """kzb_eval_packed: -> (values [n,5], probs [mv_off[-1]])."""
        bits = _arr(bits, np.uint8)
        n = bits.shape[0]
        assert bits.size == n * self._bits_bytes
        scalars = _arr(scalars, np.float32)
        assert scalars.size == n * self.mapper.input_scalar_count
        mv_idx = _arr(mv_idx, np.uint32)
        mv_off = _arr(mv_off, np.uint32)
        assert mv_off.shape[0] == n + 1
        values = np.empty((n, 5), dtype=np.float32)
        probs = np.empty((int(mv_off[-1]),), dtype=np.float32)
        rc = self._lib.kzb_eval_packed(self._handle, bits.ctypes.data, scalars.ctypes.data, n, mv_idx.ctypes.data,
                                       mv_off.ctypes.data, values.ctypes.data, probs.ctypes.data)
        if rc != 0:
            _abi.check(rc)
        return values, probs

    def set_symmetries(self, square_src: np.ndarray, policy_map: np.ndarray) -> None:
        """kzb_net_set_symmetries: square_src [n_sym, H*W], policy_map [n_sym, policy_len] (see include/kzb200.h)."""
        square_src = np.ascontiguousarray(square_src, dtype=np.int32)
        policy_map = np.ascontiguousarray(policy_map, dtype=np.int32)
        assert square_src.shape[0] == policy_map.shape[0] and policy_map.shape[1] == self.mapper.policy_len()
        _abi.check(self._lib.kzb_net_set_symmetries(self._handle, square_src.shape[0], _ptr(square_src), _ptr(policy_map)))

    def evaluate_packed_sym(self, bits, scalars, sym, mv_idx, mv_off):
        """kzb_eval_packed_sym: like evaluate_packed, every board evaluated under its symmetry sym[i] (RandomSymmetryNetwork
        on the GPU, network/symmetry.rs:41-67)."""
        bits = _arr(bits, np.uint8)
        n = bits.shape[0]
        scalars = _arr(scalars, np.float32)
        sym = _arr(sym, np.uint8)
        mv_idx = _arr(mv_idx, np.uint32)
        mv_off = _arr(mv_off, np.uint32)
        assert sym.shape == (n,) and mv_off.shape[0] == n + 1
        values = np.empty((n, 5), dtype=np.float32)
        probs = np.empty((int(mv_off[-1]),), dtype=np.float32)
        _abi.check(self._lib.kzb_eval_packed_sym(self._handle, _ptr(bits), _ptr(scalars), _ptr(sym), n, _ptr(mv_idx), _ptr(mv_off),
                                                 _ptr(values), _ptr(probs)))
        return values, probs

    def evaluate_planes(self, nchw: np.ndarray):
        """kzb_eval_planes, the twin of CudaExecutor::evaluate: -> (scalars [n,5] raw, policy logits [n,P])."""
        nchw = np.ascontiguousarray(nchw, dtype=np.float32)
        n = nchw.shape[0]
        assert tuple(nchw.shape[1:]) == (self.info().input_channels, self.info().board_h, self.info().board_w)
        scalars = np.empty((n, 5), dtype=np.float32)
        logits = np.empty((n, self.mapper.policy_len()), dtype=np.float32)
        _abi.check(self._lib.kzb_eval_planes(self._handle, _ptr(nchw), n, _ptr(scalars), _ptr(logits)))
        return scalars, logits

    def encode_planes(self, bits: np.ndarray, scalars: np.ndarray) -> np.ndarray:
        """K2 alone (GPU twin of encode_input_full): -> planes [n, Cs+Cb, H, W] f32."""
        bits = np.ascontiguousarray(bits, dtype=np.uint8)
        n = bits.shape[0]
        scalars = np.ascontiguousarray(scalars, dtype=np.float32).reshape(n, self.mapper.input_scalar_count)
        c, w, h = self.mapper.input_full_shape()
        out = np.empty((n, c, h, w), dtype=np.float32)
        _abi.check(self._lib.kzb_encode_planes(self._handle, _ptr(bits), _ptr(scalars), n, _ptr(out)))
        return out

    # -- measurement hooks -----------------------------------------------------------------------
    def info(self) -> NetInfo:
        info = NetInfo()
        _abi.check(self._lib.kzb_net_get_info(self._handle, ctypes.byref(info)))
        return info

    def stage_packed(self, bits, scalars, mv_idx, mv_off) -> None:
        bits = np.ascontiguousarray(bits, dtype=np.uint8)
        n = bits.shape[0]
        scalars = np.ascontiguousarray(scalars, dtype=np.float32)
        mv_idx = np.ascontiguousarray(mv_idx, dtype=np.uint32)
        mv_off = np.ascontiguousarray(mv_off, dtype=np.uint32)
        _abi.check(self._lib.kzb_stage_packed(self._handle, _ptr(bits), _ptr(scalars), n, _ptr(mv_idx), _ptr(mv_off)))

    def time_staged(self, iters: int, flush_l2: bool = True) -> np.ndarray:
        ms = np.empty(iters, dtype=np.float32)
        _abi.check(self._lib.kzb_time_staged(self._handle, iters, int(flush_l2), _ptr(ms)))
        return ms

    def profile_staged(self, flush_l2: bool = True):
        names = ctypes.create_string_buffer(1 << 16)
        ms = np.empty(1024, dtype=np.float32)
        n = ctypes.c_int(0)
        _abi.check(self._lib.kzb_profile_staged(self._handle, int(flush_l2), names, len(names), _ptr(ms), 1024,
                                                ctypes.byref(n)))
        return names.value.decode().split("\n"), ms[:n.value].copy()

    def launches_per_eval(self) -> int:
        return int(self._lib.kzb_launches_per_eval(self._handle))


def mapper_for(game) -> Mapper:
    """Mapper for a kzero_b200.netgen.GameSpec."""
    return Mapper((game.bool_channels, game.board_size, game.board_size), game.scalar_channels, (game.policy_size,))
