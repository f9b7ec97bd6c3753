"""Parity of the CUDA path (through the C ABI) against the oracle and the reference-derived golden files.

Bars (BASELINE.json north_star):
  input planes            bit-exact
  fp32 path               <= 1e-4 max-abs on scalars and policy logits
  bf16 tensor-core path   <= 2e-2 max-abs on policy logits, value sign agreement reported/checked
"""
import numpy as np
import pytest

import oracle
from oracle.graph_exec import OnnxOracle
from helpers import GOLDEN, load_net_fixture
from kzero_b200 import netgen
from kzero_b200.network import (B200Network, EncodedBoard, KzbError, Mapper, PRECISION_BF16, PRECISION_FP32,
                                mapper_for)

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-4
BF16_POLICY_TOL = 2e-2

FIXTURE_GAMES = {"ataxx7_2x32": "ataxx-7", "chess_conv_2x32": "chess", "chess_att_2x32": "chess-att", "go9_2x32": "go-9",
                 "ataxx5_scripted_1x16": "ataxx-5"}


def _oracle_planes(spec, bits, scalars):
    return oracle.expand_planes(bits, scalars, (spec.bool_channels, spec.board_size, spec.board_size),
                                spec.scalar_channels)


def _tiny_net(spec, **kw):
    return netgen.build_onnx(spec, 1, 16, seed=11, **kw)


# ------------------------------------------------------------------------------------------- K2 encode
@pytest.mark.parametrize("game", ["chess", "ataxx-7", "go-9", "ataxx-3", "go-19"])
def test_encode_bit_exact_vs_reference_golden(game):
    d = np.load(GOLDEN / f"planes_{game}.npz")
    cb, h, w = (int(v) for v in d["bool_shape"])
    cs = int(d["scalar_count"])
    spec = netgen.game_spec(game)
    assert (spec.bool_channels, spec.scalar_channels) == (cb, cs)
    with B200Network(mapper_for(spec), _tiny_net(spec), 8, precision=PRECISION_FP32) as net:
        out = net.encode_planes(d["bits"], d["scalars"])
    assert np.array_equal(out.view(np.uint32), d["planes"].view(np.uint32))


@pytest.mark.parametrize("game,n", [("chess", 1024), ("ataxx-7", 256), ("go-9", 333)])
def test_encode_bit_exact_vs_oracle_full_batch(game, n):
    spec = netgen.game_spec(game)
    bits, scalars, _, _ = netgen.synthetic_positions(spec, n, seed=3)
    rng = np.random.default_rng(4)
    bits[: n // 2] = rng.integers(0, 256, size=bits[: n // 2].shape, dtype=np.uint8)  # dense random bits too
    scalars[: n // 2] = rng.standard_normal(scalars[: n // 2].shape).astype(np.float32)
    with B200Network(mapper_for(spec), _tiny_net(spec), n, precision=PRECISION_FP32) as net:
        out = net.encode_planes(bits, scalars)
    ref = _oracle_planes(spec, bits, scalars)
    assert np.array_equal(out.view(np.uint32), ref.view(np.uint32))


# ------------------------------------------------------------------------------------------- fp32 path
@pytest.mark.parametrize("name", list(FIXTURE_GAMES))
def test_fp32_planes_vs_reference_pytorch_golden(name):
    """kzb_eval_planes (twin of CudaExecutor::evaluate) against the PyTorch outputs the reference's own
    check files hold (save_onnx.py:94-102)."""
    onnx_bytes, x, scalars, policy = load_net_fixture(name)
    spec = netgen.game_spec(FIXTURE_GAMES[name])
    with B200Network(mapper_for(spec), onnx_bytes, 8, precision=PRECISION_FP32) as net:
        s, p = net.evaluate_planes(x)
    assert np.abs(s - scalars).max() <= FP32_TOL
    assert np.abs(p - policy).max() <= FP32_TOL


@pytest.mark.parametrize("name", list(FIXTURE_GAMES))
def test_bf16_planes_vs_reference_pytorch_golden(name):
    onnx_bytes, x, scalars, policy = load_net_fixture(name)
    spec = netgen.game_spec(FIXTURE_GAMES[name])
    with B200Network(mapper_for(spec), onnx_bytes, 8, precision=PRECISION_BF16) as net:
        s, p = net.evaluate_planes(x)
    assert np.abs(p - policy).max() <= BF16_POLICY_TOL
    assert np.abs(s - scalars).max() <= 5e-2


@pytest.mark.parametrize("game,depth,ch,n", [("ataxx-7", 8, 64, 64), ("chess", 4, 64, 33), ("go-9", 3, 48, 17)])
@pytest.mark.parametrize("fold_bn", [True, False])
def test_fp32_planes_vs_oracle(game, depth, ch, n, fold_bn):
    spec = netgen.game_spec(game)
    onnx_bytes = netgen.build_onnx(spec, depth, ch, seed=5, fold_bn=fold_bn)
    x = np.random.default_rng(6).standard_normal((n, spec.input_channels, spec.board_size, spec.board_size)).astype(np.float32)
    ref_s, ref_p = OnnxOracle(onnx_bytes).run(x)
    with B200Network(mapper_for(spec), onnx_bytes, n, precision=PRECISION_FP32) as net:
        s, p = net.evaluate_planes(x)
    assert np.abs(s - ref_s).max() <= FP32_TOL
    assert np.abs(p - ref_p).max() <= FP32_TOL


# ------------------------------------------------------------------------------------------- packed path
def _oracle_packed(spec, onnx_bytes, bits, scalars, mv_idx, mv_off):
    planes = _oracle_planes(spec, bits, scalars)
    s, p = OnnxOracle(onnx_bytes).run(planes)
    values, probs = oracle.decode_output(s, p, mv_idx, mv_off)
    return s, p, values, probs


def _check_packed(values, probs, ref_values, ref_probs, mv_off, tol_v, tol_p):
    assert np.abs(values - ref_values).max() <= tol_v
    if probs.size:
        assert np.abs(probs - ref_probs).max() <= tol_p
    for i in range(len(mv_off) - 1):
        seg = probs[mv_off[i]:mv_off[i + 1]]
        if seg.size:
            assert abs(float(seg.sum()) - 1.0) < 1e-4


@pytest.mark.parametrize("game,depth,ch,n", [("ataxx-7", 8, 64, 256), ("chess", 2, 32, 50), ("go-9", 2, 32, 31)])
def test_fp32_packed_vs_oracle(game, depth, ch, n):
    """Full fused call (encode -> tower -> heads -> masked softmax) vs oracle expand + graph + decode_output.
    ataxx-7 8x64 batch 256 is BASELINE.json configs[0]."""
    spec = netgen.game_spec(game)
    onnx_bytes = netgen.build_onnx(spec, depth, ch, seed=7)
    bits, scalars, mv_idx, mv_off = netgen.synthetic_positions(spec, n, seed=8)
    _, _, ref_values, ref_probs = _oracle_packed(spec, onnx_bytes, bits, scalars, mv_idx, mv_off)
    with B200Network(mapper_for(spec), onnx_bytes, n, precision=PRECISION_FP32) as net:
        values, probs = net.evaluate_packed(bits, scalars, mv_idx, mv_off)
    _check_packed(values, probs, ref_values, ref_probs, mv_off, FP32_TOL, FP32_TOL)


@pytest.mark.parametrize("variant", ["default", "no_heads8", "no_tower8", "no_conv8", "linear", "no_embed8", "no_pdl", "no_conv_split"])
@pytest.mark.parametrize("game,depth,ch,n", [("ataxx-7", 8, 64, 256), ("chess", 16, 128, 64), ("go-9", 4, 64, 40),
                                              ("chess", 2, 32, 7), ("chess", 3, 64, 130), ("chess", 2, 256, 12),
                                              ("chess", 2, 32, 9600)])
def test_bf16_packed_vs_oracle(game, depth, ch, n, variant, monkeypatch):
    """The tensor-core path in all its forms: whole-tower persistent kernel + fused heads kernel (tower8k.cu, heads8.cu, default for 8x8
    boards), the same tower with per-op head convs + tail kernel (KZB_NO_HEADS8=1), conv_i2c.cu on 8x8 boards with the fused heads kernel
    (KZB_NO_TOWER8=1; by default for layers wider than 128 channels, and for chess batch 9600, which has more 4-board units per SM than
    the whole-tower kernel keeps), no 8x8 conv kernel at all (KZB_NO_TOWER8=1 and KZB_NO_HEADS8=1: conv_i2c.cu on 8x8 boards, per-op
    head convs + tail kernel), and the row kernels of every other board (go; KZB_FORCE_LINEAR=1 / KZB_NO_EMBED8=1 push chess / ataxx
    there): dense rows with TMA im2col loads and the CTA-pair MMA (conv_i2c.cu, also the head 1x1 convs) and the tail kernel,
    without programmatic dependent launch (KZB_PDL=0), and without sharing a tile's output channels between two SM pairs at small
    batches (KZB_CONV_SPLIT=0).  Boards smaller than 8x8 (ataxx 7x7) are embedded in the 8x8 grid and masked after every layer."""
    row_variants = ("linear", "no_pdl", "no_conv_split")  # everything off the 8x8 kernels
    if variant == "no_embed8":
        if game != "ataxx-7":
            pytest.skip("only boards smaller than 8x8 are embedded")
    elif variant in row_variants:
        if game == "ataxx-7":
            pytest.skip("covered by go-9 and the chess nets on the row kernels")
    elif variant != "default" and game != "chess":
        pytest.skip("the kernel variants are 8x8 specialisations")
    monkeypatch.setenv("KZB_NO_EMBED8", "1" if variant == "no_embed8" else "0")
    force_linear = "1" if variant in row_variants else "0"
    monkeypatch.setenv("KZB_PDL", "0" if variant == "no_pdl" else "1")
    monkeypatch.setenv("KZB_CONV_SPLIT", "0" if variant == "no_conv_split" else "1")
    monkeypatch.setenv("KZB_FORCE_LINEAR", force_linear)
    monkeypatch.setenv("KZB_NO_TOWER8", "1" if variant in ("no_tower8", "no_conv8") else "0")
    monkeypatch.setenv("KZB_NO_HEADS8", "1" if variant in ("no_heads8", "no_conv8") else "0")
    spec = netgen.game_spec(game)
    onnx_bytes = netgen.build_onnx(spec, depth, ch, seed=9)
    bits, scalars, mv_idx, mv_off = netgen.synthetic_positions(spec, n, seed=10)
    ref_s, ref_p, ref_values, ref_probs = _oracle_packed(spec, onnx_bytes, bits, scalars, mv_idx, mv_off)
    with B200Network(mapper_for(spec), onnx_bytes, n, precision=PRECISION_BF16) as net:
        # 8x8 boards, and smaller boards embedded in the 8x8 grid (ataxx 7x7), run on the 8x8 kernels; go-9 on the row kernels
        on_8x8 = (game == "chess" and force_linear == "0") or (game == "ataxx-7" and variant == "default")
        assert net.info().conv_mode == (1 if on_8x8 else 0)
        if n > 4 * 16 * 148 and variant == "default":  # 148 SMs: conv_i2c.cu runs the tower layer by layer, then heads8
            assert net.launches_per_eval() == 2 * depth + 3
        values, probs = net.evaluate_packed(bits, scalars, mv_idx, mv_off)
        planes = _oracle_planes(spec, bits, scalars)
        s, p = net.evaluate_planes(planes)
    err_p = np.abs(p - ref_p).max()
    assert err_p <= BF16_POLICY_TOL, err_p
    # value sign agreement wherever the oracle's value is not within rounding distance of zero
    clear = np.abs(ref_s[:, 0]) > 0.05
    agree = np.sign(s[clear, 0]) == np.sign(ref_s[clear, 0])
    assert agree.all(), f"value sign agreement {agree.mean():.4f}"
    _check_packed(values, probs, ref_values, ref_probs, mv_off, 5e-2, 1e-2)


@pytest.mark.parametrize("precision,tol_logit,tol_v,tol_p", [(PRECISION_FP32, FP32_TOL, FP32_TOL, FP32_TOL),
                                                              (PRECISION_BF16, BF16_POLICY_TOL, 5e-2, 1e-2)])
@pytest.mark.parametrize("depth,ch,q,n", [(2, 32, 32, 19), (3, 128, 128, 70)])
def test_attention_head_vs_oracle(depth, ch, q, n, precision, tol_logit, tol_v, tol_p):
    """AttentionPolicyHead (post_act.py:115-141), incl. Q = channels = 128 as supervised_main_alpha.py:76 builds it
    (conv_under has 384 output channels -> two launches)."""
    spec = netgen.game_spec("chess-att")
    onnx_bytes = netgen.build_onnx(spec, depth, ch, seed=21, query_channels=q)
    bits, scalars, mv_idx, mv_off = netgen.synthetic_positions(spec, n, seed=22)
    ref_s, ref_p, ref_values, ref_probs = _oracle_packed(spec, onnx_bytes, bits, scalars, mv_idx, mv_off)
    with B200Network(mapper_for(spec), onnx_bytes, n, precision=precision) as net:
        values, probs = net.evaluate_packed(bits, scalars, mv_idx, mv_off)
        s, p = net.evaluate_planes(_oracle_planes(spec, bits, scalars))
    assert np.abs(p - ref_p).max() <= tol_logit, np.abs(p - ref_p).max()
    _check_packed(values, probs, ref_values, ref_probs, mv_off, tol_v, tol_p)


@pytest.mark.parametrize("path", ["heads8", "tail", "fp32", "attention"])
def test_long_legal_move_lists_vs_oracle(path, monkeypatch):
    """Legal-move lists longer than real positions have, so that every form of the masked softmax (head_decode.cuh) runs: up to
    256 moves (registers in both kernels), 257..384 (registers in the tail kernel, the long-list form in heads8) and more than 384
    (the long-list form in both).  On heads8 (bf16 default), the tail kernel (bf16 with KZB_NO_HEADS8=1, and fp32) and the tail
    kernel's attention logits (chess-att)."""
    monkeypatch.setenv("KZB_NO_HEADS8", "1" if path == "tail" else "0")
    spec = netgen.game_spec("chess-att" if path == "attention" else "chess")
    precision = PRECISION_FP32 if path == "fp32" else PRECISION_BF16
    onnx_bytes = netgen.build_onnx(spec, 2, 32, seed=23)
    bits, scalars, mv_idx, mv_off = netgen.synthetic_positions(spec, 24, seed=42, min_moves=200, max_moves=600)
    n_moves = np.diff(mv_off)
    assert (n_moves <= 256).any() and ((n_moves > 256) & (n_moves <= 384)).any() and (n_moves > 384).any()
    _, _, ref_values, ref_probs = _oracle_packed(spec, onnx_bytes, bits, scalars, mv_idx, mv_off)
    with B200Network(mapper_for(spec), onnx_bytes, 24, precision=precision) as net:
        assert (net.launches_per_eval() == 3) == (path == "heads8")  # encode, tower8k, heads8
        values, probs = net.evaluate_packed(bits, scalars, mv_idx, mv_off)
    tol_v, tol_p = (FP32_TOL, FP32_TOL) if precision == PRECISION_FP32 else (5e-2, 1e-2)
    _check_packed(values, probs, ref_values, ref_probs, mv_off, tol_v, tol_p)


@pytest.mark.parametrize("n", [887, 888, 1024, 1036, 1184, 1185])
def test_bf16_balanced_units_match_uniform_units(n, monkeypatch):
    """tower8k's balanced board assignment (every SM owns 6..8 boards as two units of 4 / 3 boards, batches 888..1184)
    against the uniform 4-board units (KZB_NO_BALANCE=1): a board's result must not depend on which unit computed it."""
    spec = netgen.game_spec("chess")
    onnx_bytes = netgen.build_onnx(spec, 3, 128, seed=41)
    bits, scalars, mv_idx, mv_off = netgen.synthetic_positions(spec, n, seed=42)
    monkeypatch.setenv("KZB_NO_BALANCE", "1")
    with B200Network(mapper_for(spec), onnx_bytes, n) as net:
        v0, p0 = net.evaluate_packed(bits, scalars, mv_idx, mv_off)
    monkeypatch.setenv("KZB_NO_BALANCE", "0")
    with B200Network(mapper_for(spec), onnx_bytes, n) as net:
        v1, p1 = net.evaluate_packed(bits, scalars, mv_idx, mv_off)
    assert np.array_equal(v0, v1) and np.array_equal(p0, p1)
    # and against the oracle on a sample of boards (the tolerance of the bf16 path)
    pick = np.array([0, 1, n // 2, n - 2, n - 1])
    planes = _oracle_planes(spec, bits[pick], scalars[pick])
    ref_s, _ = OnnxOracle(onnx_bytes).run(planes)
    assert np.abs(np.tanh(ref_s[:, 0]) - v1[pick, 0]).max() <= 5e-2


def test_chess_history_mapper_shapes():
    """ChessHistoryMapper (rust/kz-core/src/mapping/chess.rs:25-95, row N4): (7 + N + 1) scalars and 1 + 12 (N + 1) bool
    planes go through the same encode / tower / heads path; planes bit-exact, fp32 within 1e-4, bf16 within 2e-2."""
    spec = netgen.game_spec("chess-hist-2")
    assert (spec.scalar_channels, spec.bool_channels) == (10, 37)
    onnx_bytes = netgen.build_onnx(spec, 2, 64, seed=51)
    bits, scalars, mv_idx, mv_off = netgen.synthetic_positions(spec, 40, seed=52)
    ref_s, ref_p, ref_values, ref_probs = _oracle_packed(spec, onnx_bytes, bits, scalars, mv_idx, mv_off)
    with B200Network(mapper_for(spec), onnx_bytes, 40, precision=PRECISION_FP32) as net:
        planes = net.encode_planes(bits, scalars)
        values, probs = net.evaluate_packed(bits, scalars, mv_idx, mv_off)
    assert np.array_equal(planes.view(np.uint32), _oracle_planes(spec, bits, scalars).view(np.uint32))
    _check_packed(values, probs, ref_values, ref_probs, mv_off, FP32_TOL, FP32_TOL)
    with B200Network(mapper_for(spec), onnx_bytes, 40, precision=PRECISION_BF16) as net:
        values, probs = net.evaluate_packed(bits, scalars, mv_idx, mv_off)
        s, p = net.evaluate_planes(_oracle_planes(spec, bits, scalars))
    assert np.abs(p - ref_p).max() <= BF16_POLICY_TOL
    _check_packed(values, probs, ref_values, ref_probs, mv_off, 5e-2, 1e-2)


def _ataxx7_symmetry_tables():
    """From the reference's golden table (tests/golden/ataxx7_symmetry.json <- python/lib/mapping/ataxx_symmetry.json):
    square_src as AtaxxSymmetry.map_bools moves planes (python/lib/games.py:115-131), policy_map = map_mv."""
    import json

    rows = json.loads((GOLDEN / "ataxx7_symmetry.json").read_text())
    square_src, policy_map = [], []
    for r in rows:
        idx = np.arange(49).reshape(1, 7, 7)
        if r["transpose"]:
            idx = np.transpose(idx, (0, 2, 1))
        if r["flip_x"]:
            idx = idx[:, :, ::-1]
        if r["flip_y"]:
            idx = idx[:, ::-1, :]
        square_src.append(idx.reshape(-1))
        policy_map.append(np.array(r["map_mv"]))
    return np.stack(square_src), np.stack(policy_map), rows


@pytest.mark.parametrize("precision,tol_v,tol_p", [(PRECISION_FP32, FP32_TOL, FP32_TOL), (PRECISION_BF16, 5e-2, 1e-2)])
def test_symmetries_on_the_gpu_match_mapping_on_the_host(precision, tol_v, tol_p):
    """Row N4: kzb_eval_packed_sym == what RandomSymmetryNetwork computes (network/symmetry.rs:41-67,126-148): evaluate
    the MAPPED board, read every original move's probability at the mapped move.  Host side of the comparison: planes
    transformed with the reference's own flags, indices mapped with the reference's own map_mv table, then the oracle."""
    spec = netgen.game_spec("ataxx-7")
    onnx_bytes = netgen.build_onnx(spec, 2, 32, seed=53)
    n = 48
    bits, scalars, mv_idx, mv_off = netgen.synthetic_positions(spec, n, seed=54)
    square_src, policy_map, rows = _ataxx7_symmetry_tables()
    # legal lists only hold indices that are moves (python/lib/mapping/ataxx_valid.txt); the others map to -1
    valid = np.nonzero((policy_map >= 0).all(axis=0))[0].astype(np.uint32)
    assert len(valid) > 400 and (policy_map[:, valid] >= 0).all()
    rng = np.random.default_rng(55)
    for i in range(n):
        k = int(mv_off[i + 1] - mv_off[i])
        mv_idx[mv_off[i]:mv_off[i + 1]] = rng.choice(valid, size=k, replace=False)
    sym = (np.arange(n) % 8).astype(np.uint8)
    planes = _oracle_planes(spec, bits, scalars)  # [n, 1 + 3, 7, 7]
    mapped = planes.copy()
    mapped_idx = mv_idx.copy()
    for i in range(n):
        r = rows[sym[i]]
        b = planes[i, 1:]
        if r["transpose"]:
            b = np.transpose(b, (0, 2, 1))
        if r["flip_x"]:
            b = b[:, :, ::-1]
        if r["flip_y"]:
            b = b[:, ::-1, :]
        mapped[i, 1:] = b
        sl = slice(int(mv_off[i]), int(mv_off[i + 1]))
        mapped_idx[sl] = policy_map[sym[i]][mv_idx[sl]]
    s, p = OnnxOracle(onnx_bytes).run(mapped)
    ref_values, ref_probs = oracle.decode_output(s, p, mapped_idx, mv_off)
    with B200Network(mapper_for(spec), onnx_bytes, n, precision=precision) as net:
        net.set_symmetries(square_src, policy_map)
        values, probs = net.evaluate_packed_sym(bits, scalars, sym, mv_idx, mv_off)
        plain_v, plain_p = net.evaluate_packed(bits, scalars, mv_idx, mv_off)  # a later plain call is not affected
        ident_v, ident_p = net.evaluate_packed_sym(bits, scalars, np.zeros(n, np.uint8), mv_idx, mv_off)
        with pytest.raises(KzbError, match="symmetry index"):
            net.evaluate_packed_sym(bits, scalars, np.full(n, 8, np.uint8), mv_idx, mv_off)
    _check_packed(values, probs, ref_values, ref_probs, mv_off, tol_v, tol_p)
    assert not (rows[0]["transpose"] or rows[0]["flip_x"] or rows[0]["flip_y"])  # symmetry 0 is the identity ...
    assert np.array_equal(policy_map[0][valid], valid)                            # ... on everything that is a move
    assert np.array_equal(ident_v, plain_v) and np.array_equal(ident_p, plain_p)
    assert not np.allclose(plain_p, probs, atol=1e-3)  # the symmetries did change the evaluations of a random net


# ------------------------------------------------------------------------------------------- contract edges
@pytest.mark.parametrize("precision", [PRECISION_FP32, PRECISION_BF16])
def test_rows_independent_of_batch(precision):
    """Result for row i must not depend on the other rows or on `batch` (SURVEY.md 8(b) batch semantics)."""
    spec = netgen.game_spec("chess")
    onnx_bytes = netgen.build_onnx(spec, 2, 32, seed=12)
    bits, scalars, mv_idx, mv_off = netgen.synthetic_positions(spec, 37, seed=13)
    with B200Network(mapper_for(spec), onnx_bytes, 64, precision=precision) as net:
        v_all, p_all = net.evaluate_packed(bits, scalars, mv_idx, mv_off)
        for i in [0, 5, 36]:
            sl = slice(int(mv_off[i]), int(mv_off[i + 1]))
            v1, p1 = net.evaluate_packed(bits[i:i + 1], scalars[i:i + 1], mv_idx[sl], np.array([0, sl.stop - sl.start], np.uint32))
            assert np.array_equal(v1[0], v_all[i])
            assert np.array_equal(p1, p_all[sl])


def test_evaluate_batch_interface_and_terminal_board():
    spec = netgen.game_spec("ataxx-7")
    onnx_bytes = netgen.build_onnx(spec, 2, 32, seed=14)
    bits, scalars, mv_idx, mv_off = netgen.synthetic_positions(spec, 5, seed=15)
    boards = [EncodedBoard(bits[i], scalars[i], mv_idx[mv_off[i]:mv_off[i + 1]]) for i in range(5)]
    boards[2] = EncodedBoard(bits[2], scalars[2], np.zeros(0, np.uint32))  # terminal: no available moves
    with B200Network(mapper_for(spec), onnx_bytes, 8, precision=PRECISION_FP32) as net:
        assert net.max_batch_size() == 8
        evals = net.evaluate_batch(boards)
        single = net.evaluate(boards[3])
    assert len(evals) == 5
    assert evals[2].policy.shape == (0,)  # common.rs:77
    for i, e in enumerate(evals):
        assert -1 < e.values.value < 1 and abs(sum(e.values.wdl) - 1) < 1e-5
        if i != 2:
            assert e.policy.shape == (len(boards[i].policy_indices),) and abs(e.policy.sum() - 1) < 1e-5
    assert np.array_equal(single.policy, evals[3].policy)


def test_errors_match_reference_panics():
    spec = netgen.game_spec("ataxx-7")
    onnx_bytes = netgen.build_onnx(spec, 1, 16, seed=16)
    bits, scalars, mv_idx, mv_off = netgen.synthetic_positions(spec, 9, seed=17)
    with B200Network(mapper_for(spec), onnx_bytes, 8, precision=PRECISION_FP32) as net:
        with pytest.raises(KzbError, match="max_batch_size"):  # cudnn.rs:58
            net.evaluate_packed(bits, scalars, mv_idx, mv_off)
        bad = scalars[:4].copy()
        bad[1, 0] = np.nan  # NaN input -> NaN logits -> the reference panics in softmax (common.rs:110)
        with pytest.raises(KzbError, match="strictly positive"):
            net.evaluate_packed(bits[:4], bad, mv_idx[: mv_off[4]], mv_off[:5])
        # the handle stays usable after an error
        v, p = net.evaluate_packed(bits[:4], scalars[:4], mv_idx[: mv_off[4]], mv_off[:5])
        assert np.isfinite(v).all() and np.isfinite(p).all()
    wrong = Mapper((spec.bool_channels + 1, 7, 7), spec.scalar_channels, (spec.policy_size,))
    with pytest.raises(KzbError, match="Input shape mismatch"):  # common.rs:171-174
        B200Network(wrong, onnx_bytes, 8)
    wrong = Mapper((spec.bool_channels, 7, 7), spec.scalar_channels, (spec.policy_size + 1,))
    with pytest.raises(KzbError, match="policy shape"):  # common.rs:182
        B200Network(wrong, onnx_bytes, 8)


def test_bf16_rejects_boards_wider_than_255_squares():
    """The bf16 row kernels take boards of up to 255 x 255 squares: a larger board is refused when the network is created, with a
    message that points to the fp32 path, which does create it."""
    spec = netgen.game_spec("go-256")
    onnx_bytes = netgen.build_onnx(spec, 1, 8, seed=18)
    with pytest.raises(KzbError, match="precision=fp32"):
        B200Network(mapper_for(spec), onnx_bytes, 1, precision=PRECISION_BF16)
    with B200Network(mapper_for(spec), onnx_bytes, 1, precision=PRECISION_FP32) as net:
        assert net.info().conv_mode == -1


@pytest.mark.parametrize("game", ["chess", "ataxx-7", "go-9"])
def test_bf16_nan_inputs_are_reported_not_emitted(game):
    """The tensor-core paths (whole-tower + fused heads for chess / ataxx, per-layer for go) must surface NaN logits as an
    error like the reference's softmax assert (common.rs:110), never as NaN probabilities."""
    spec = netgen.game_spec(game)
    onnx_bytes = netgen.build_onnx(spec, 2, 64, seed=61)
    bits, scalars, mv_idx, mv_off = netgen.synthetic_positions(spec, 9, seed=62)
    bad = scalars.copy()
    bad[4, 0] = np.nan
    with B200Network(mapper_for(spec), onnx_bytes, 16, precision=PRECISION_BF16) as net:
        with pytest.raises(KzbError, match="strictly positive"):
            net.evaluate_packed(bits, bad, mv_idx, mv_off)
        v, p = net.evaluate_packed(bits, scalars, mv_idx, mv_off)  # the handle stays usable
        assert np.isfinite(v).all() and np.isfinite(p).all()


def test_concurrent_instances_match(tmp_path):
    """Pattern of rust/kz-misc/src/bin/test_concurrent.rs:32-145: several executors on one device, each in
    its own thread, must keep reproducing the same outputs."""
    import threading

    spec = netgen.game_spec("chess")
    onnx_bytes = netgen.build_onnx(spec, 2, 32, seed=18)
    bits, scalars, mv_idx, mv_off = netgen.synthetic_positions(spec, 48, seed=19)
    with B200Network(mapper_for(spec), onnx_bytes, 48) as net:
        ref_v, ref_p = net.evaluate_packed(bits, scalars, mv_idx, mv_off)
    failures = []

    def worker():
        try:
            with B200Network(mapper_for(spec), onnx_bytes, 48) as n2:
                for _ in range(10):
                    v, p = n2.evaluate_packed(bits, scalars, mv_idx, mv_off)
                    if not (np.array_equal(v, ref_v) and np.array_equal(p, ref_p)):
                        failures.append("mismatch")
        except Exception as e:  # noqa: BLE001
            failures.append(repr(e))

    threads = [threading.Thread(target=worker) for _ in range(4)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not failures, failures


# ------------------------------------------------------------------------------------------- boundary loose ends (VERDICT r01)
@pytest.mark.parametrize("game,depth,ch", [("chess", 2, 64), ("ataxx-7", 2, 32), ("go-9", 2, 64)])
def test_net_created_from_raw_weights_equals_the_onnx_net(game, depth, ch):
    """kzb_net_create (weights the caller already holds: the reference's load_graph stays untouched and hands the optimised Graph's
    constants over, network/cudnn.rs:29-43) must give the network kzb_net_create_from_onnx builds from the file."""
    from helpers import raw_weights_from_netgen

    spec = netgen.game_spec(game)
    weights = {}
    onnx_bytes = netgen.build_onnx(spec, depth, ch, seed=71, weights_out=weights)
    bits, scalars, mv_idx, mv_off = netgen.synthetic_positions(spec, 21, seed=72)
    for precision, tol in ((PRECISION_FP32, 2e-6), (PRECISION_BF16, 2e-3)):
        with B200Network(mapper_for(spec), onnx_bytes, 24, precision=precision) as a:
            va, pa = a.evaluate_packed(bits, scalars, mv_idx, mv_off)
        with B200Network(mapper_for(spec), raw_weights_from_netgen(spec, depth, weights), 24, precision=precision) as b:
            assert (b.info().channels, b.info().depth, b.info().policy_len) == (ch, depth, spec.policy_size)
            vb, pb = b.evaluate_packed(bits, scalars, mv_idx, mv_off)
        # not bit-identical: the final BN reaches this path as an f32 affine, the ONNX path folds it in f64
        assert np.abs(va - vb).max() <= tol and np.abs(pa - pb).max() <= tol


def test_go_with_territory_planes_13_channels():
    """GoStdMapper::new(size, true), what the reference's self-play SERVER constructs (rust/kz-selfplay/src/server/server.rs:193;
    mapping/go.rs:46-59): 6 scalar + 7 bool planes = 13 input channels.  Same encode / tower / heads path as the 10-channel form."""
    spec = netgen.game_spec("go-9-territory")
    assert (spec.scalar_channels, spec.bool_channels, spec.input_channels) == (6, 7, 13)
    onnx_bytes = netgen.build_onnx(spec, 3, 64, seed=81)
    bits, scalars, mv_idx, mv_off = netgen.synthetic_positions(spec, 33, seed=82)
    ref_s, ref_p, ref_values, ref_probs = _oracle_packed(spec, onnx_bytes, bits, scalars, mv_idx, mv_off)
    with B200Network(mapper_for(spec), onnx_bytes, 40, precision=PRECISION_FP32) as net:
        planes = net.encode_planes(bits, scalars)
        values, probs = net.evaluate_packed(bits, scalars, mv_idx, mv_off)
    assert np.array_equal(planes.view(np.uint32), _oracle_planes(spec, bits, scalars).view(np.uint32))
    _check_packed(values, probs, ref_values, ref_probs, mv_off, FP32_TOL, FP32_TOL)
    with B200Network(mapper_for(spec), onnx_bytes, 40, precision=PRECISION_BF16) as net:
        values, probs = net.evaluate_packed(bits, scalars, mv_idx, mv_off)
        s, p = net.evaluate_planes(_oracle_planes(spec, bits, scalars))
    assert np.abs(p - ref_p).max() <= BF16_POLICY_TOL
    _check_packed(values, probs, ref_values, ref_probs, mv_off, 5e-2, 1e-2)


@pytest.mark.parametrize("game,depth,ch", [("chess", 3, 64), ("go-9", 3, 64)])
def test_partial_batches_replay_their_own_cuda_graph(game, depth, ch, monkeypatch):
    """Batch sizes that keep coming back get a CUDA graph of their own (the role of MultiBatchNetwork, network/multibatch.rs:19-35,
    without padding rows): first call direct launches, second call captures + launches, third call replays -- all bit-identical to
    each other and to a network that never uses graphs; interleaved sizes keep their own graphs."""
    spec = netgen.game_spec(game)
    onnx_bytes = netgen.build_onnx(spec, depth, ch, seed=91)
    bits, scalars, mv_idx, mv_off = netgen.synthetic_positions(spec, 64, seed=92)

    def part(n):
        return bits[:n], scalars[:n], mv_idx[:mv_off[n]], mv_off[:n + 1]

    monkeypatch.setenv("KZB_NO_GRAPH", "1")
    with B200Network(mapper_for(spec), onnx_bytes, 64) as net:
        want = {n: net.evaluate_packed(*part(n)) for n in (64, 37, 5)}
    monkeypatch.setenv("KZB_NO_GRAPH", "0")
    with B200Network(mapper_for(spec), onnx_bytes, 64) as net:
        for n in (37, 64, 37, 5, 37, 64, 5, 5, 37):
            v, p = net.evaluate_packed(*part(n))
            assert np.array_equal(v, want[n][0]) and np.array_equal(p, want[n][1]), n
