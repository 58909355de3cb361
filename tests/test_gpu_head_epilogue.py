"""The fused head's arg-max epilogue on logits it cannot get wrong by accident, and the head's GEMM off the presets.

Crafted logits.  The activations are one-hot per cell (feat[b, k, cell] = 1 iff k == pat[b, cell]) and the weights are
exact in the operand type, so the convolution output is W[c, pat] exactly and the logit is fl32(W[c, pat] + bias[c]),
known bit for bit on the host.  The weights carry the coarse structure (a pattern either keeps a window position live
or pushes it 256 down), the fp32 bias the fine one: ulp-level near-ties of the sigmoid just below +-6 and above 6,
steps of fl(m + 1e-3) +- 1 ulp around the epilogue's sure-step threshold, saturated runs, the denormal and zero tail
below -87, NaN and +-inf.  Patterns cut every window at different places, so maxima and ties fall at every phase of
an 8-column group, a sub-warp's run, a 128- or 256-channel accumulator tile and a piece.  The speculative hot loop
(`emit=False`) must then give exactly numpy's arg-max of the emitted sigmoid (first maximum, first NaN) — the answer of
the exact per-column rule that an emitting call runs everywhere.

Random data at other geometries.  1 x 1, 3 x 5 and 13 x 13 windows, 6K > 256, E = 0 and 1, grids whose cell count is
not a multiple of 32 (or, 16-bit path, is odd), every input-channel count class; the logits against a float64
convolution within a bound derived from the operation, everything downstream bit-exact on the emitted head.
"""
import numpy as np
import pytest
import torch

from oracle import c_oracle, ppn_oracle as O
from tests.test_gpu_head import check_against_emitted, geometry, make_layer
from tests.test_gpu_parity import _random_tree, assert_packed_equals_oracle, bits, parser_for

pytestmark = pytest.mark.gpu

F32 = np.float32
SUPPRESS = F32(-256.0)                 # weight of a pattern's dead window positions: exact in every operand type


def ulps(v, n):
    """v moved by n float32 steps along its bit pattern (v > 0: n > 0 is up; v < 0: n > 0 is down)."""
    return (F32(v).view(np.int32) + np.int32(n)).view(F32)


# gaps of a rising stream: ("ulp", n) = n ulps up, ("thr", n) = fl(v + 1e-3) moved n ulps (the sure-step threshold,
# kSureStep, sits right there), a float = fl(v + gap)
GAPS_TIE = [("ulp", 1), ("ulp", 3), 1e-5, 1.5e-5, 2e-5, 2.4e-5, 3e-5, 1e-4, ("thr", -1), ("thr", 0), ("thr", 1), 2e-3, 5e-4]
GAPS_SAT = [("thr", -1), ("thr", 0), ("thr", 1), 1.2e-3, 1.5e-3, 2e-3, 2.5e-3, 5e-4, ("ulp", 2)]


def stream(start, gaps, n, phase):
    v, out = F32(start), np.empty(n, F32)
    for i in range(n):
        out[i] = v
        gap = gaps[(i + phase) % len(gaps)]
        if isinstance(gap, tuple):
            v = ulps(v, gap[1] if v > 0 else -gap[1]) if gap[0] == "ulp" else \
                ulps(F32(v + F32(1e-3)), gap[1] if v > 0 else -gap[1])
        else:
            v = F32(v + F32(gap))
    return out


FAMILIES = ["below6", "above6", "lower_tail", "cross6", "saturated", "nan", "inf", "rising", "falling", "sawtooth",
            "near_minus6"]


def window_values(fam, S, ei, first_channel, rng):
    """The fp32 bias of one limb window of family `fam`."""
    pos = np.arange(S)
    if fam in ("below6", "cross6", "near_minus6"):
        span = float(stream(5.0, GAPS_TIE, S, ei)[-1]) - 5.0
        start = {"below6": 6.0 - span - 1e-4, "cross6": 6.0 - span / 2, "near_minus6": -6.0 - span / 2}[fam]
        return stream(start, GAPS_TIE, S, ei)
    if fam == "above6":                                  # sigmoids of 10.5 .. 12 tie over steps of ~1e-3
        return stream(10.5, GAPS_SAT, S, ei)
    if fam == "lower_tail":                              # denormal sigmoids above -88.7, zero below
        return (np.linspace(-110.0, -87.0, S) + rng.uniform(0, 1e-3, S)).astype(F32)
    if fam == "saturated":                               # (6, 20]: sigmoid 1.0 from 16.7 on
        v = rng.uniform(6.0, 20.0, S).astype(F32)
        v[: S // 2] = np.sort(v[: S // 2])
        return v
    if fam == "rising":
        return (np.linspace(-5.0, 5.0, S) + 2.0 ** -7).astype(F32)
    if fam == "falling":
        return (np.linspace(5.0, -5.0, S) + 2.0 ** -7).astype(F32)
    if fam == "sawtooth":                                # every tooth starts below -6 and steps into range
        return (-9.0 + (pos % 13) * 1.05).astype(F32)
    v = rng.uniform(-3.0, 3.0, S).astype(F32)
    if fam == "nan":
        # two NaNs of different sign and payload, the first one wins: where a payload survives the sigmoid (whose
        # 1 / (1 + exp(-x)) flips its sign), the later NaN's bits are the larger ones, so keying NaN by those bits fails
        nan_first = F32(np.uint32(0xFFC00001).view(F32))
        nan_later = F32(np.uint32(0x7FC00001).view(F32))
        # a NaN where the window meets a 128-channel boundary (a tile, hence a piece, starts there) when it has one
        at_tile = [p for p in range(S) if (first_channel + p) % 128 == 0]
        first, second = [(0, S - 1), (S - 1, None), (at_tile[0] if at_tile else S // 2, S - 2)][ei % 3]
        if second is not None and second > first:
            v[second] = nan_later
        v[first] = nan_first
        return v
    if fam == "inf":
        kind = ei % 3
        if kind == 0:                                    # a saturated 1.0 before +inf's 1.0: the earlier one wins
            v[S // 3] = 30.0
            v[(2 * S) // 3] = np.inf
            v[S - 1] = -np.inf
        elif kind == 1:
            v[:] = -np.inf                               # sigmoid 0 everywhere: position 0
        else:
            v[0] = np.inf
            v[1::5] = -np.inf
        return v
    raise ValueError(fam)


def round_operand(x, operand):
    """x rounded to a value the operand type holds exactly (11 significant bits for TF32, fp16 or bf16's own)."""
    t = torch.from_numpy(np.ascontiguousarray(x, F32))
    if operand == "f16":
        return t.half().float().numpy()
    if operand == "bf16":
        return t.bfloat16().float().numpy()
    b = t.view(torch.int32)
    return ((b + 0x1000) & ~0x1FFF).view(torch.float32).numpy()


def crafted_layer(g, B, Cin, operand, with_bias, seed):
    """-> feat [B, Cin, H, W], weight [C, Cin], bias [C] or None (numpy float32) and the exact logits [B, C, H*W]."""
    rng = np.random.default_rng(seed)
    K6, S, C, HW = 6 * g.K, g.S, 6 * g.K + g.S * g.E, g.H * g.W
    bias = np.empty(C, F32)
    W = np.zeros((C, Cin), F32)
    bias[:K6] = rng.normal(0.0, 1.0, K6)
    bias[:2 * g.K] += 1.0
    W[:K6] = rng.integers(-24, 25, (K6, Cin)) / 16.0       # decode channels: coarse per-pattern structure
    for ei in range(g.E):
        c0 = K6 + ei * S
        bias[c0:c0 + S] = window_values(FAMILIES[ei % len(FAMILIES)], S, ei, c0, rng)
        for k in range(1, Cin):                          # pattern 0 keeps the whole window live
            if k == 1:
                a, b = 0, max(1, S // 2)
            elif k == 2:
                a, b = S // 2, S
            else:
                a = int(rng.integers(0, S))
                b = int(rng.integers(a + 1, S + 1))
            W[c0:c0 + a, k] = SUPPRESS
            W[c0 + b:c0 + S, k] = SUPPRESS
    if not with_bias:                                    # the whole logit in the weights: coarse, finite values only
        full = W + bias[:, None]
        full[np.isnan(full)] = 17.5
        full[np.isposinf(full)] = 1000.0
        full[np.isneginf(full)] = -1000.0
        W, bias = round_operand(full, operand), None
    pat = rng.integers(0, Cin, (B, HW))
    pat[:, :Cin] = np.arange(min(Cin, HW))               # every pattern occurs (where the grid has room)
    rng.shuffle(pat, axis=1)
    feat = np.zeros((B, Cin, HW), F32)
    np.put_along_axis(feat, pat[:, None, :], F32(1.0), axis=1)
    logits = W[:, pat] + (bias[:, None, None] if bias is not None else F32(-0.0))      # [C, B, HW], fl32 sums
    return (feat.reshape(B, Cin, g.H, g.W), W, bias, np.ascontiguousarray(logits.transpose(1, 0, 2)))


def assert_logits_exact(got, want):
    got = got.reshape(want.shape)
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan), "NaN logits where the exact sum has none, or the other way round"
    g, w = bits(got[~nan]), bits(want[~nan])
    g = np.where(g == 0x80000000, 0, g)                  # +-0: the sign of an exact zero sum is not specified
    w = np.where(w == 0x80000000, 0, w)
    bad = int((g != w).sum())
    assert bad == 0, f"{bad} logits differ from fl32(W[c, pat] + bias[c])"


def parse_ref(parser, g, feat, weight, bias, head, operand):
    """c_oracle on the emitted head, or None where the fused parse does not take the shape."""
    from pytorch_pose_proposal_network_b200 import _lib
    try:
        parser.parse_features(feat, weight, bias, operand=operand)
    except _lib.PPNError as e:
        if e.code != -2:                                 # PPN_E_UNSUPPORTED
            raise
        return None
    return c_oracle.parse_batch(head.cpu().numpy(), g, n_threads=8)


@pytest.mark.parametrize("with_bias", [True, False], ids=["bias", "no_bias"])
@pytest.mark.parametrize("name,B", [("native", 1), ("cfg2", 136)], ids=["native_B1", "cfg2_B136"])
@pytest.mark.parametrize("operand,acc", [("tf32", 256), ("f16", 256), ("bf16", 256), ("f16", 128), ("bf16", 128)])
def test_crafted_logits_every_epilogue_width(operand, acc, name, B, with_bias):
    """B = 1 of the reference's shape: 5 cell tiles, every tile's channel tiles spread over the SMs, pieces of one
    window from different CTAs meet in the key maxima.  cfg2 at B = 136: more cell tiles than SMs, so the persistent
    loop runs and the accumulator phases wrap."""
    from pytorch_pose_proposal_network_b200 import _lib
    g = geometry(name)
    parser = parser_for(g)
    Cin = 32 if operand == "tf32" else 64
    feat, W, bias, want = crafted_layer(g, B, Cin, operand, with_bias, seed=len(name) * 100 + len(operand) * 10 + with_bias)
    feat = torch.from_numpy(feat).cuda()
    weight = torch.from_numpy(W).cuda()
    bias = torch.from_numpy(bias).cuda() if bias is not None else None
    first = None
    try:
        _lib.tune(head_acc=acc)
        for subs in (1, 2, 4, 6):
            _lib.tune(head_subs=subs)
            dec, amax, logits, head = parser.head_gemm_argmax(feat, weight, bias, emit=True, operand=operand)
            torch.cuda.synchronize()
            if first is None:
                assert_logits_exact(logits.cpu().numpy(), want)
                check_against_emitted(g, parser, dec, amax, logits, head)
                ref = parse_ref(parser, g, feat, weight, bias, head, operand)
                first = (dec, amax, logits.view(torch.int32), head.view(torch.int32))
            else:
                assert torch.equal(logits.view(torch.int32), first[2]) and torch.equal(head.view(torch.int32), first[3]), subs
                assert torch.equal(amax.view(torch.int16), first[1].view(torch.int16)), f"emitting call, subs={subs}"
            # the production path: no emit buffers, the speculative hot loop
            dec2, amax2, _, _ = parser.head_gemm_argmax(feat, weight, bias, operand=operand)
            torch.cuda.synchronize()
            miss = int((amax2.view(torch.int16) != first[1].view(torch.int16)).sum())
            assert miss == 0, f"subs={subs}: {miss} arg-max entries differ from numpy's arg-max of the emitted sigmoid"
            assert torch.equal(dec2.view(torch.int32), first[0].view(torch.int32)), f"subs={subs}: decode planes"
            if ref is not None:
                packed = parser.parse_features(feat, weight, bias, operand=operand).numpy()
                torch.cuda.synchronize()
                assert_packed_equals_oracle(packed, ref, B)
    finally:
        _lib.tune(head_subs=0, head_acc=256)


# ---------------------------------------------------------------------------------------------------------------
# random data off the presets
# ---------------------------------------------------------------------------------------------------------------
def _config(name):
    from pytorch_pose_proposal_network_b200.config import PPNConfig
    mpii = PPNConfig.mpii16
    if name == "k44":                                   # 6K = 264: the decode planes cross a 256-channel tile
        graphs, E = _random_tree(np.random.default_rng(44), 44)
        return PPNConfig(K=44, E=E, insize=(128, 128), outsize=(8, 8), local_grid_size=(3, 3), directed_graphs=graphs)
    return {
        "window1x1": lambda: mpii(outsize=(12, 12), local_grid_size=(1, 1)),
        "window3x5": lambda: mpii(outsize=(12, 12), local_grid_size=(3, 5)),
        "window13x13": lambda: mpii(insize=(256, 256), outsize=(16, 16), local_grid_size=(13, 13)),
        "e0": lambda: PPNConfig(K=1, E=0, directed_graphs=(), insize=(160, 160), outsize=(10, 10), local_grid_size=(5, 5)),
        "e1": lambda: PPNConfig(K=2, E=1, directed_graphs=(((0,), (1,)),), insize=(32, 32), outsize=(2, 2),
                                local_grid_size=(3, 3)),
        "grid10x10": lambda: mpii(insize=(160, 160), outsize=(10, 10), local_grid_size=(9, 9)),
        "grid2x2": lambda: mpii(insize=(64, 64), outsize=(2, 2), local_grid_size=(3, 3)),
        "grid5x7": lambda: mpii(insize=(80, 112), outsize=(5, 7), local_grid_size=(3, 5)),
    }[name]()


GEOMETRIES = ["window1x1", "window3x5", "window13x13", "k44", "e0", "e1", "grid10x10", "grid2x2", "grid5x7"]
CIN = {"tf32": [32, 96, 160, 1024], "f16": [64, 192, 448, 512], "bf16": [64, 192, 448, 512]}
# operand rounding: TF32 may drop the low 13 mantissa bits of an fp32 operand (chopping: 2^-10 relative); fp16 and
# bf16 operands are rounded to nearest by the pack kernel
U_OP = {"tf32": 2.0 ** -10, "f16": 2.0 ** -11, "bf16": 2.0 ** -8}


def conv64(feat, weight, bias):
    out = torch.einsum("bkn,ck->bcn", feat.double().flatten(2), weight.double())
    return out + bias.double()[None, :, None]


@pytest.mark.parametrize("operand", ["tf32", "f16", "bf16"])
@pytest.mark.parametrize("geom", GEOMETRIES)
def test_random_geometries_and_input_channels(geom, operand):
    from pytorch_pose_proposal_network_b200 import _lib
    from pytorch_pose_proposal_network_b200.parser import PoseParser
    cfg = _config(geom)
    g = O.Geometry.of(cfg)
    parser = PoseParser(cfg)
    Cin = CIN[operand][(GEOMETRIES.index(geom) + (operand == "bf16")) % 4]
    B = 3
    feat, weight, bias = make_layer(g, B, Cin, seed=GEOMETRIES.index(geom) * 10 + len(operand))
    if operand == "tf32" and cfg.HW % 4:
        with pytest.raises(_lib.PPNError):               # the TF32 path reads 16-byte rows of cells
            parser.head_gemm_argmax(feat, weight, bias, emit=True, operand=operand)
        return
    dec, amax, logits, head = parser.head_gemm_argmax(feat, weight, bias, emit=True, operand=operand)
    torch.cuda.synchronize()
    # |error| <= A * (2 u_op + Cin 2^-23) with A = conv(|x|, |w|) + |bias|: two rounded operands per product, then the
    # fp32 sum of Cin products and the bias (2^-23 per addition: the tensor core's additions need not round to
    # nearest); fp16 adds an absolute 2^-25 per subnormal operand.  A dropped or repeated K block, or a tile read at
    # the wrong stride, is far outside.
    ref = conv64(feat, weight, bias)
    A = conv64(feat.abs(), weight.abs(), bias.abs())
    bound = A * (2 * U_OP[operand] + Cin * 2.0 ** -23) + 1e-30
    if operand == "f16":
        bound = bound + 2.0 ** -24 * (weight.double().abs().sum(1)[None, :, None] + feat.double().abs().sum(1).flatten(1)[:, None, :])
    err = (logits.double().flatten(2) - ref).abs()
    worst = float((err / bound).max())
    assert worst <= 1.0, f"logit error reaches {worst:.2f} x the bound (Cin={Cin})"
    check_against_emitted(g, parser, dec, amax, logits, head)
    dec2, amax2, _, _ = parser.head_gemm_argmax(feat, weight, bias, operand=operand)
    torch.cuda.synchronize()
    assert torch.equal(dec2.view(torch.int32), dec.view(torch.int32))
    assert torch.equal(amax2.view(torch.int16), amax.view(torch.int16))
    oracle = parse_ref(parser, g, feat, weight, bias, head, operand)
    if oracle is not None:
        packed = parser.parse_features(feat, weight, bias, operand=operand).numpy()
        torch.cuda.synchronize()
        assert_packed_equals_oracle(packed, oracle, B)


@pytest.mark.parametrize("operand", ["f16", "bf16"])
def test_head16_rejects_more_than_512_input_channels(operand):
    from pytorch_pose_proposal_network_b200 import _lib
    g = geometry("cfg1")
    parser = parser_for(g)
    feat, weight, bias = make_layer(g, 1, 576, seed=3)   # nine 64-wide K blocks: the resident A tile holds eight
    with pytest.raises(_lib.PPNError):
        parser.head_gemm_argmax(feat, weight, bias, operand=operand)
