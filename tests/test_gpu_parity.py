"""GPU parity tests proper: every call goes through the C ABI (ctypes) of libavsr_b200.so and is compared with
the CPU oracle / the committed golden vectors of the reference.

Tolerances are pinned at <= 4x the errors a B200 produced in round 2 (every comparison prints its observed value and
appends it to gpurun_out/parity_observed.jsonl; the run the bounds come from is profiles/r02_parity_observed.txt).
Outputs have rms ~1; errors are max-abs / rms against the fp64 reference:
  fp32 path  (CUDA-core FMA):       observed 8.6e-6 / 6.3e-7 on the 12-layer encoder -- fp32 summation-order noise only
  tf32 path  (tcgen05 kind::tf32):  observed 4.7e-3 / 3.1e-4 (12 layers), 6.4e-4 / 8.9e-5 (2 layers); operands rounded
                                    to TF32 (10-bit mantissa, RN), fp32 accumulate -- the arithmetic class of PyTorch's
                                    own `allow_tf32` GPU path.
  f16 path   (tcgen05 kind::f16):   observed 4.5e-3 / 3.1e-4 (12 layers), 5.8e-4 / 8.9e-5 (2 layers): IEEE half operands
                                    carry the same 10-bit mantissa (values saturate at +-65504, see the range tests),
                                    fp32 accumulate; residual stream / LN / softmax stay fp32.
"""
import math

import numpy as np
import pytest
import torch

from helpers import err_stats, load_case, record
from oracle import conformer_oracle as O

pytestmark = pytest.mark.gpu

PRECS = ["fp32", "tf32", "f16"]
# (max-abs, rms) vs the fp64 reference on the 12-layer encoder / on encoders of <= 2 layers
TOL_ENC = {"fp32": (3.5e-5, 2.5e-6), "tf32": (1.8e-2, 1.2e-3), "f16": (1.8e-2, 1.2e-3)}
TOL_ENC_SHALLOW = {"fp32": (8e-6, 8e-7), "tf32": (2.5e-3, 3.5e-4), "f16": (2.5e-3, 3.5e-4)}
TOL_OP = {"fp32": 8e-6, "tf32": 4e-3, "f16": 1.5e-3}                           # single GEMMs, relative to output scale
TOL_ATT = {"fp32": 4e-6, "tf32": 4e-3, "f16": 4e-3}                            # attention context, relative
TOL_TAP = {"fp32": 1e-6, "tf32": 3.5e-5, "f16": 3.5e-5}                        # layer-0 residual stages, relative
TOL_BATCH = {"fp32": 1e-5, "tf32": 2e-3, "f16": 2e-3}                          # same utterance in another batch slot
TOL_EDGE = {"fp32": 1e-5, "tf32": 1.5e-4, "f16": 1.5e-4}                       # 1-layer edge shapes, max-abs


def tol_enc(prec, num_blocks):
    return TOL_ENC[prec] if num_blocks > 2 else TOL_ENC_SHALLOW[prec]


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "run with gpurun"
    import __graft_entry__ as g
    g.build()
    return torch.device("cuda:0")


def _encoder(case, dev, prec):
    from auto_avsr_b200 import ConformerEncoder
    cfg = case["cfg"]
    enc = ConformerEncoder(attention_dim=cfg["d_model"], attention_heads=cfg["n_heads"],
                           linear_units=cfg["linear_units"], num_blocks=cfg["num_blocks"],
                           cnn_module_kernel=cfg["cnn_kernel"])
    enc.load_state_dict(case["sd"], strict=True)
    enc = enc.to(dev).eval()
    enc.precision = prec
    enc.graph_after = 1          # capture the CUDA graph at first sight (default: after the shape was seen 3 times)
    return enc


def _mask(case, dev):
    return O.non_pad_mask(case["lengths"]).unsqueeze(1).to(dev) if case["masked"] else None


# ------------------------------------------------------------------------------------------ unit ops
def test_layernorm(dev):
    from auto_avsr_b200 import ops
    g = torch.Generator().manual_seed(1)
    for rows, d in [(1, 768), (37, 768), (1600, 768), (5, 128), (9, 1024), (3, 4)]:
        x = torch.randn(rows, d, generator=g) * 3 + 0.5
        w, b = torch.rand(d, generator=g) + 0.5, torch.randn(d, generator=g) * 0.1
        y = ops.layernorm(x.to(dev), w.to(dev), b.to(dev)).cpu()
        ref = O.layer_norm(x.double(), w.double(), b.double())
        assert err_stats(y, ref)[0] < 5e-6 * max(1.0, ref.abs().max().item()), (rows, d)
    # constant rows: variance 0 -> eps 1e-12 keeps it finite and equal to beta
    x = torch.full((2, 768), 3.25)
    y = ops.layernorm(x.to(dev), torch.ones(768, device=dev), torch.full((768,), 0.5, device=dev)).cpu()
    assert torch.allclose(y, torch.full_like(y, 0.5))


def test_sinusoid_table(dev):
    from auto_avsr_b200 import ops
    for T, d in [(1, 768), (7, 16), (100, 768), (400, 768)]:
        pe = ops.rel_sinusoid_table(T, d, dev).cpu()
        ref = O.rel_sinusoid_table(T, d, torch.float32)
        assert pe.shape == ref.shape
        # a 1-ulp difference in the fp32 frequency exp() moves the fp32 argument rel*w by up to T * 6e-8
        assert err_stats(pe, ref)[0] < 1e-6 + 1.5e-7 * T, (T, d)


@pytest.mark.parametrize("prec", PRECS)
def test_linear(dev, prec):
    from auto_avsr_b200 import ops
    g = torch.Generator().manual_seed(2)
    for rows, n, k in [(200, 768, 768), (129, 3072, 768), (77, 768, 3072), (1, 128, 256), (300, 256, 128),
                       (1600, 768, 768)]:
        x = torch.randn(rows, k, generator=g)
        w = (torch.rand(n, k, generator=g) * 2 - 1) / math.sqrt(k)
        b = torch.randn(n, generator=g) * 0.1
        r = torch.randn(rows, n, generator=g)
        ref = x.double() @ w.double().T + b.double()
        scale = ref.abs().max().item()
        y = ops.linear(x.to(dev), w.to(dev), b.to(dev), precision=prec).cpu()
        record("linear", (prec, rows, n, k), err_stats(y, ref)[0] / scale, TOL_OP[prec])
        assert err_stats(y, ref)[0] < TOL_OP[prec] * scale, (rows, n, k)
        y = ops.linear(x.to(dev), w.to(dev), b.to(dev), relu=True, precision=prec).cpu()
        assert err_stats(y, ref.clamp_min(0))[0] < TOL_OP[prec] * scale
        y = ops.linear(x.to(dev), w.to(dev), None, residual=r.to(dev), alpha=0.5, precision=prec).cpu()
        assert err_stats(y, r.double() + 0.5 * (ref - b.double()))[0] < TOL_OP[prec] * scale


@pytest.mark.parametrize("prec", PRECS)
def test_pointwise_glu(dev, prec):
    from auto_avsr_b200 import ops
    g = torch.Generator().manual_seed(3)
    for rows, C in [(150, 768), (33, 128)]:
        x = torch.randn(rows, C, generator=g)
        w = (torch.rand(2 * C, C, 1, generator=g) * 2 - 1) / math.sqrt(C)
        b = torch.randn(2 * C, generator=g) * 0.1
        y = ops.pointwise_glu(x.to(dev), w.to(dev), b.to(dev), prec).cpu()
        full = x.double() @ w.squeeze(-1).double().T + b.double()
        ref = full[:, :C] * torch.sigmoid(full[:, C:])
        record("pointwise_glu", (prec, rows, C), err_stats(y, ref)[0] / max(1.0, ref.abs().max().item()), TOL_OP[prec])
        assert err_stats(y, ref)[0] < TOL_OP[prec] * max(1.0, ref.abs().max().item()), (rows, C)


def test_dwconv_bn_silu(dev):
    from auto_avsr_b200 import ops
    g = torch.Generator().manual_seed(4)
    for B, T, C, K in [(3, 37, 128, 31), (1, 5, 768, 31), (2, 100, 768, 31), (1, 23, 128, 7), (2, 64, 64, 1)]:
        x = torch.randn(B, T, C, generator=g)
        w = torch.randn(C, 1, K, generator=g) / math.sqrt(K)
        b, bw, bb = (torch.randn(C, generator=g) * 0.1, torch.rand(C, generator=g) + 0.5,
                     torch.randn(C, generator=g) * 0.1)
        mean, var = torch.randn(C, generator=g) * 0.1, torch.rand(C, generator=g) + 0.5
        y = ops.dwconv_bn_silu(*[t.to(dev) for t in (x, w, b, bw, bb, mean, var)]).cpu()
        conv = torch.nn.functional.conv1d(x.double().transpose(1, 2), w.double(), b.double(), padding=(K - 1) // 2,
                                          groups=C)
        h = (conv - mean.double()[:, None]) / torch.sqrt(var.double()[:, None] + 1e-5) * bw.double()[:, None] \
            + bb.double()[:, None]
        ref = (h * torch.sigmoid(h)).transpose(1, 2)
        assert err_stats(y, ref)[0] < 1e-5 * max(1.0, ref.abs().max().item()), (B, T, C, K)


@pytest.mark.parametrize("prec", PRECS)
def test_relpos_attention(dev, prec):
    from auto_avsr_b200 import ops
    g = torch.Generator().manual_seed(5)
    for B, T, H, lengths in [(3, 37, 2, [37, 29, 18]), (1, 100, 12, None), (2, 130, 3, [130, 1]),
                             (2, 9, 2, [0, 9]), (1, 1, 2, None), (2, 257, 2, [257, 200])]:
        D = H * 64
        q, k, v = (torch.randn(B, T, D, generator=g) for _ in range(3))
        p = torch.randn(2 * T - 1, D, generator=g)
        u, vb = torch.randn(H, 64, generator=g) * 0.3, torch.randn(H, 64, generator=g) * 0.3
        ln = None if lengths is None else torch.tensor(lengths, dtype=torch.int32, device=dev)
        ctx = ops.relpos_attention(q.to(dev), k.to(dev), v.to(dev), p.to(dev), u.to(dev), vb.to(dev), ln, H,
                                   precision=prec).cpu()

        def heads(t):
            return t.double().view(B, T, H, 64).transpose(1, 2)
        scores = O.rel_attention_scores(heads(q), heads(k), p.double().view(2 * T - 1, H, 64).transpose(0, 1),
                                        u.double(), vb.double())
        if lengths is not None:
            pad = torch.arange(T)[None, :] >= torch.tensor(lengths)[:, None]
            scores = scores.masked_fill(pad[:, None, None, :], float("-inf"))
        attn = torch.softmax(scores, dim=-1)
        attn = torch.where(torch.isnan(attn), torch.zeros_like(attn), attn)       # fully masked rows -> 0
        ref = (attn @ heads(v)).transpose(1, 2).reshape(B, T, D)
        tol = TOL_ATT[prec]                        # scores of randn q,k have sd ~8: 11-bit operand rounding shows
        record("relpos_attention", (prec, B, T, H, lengths), err_stats(ctx, ref)[0] / max(1.0, ref.abs().max().item()), tol)
        assert err_stats(ctx, ref)[0] < tol * max(1.0, ref.abs().max().item()), (B, T, H, lengths)


def test_relpos_attention_moving_reference_maximum(dev):
    """Scores with a wide spread (q, k x3: logits of sd ~9, hundreds of rows whose later key tiles exceed the running
    reference maximum by more than 2^8) drive the fp16 kernel's rescale-O-in-tensor-memory path in divergent
    patterns (some rows of a warp move, others do not); S2-sized so that every SM holds two CTAs."""
    from auto_avsr_b200 import ops
    g = torch.Generator().manual_seed(15)
    B, T, H = 4, 400, 12
    D = H * 64
    q, k = torch.randn(B, T, D, generator=g) * 3, torch.randn(B, T, D, generator=g) * 3
    v = torch.randn(B, T, D, generator=g)
    p = torch.randn(2 * T - 1, D, generator=g)
    u, vb = torch.randn(H, 64, generator=g) * 0.3, torch.randn(H, 64, generator=g) * 0.3
    lengths = [400, 333, 7, 129]
    ln = torch.tensor(lengths, dtype=torch.int32, device=dev)
    outs = [ops.relpos_attention(q.to(dev), k.to(dev), v.to(dev), p.to(dev), u.to(dev), vb.to(dev), ln, H,
                                 precision="f16").cpu() for _ in range(3)]
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])

    def heads(t):
        return t.double().view(B, T, H, 64).transpose(1, 2)
    scores = O.rel_attention_scores(heads(q), heads(k), p.double().view(2 * T - 1, H, 64).transpose(0, 1),
                                    u.double(), vb.double())
    pad = torch.arange(T)[None, :] >= torch.tensor(lengths)[:, None]
    attn = torch.softmax(scores.masked_fill(pad[:, None, None, :], float("-inf")), dim=-1)
    ref = (attn @ heads(v)).transpose(1, 2).reshape(B, T, D)
    mx, rms = err_stats(outs[0], ref)
    record("relpos_attention_moving_ref", (B, T, H), [mx, rms], [6e-2, 4e-3])
    # logits of magnitude ~30 carry 11-bit operand rounding of ~0.02 absolute: a few % on the sharpest rows
    assert mx < 6e-2 and rms < 4e-3, (mx, rms)


# ------------------------------------------------------------------------------------------ whole encoder
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("name", ["tiny_ragged", "tiny_k7_nomask", "full2_ragged", "full12_s1", "full12_ragged"])
def test_encoder_matches_reference_golden(dev, name, prec):
    c = load_case(name)
    enc = _encoder(c, dev, prec)
    ref = torch.from_numpy(c["z"]["out_f64"]).double()
    outs = {}
    for graph in (False, True):
        enc.use_graph = graph
        out, m = enc(c["xs"].to(dev), _mask(c, dev))
        outs[graph] = out.cpu()
        mx, rms = err_stats(outs[graph], ref)
        tol = tol_enc(prec, c["cfg"]["num_blocks"])
        record("encoder_golden", (name, prec, graph), [mx, rms], list(tol))
        assert mx < tol[0] and rms < tol[1], (name, prec, graph, mx, rms)
        assert (m is None) == (not c["masked"])
    assert torch.equal(outs[False], outs[True]), "CUDA-graph replay must be bit-identical to direct launches"


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("name", ["tiny_ragged", "full2_ragged"])
def test_layer0_stage_taps(dev, name, prec):
    c = load_case(name)
    enc = _encoder(c, dev, prec)
    B, T, D = c["xs"].shape
    taps = torch.empty(5, B * T, D, device=dev)
    enc(c["xs"].to(dev), _mask(c, dev), taps=taps)
    for i in range(5):
        g = torch.from_numpy(c["z"][f"stage{i}"]).double().reshape(B * T, D)
        mx, rms = err_stats(taps[i].cpu(), g)
        scale = g.abs().max().item()
        tol = TOL_TAP[prec]
        record("stage_taps", (name, prec, i), mx / scale, tol)
        assert mx < tol * scale, (name, prec, i, mx, scale)


@pytest.mark.parametrize("prec", PRECS)
def test_per_module_layer_forward(dev, prec):
    """EncoderLayer / sub-module forwards (per-op C-ABI entry points) agree with the fused whole-encoder call."""
    c = load_case("tiny_ragged")
    enc = _encoder(c, dev, prec)
    for m in enc.modules():
        if hasattr(m, "precision"):
            m.precision = prec
    xs, mask = c["xs"].to(dev), _mask(c, dev)
    x, pos = enc.embed(xs)
    (x, _), _ = enc.encoders((x, pos), mask)
    y = enc.after_norm(x).cpu()
    ref = torch.from_numpy(c["z"]["out_f64"])
    mx, rms = err_stats(y, ref)
    tol = (8e-6, 8e-7) if prec == "fp32" else (8e-3, 1.2e-3)   # per-op path converts operands per call (tf32: truncation)
    record("per_module", (prec,), [mx, rms], list(tol))
    assert mx < tol[0] and rms < tol[1], (mx, rms)


@pytest.mark.parametrize("prec", PRECS)
def test_full_size_s2_against_oracle(dev, prec):
    """BASELINE.json configs[1]: 12 layers, d=768, max-frames 1600 as [400]*4 -- compared with the fp32 CPU oracle
    (itself pinned to the reference, tests/test_oracle_golden.py) and checked for batch-independence."""
    from auto_avsr_b200.synthetic import SHAPES, encoder_input, encoder_state_dict
    lengths = SHAPES["S2"]
    sd = encoder_state_dict(0)
    xs = encoder_input(lengths, 768, 1234)
    case = dict(cfg=dict(d_model=768, n_heads=12, linear_units=3072, num_blocks=12, cnn_kernel=31), sd=sd)
    enc = _encoder(case, dev, prec)
    mask = O.non_pad_mask(lengths).unsqueeze(1).to(dev)
    out = enc(xs.to(dev), mask)[0].cpu()
    torch.set_num_threads(max(1, torch.get_num_threads()))
    ref = O.encoder_forward(sd, xs.float(), lengths, 12)
    mx, rms = err_stats(out, ref)
    record("full_s2", (prec,), [mx, rms], list(TOL_ENC[prec]))
    assert mx < TOL_ENC[prec][0] and rms < TOL_ENC[prec][1], (prec, mx, rms)
    assert torch.isfinite(out).all()
    # utterances do not interact (no padding here): running utterance 2 alone gives the same rows
    alone = enc(xs[2:3].to(dev), None)[0].cpu()
    mx2, _ = err_stats(alone[0], out[2])
    record("full_s2_alone", (prec,), mx2, TOL_BATCH[prec])
    assert mx2 < TOL_BATCH[prec], mx2
    # batch permutation permutes the output
    perm = [3, 1, 0, 2]
    outp = enc(xs[perm].to(dev), mask)[0].cpu()
    record("full_s2_perm", (prec,), err_stats(outp, out[perm])[0], TOL_BATCH[prec])
    assert err_stats(outp, out[perm])[0] < TOL_BATCH[prec]


@pytest.mark.parametrize("shape", ["S1", "S2r", "S3", "S4"])
def test_survey_shapes_against_oracle(dev, shape):
    """The other canonical shapes of SURVEY.md section 8 at full size (12 layers, d=768) in the default arithmetic:
    S1 = one 100-frame utterance with mask None (configs[0]), S2r = ragged max-frames bucket (400 padded frames),
    S3 = 16 x 100 frames, S4 = one 1600-frame utterance (13 key tiles, 3199-row rel-pos table)."""
    from auto_avsr_b200.synthetic import SHAPES, encoder_input, encoder_state_dict
    lengths = list(SHAPES[shape])
    sd = encoder_state_dict(0)
    xs = encoder_input(lengths, 768, 1234)
    case = dict(cfg=dict(d_model=768, n_heads=12, linear_units=3072, num_blocks=12, cnn_kernel=31), sd=sd)
    enc = _encoder(case, dev, "f16")
    masked = shape != "S1"
    mask = O.non_pad_mask(lengths).unsqueeze(1).to(dev) if masked else None
    out = enc(xs.to(dev), mask)[0].cpu()
    ref = O.encoder_forward(sd, xs.float(), lengths if masked else None, 12)
    assert torch.isfinite(out).all()
    mx, rms = err_stats(out, ref)
    record("survey_shapes", (shape,), [mx, rms], list(TOL_ENC["f16"]))
    assert mx < TOL_ENC["f16"][0] and rms < TOL_ENC["f16"][1], (shape, mx, rms)
    again = enc(xs.to(dev), mask)[0].cpu()
    assert torch.equal(out, again), "graph replay must be bit-identical run to run"


@pytest.mark.parametrize("prec", PRECS)
def test_edge_shapes(dev, prec):
    from auto_avsr_b200 import ConformerEncoder
    from auto_avsr_b200.synthetic import encoder_input, encoder_state_dict
    sd = encoder_state_dict(5, num_blocks=1)
    enc = ConformerEncoder(num_blocks=1)
    enc.load_state_dict(sd)
    enc = enc.to(dev).eval()
    enc.precision = prec
    # empty batch / zero frames
    assert enc(torch.zeros(0, 10, 768, device=dev), None)[0].shape == (0, 10, 768)
    assert enc(torch.zeros(2, 0, 768, device=dev), None)[0].shape == (2, 0, 768)
    tol = TOL_EDGE[prec]
    for lengths, masked in [([1], False), ([3, 2], True), ([130, 127, 5], True), ([17, 0], True), ([33], False)]:
        xs = encoder_input(lengths, 768, 99)
        if max(lengths) == 17:            # zero-length utterance: keep T = 17
            xs = encoder_input([17, 17], 768, 99)
        mask = O.non_pad_mask(lengths, xs.size(1)).unsqueeze(1).to(dev) if masked else None
        out = enc(xs.to(dev), mask)[0].cpu()
        ref = O.encoder_forward(sd, xs.double(), lengths if masked else None, 12)
        mx, _ = err_stats(out, ref)
        record("edge_shapes", (prec, lengths, masked), mx, tol)
        assert mx < tol, (lengths, masked, mx)


def test_weight_refresh_on_parameter_update(dev):
    from auto_avsr_b200 import ConformerEncoder
    from auto_avsr_b200.synthetic import encoder_input, encoder_state_dict
    enc = ConformerEncoder(num_blocks=1)
    enc.load_state_dict(encoder_state_dict(5, num_blocks=1))
    enc = enc.to(dev).eval()
    enc.precision = "fp32"
    xs = encoder_input([20], 768, 1).to(dev)
    a = enc(xs, None)[0].clone()
    sd2 = encoder_state_dict(6, num_blocks=1)
    enc.load_state_dict(sd2)                       # in-place copy_ bumps tensor versions -> weights re-prepared
    b = enc(xs, None)[0]
    ref = O.encoder_forward(sd2, xs.cpu().double(), None, 12)
    assert not torch.allclose(a, b)
    assert err_stats(b.cpu(), ref)[0] < 1e-5


def test_launch_counter_counts_kernels(dev):
    from auto_avsr_b200 import _cabi, ops
    before = _cabi.launch_count()
    ops.layernorm(torch.randn(4, 768, device=dev), torch.ones(768, device=dev), torch.zeros(768, device=dev))
    assert _cabi.launch_count() == before + 1


def test_forward_is_run_to_run_deterministic(dev):
    c = load_case("full12_ragged")
    enc = _encoder(c, dev, "f16")
    xs, mask = c["xs"].to(dev), _mask(c, dev)
    outs = [enc(xs, mask)[0].clone() for _ in range(4)]
    for o in outs[1:]:
        assert torch.equal(o, outs[0])


def test_pipelined_encoder_matches_plain_forward(dev):
    """auto_avsr_b200.pipeline.PipelinedEncoder (copy/compute overlap on 3 streams) returns exactly what the plain
    forward returns, batch by batch, including ragged lengths."""
    from auto_avsr_b200 import ConformerEncoder
    from auto_avsr_b200.pipeline import PipelinedEncoder
    from auto_avsr_b200.synthetic import encoder_input, encoder_state_dict
    enc = ConformerEncoder(num_blocks=2)
    enc.load_state_dict(encoder_state_dict(4, num_blocks=2))
    enc = enc.to(dev).eval()
    lengths = [[96, 70, 33], [96, 96, 96], [96, 5, 90], [50, 96, 96], [96, 1, 2]]
    xs = [encoder_input([96] * 3, 768, 40 + i).pin_memory() for i in range(len(lengths))]
    lens = [torch.tensor(l, dtype=torch.int32).pin_memory() for l in lengths]
    outs = [torch.empty(3, 96, 768).pin_memory() for _ in lengths]
    pipe = PipelinedEncoder(enc, 3, 96, depth=2, device=dev)
    pipe.run(xs, lens, outs)
    pipe.synchronize()
    for x, l, o in zip(xs, lengths, outs):
        mask = O.non_pad_mask(l, 96).unsqueeze(1).to(dev)
        ref = enc(x.to(dev), mask)[0].cpu()
        assert torch.equal(o, ref)


# ------------------------------------------------------------------------------------------ round 2 additions
def test_shape_policy_direct_until_seen_then_graph(dev):
    """The reference's eval loop (lightning.py:69-72) calls encoder(x, None) with B=1 and a new T per utterance: such
    first-seen shapes must run on direct launches (no graph capture, one shared workspace); a shape that keeps coming
    back gets its CUDA graph after `graph_after` sightings and then replays bit-identically."""
    from auto_avsr_b200 import ConformerEncoder
    from auto_avsr_b200.synthetic import encoder_input, encoder_state_dict
    sd = encoder_state_dict(5, num_blocks=2)
    enc = ConformerEncoder(num_blocks=2)
    enc.load_state_dict(sd)
    enc = enc.to(dev).eval()
    Ts = [37, 100, 64, 251, 99, 180, 33, 400, 12, 77, 313, 58, 129, 240, 91, 17, 365, 204, 146, 63]
    for T in Ts:                                          # 20 distinct utterance lengths, mask None (configs[0] shape)
        xs = encoder_input([T], 768, T)
        out = enc(xs.to(dev), None)[0].cpu()
        ref = O.encoder_forward(sd, xs.double(), None, 12)
        mx, _ = err_stats(out, ref)
        record("shape_policy", (T,), mx, TOL_ENC_SHALLOW["f16"][0])
        assert mx < TOL_ENC_SHALLOW["f16"][0], (T, mx)
    st = enc._engine.stats
    assert st["plans_built"] == 0 and st["graph"] == 0 and st["direct"] == len(Ts), st
    assert len(enc._engine._workspaces) == 1              # one growable direct-launch workspace, not one per shape
    xs = encoder_input([100], 768, 100).to(dev)
    outs = [enc(xs, None)[0].clone() for _ in range(4)]   # the T=100 shape was seen once above: 2nd direct, 3rd+ graph
    st = enc._engine.stats
    assert st["plans_built"] == 1 and st["graph"] == 3, st
    for o in outs[1:]:
        assert torch.equal(o, outs[0])


@pytest.mark.parametrize("scale", [8.0, 64.0, 1024.0])
def test_fp16_range_saturation_is_detected_or_within_tolerance(dev, scale):
    """fp16 operand stores saturate at +-65504.  With LayerNorm gains, FFN w_1 weights and the input scaled up the
    hidden activations approach / pass that limit: the checked forward must either report it (SaturationError) or the
    result must still meet the f16 tolerance; tf32 operands (fp32 range) must meet it regardless."""
    from auto_avsr_b200 import ConformerEncoder
    from auto_avsr_b200.engine import SaturationError
    from auto_avsr_b200.synthetic import encoder_input, encoder_state_dict
    lengths = [48, 31]
    sd = encoder_state_dict(3, num_blocks=2)
    # magnitudes grow, conditioning does not: the FFN branch is linear up to the ReLU, so scaling its LayerNorm gain and
    # w_1 by `scale` each multiplies the hidden activations by scale^2 (x64 / x4096) without sharpening any softmax
    for k in list(sd):
        if k.endswith((".norm_ff.weight", ".norm_ff_macaron.weight", ".w_1.weight", ".w_1.bias", ".linear_v.weight")):
            sd[k] = sd[k] * scale
    xs = encoder_input(lengths, 768, 7) * scale
    ref = O.encoder_forward(sd, xs.double(), lengths, 12)
    rscale = ref.abs().max().item()
    enc = ConformerEncoder(num_blocks=2)
    enc.load_state_dict(sd, strict=True)
    enc = enc.to(dev).eval()
    mask = O.non_pad_mask(lengths).unsqueeze(1).to(dev)
    enc.precision = "tf32"
    mx, rms = err_stats(enc(xs.to(dev), mask)[0].cpu(), ref)
    tol = (2.2e-3, 3.2e-4)          # relative to the output's max-abs (observed 5.4e-4 / 7.9e-5 on B200)
    record("range_tf32", (scale,), [mx / rscale, rms / rscale], list(tol))
    assert mx < tol[0] * rscale and rms < tol[1] * rscale, (scale, mx, rms, rscale)
    enc.precision = "f16"
    enc.check_saturation = True
    try:
        out = enc(xs.to(dev), mask)[0].cpu()
    except SaturationError as e:
        record("range_f16", (scale,), "SaturationError", str(e)[:40])
        enc.check_saturation = False
        raw = enc(xs.to(dev), mask)[0].cpu()               # the unchecked path still returns finite numbers
        assert torch.isfinite(raw).all()
        return
    mx, rms = err_stats(out, ref)
    record("range_f16", (scale,), [mx / rscale, rms / rscale], list(tol))
    assert mx < tol[0] * rscale and rms < tol[1] * rscale, (scale, mx, rms, rscale)


def test_saturation_counter_counts(dev):
    """A weight set that certainly overflows half (w_1 x 2^20) must trip the counter; the unscaled one must not."""
    from auto_avsr_b200 import ConformerEncoder
    from auto_avsr_b200.engine import SaturationError
    from auto_avsr_b200.synthetic import encoder_input, encoder_state_dict
    sd = encoder_state_dict(3, num_blocks=1)
    xs = encoder_input([40], 768, 7).to(dev)
    enc = ConformerEncoder(num_blocks=1)
    enc.load_state_dict(sd)
    enc = enc.to(dev).eval()
    enc.check_saturation = True
    enc(xs, None)                                          # in range: no exception
    sd["encoders.0.feed_forward.w_1.weight"] = sd["encoders.0.feed_forward.w_1.weight"] * float(2 ** 20)
    enc.load_state_dict(sd)
    with pytest.raises(SaturationError):
        enc(xs, None)
    enc.precision = "tf32"                                 # fp32-range operands: the check does not apply
    assert torch.isfinite(enc(xs, None)[0]).all()


def test_wrong_device_and_mask_checks(dev):
    from auto_avsr_b200 import ConformerEncoder
    from auto_avsr_b200.synthetic import encoder_input, encoder_state_dict
    enc = ConformerEncoder(num_blocks=1)
    enc.load_state_dict(encoder_state_dict(5, num_blocks=1))
    enc = enc.to(dev).eval()
    enc.check_mask = True
    xs = encoder_input([20, 20], 768, 1).to(dev)
    holes = torch.ones(2, 1, 20, dtype=torch.bool, device=dev)
    holes[1, 0, 3] = False
    with pytest.raises(NotImplementedError):
        enc(xs, holes)
    ok = O.non_pad_mask([20, 11]).unsqueeze(1).to(dev)
    enc(xs, ok)
