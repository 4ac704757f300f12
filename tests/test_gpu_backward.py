"""Training slice (SURVEY.md 8f #2, first slice) on a B200: forward AND backward of the drop-in LayerNorm,
PositionwiseFeedForward and ConvolutionModule in train() mode run in libavsr_b200 (auto_avsr_b200/train.py) and must
reproduce outputs, input gradients, parameter gradients and BatchNorm running statistics of the UNMODIFIED reference
modules (fixtures tests/golden/train_*.npz from oracle/make_golden_train.py: float64, dropout p = 0).

Bounds: forward like the inference tests; gradients relative to the largest reference gradient entry -- backward GEMMs
run on TF32 operands (f16 / tf32 precision) or fp32 FMAs (fp32 precision); bounds are <= 4x what a B200 produced."""
import os

import numpy as np
import pytest
import torch

from helpers import GOLDEN, err_stats, record
from auto_avsr_b200.synthetic import encoder_state_dict

pytestmark = pytest.mark.gpu

D, F, K = 768, 3072, 31
PRECS = ["fp32", "tf32", "f16"]
TOL_FWD = {"fp32": 2e-5, "tf32": 4e-3, "f16": 4e-3}       # relative to the output's max-abs
TOL_GRAD = {"fp32": 2e-5, "tf32": 4e-3, "f16": 4e-3}      # relative to the reference gradient's max-abs


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "run with gpurun"
    import __graft_entry__ as g
    g.build()
    return torch.device("cuda:0")


def load(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    g = torch.Generator().manual_seed(int(z["seed"]))
    x = torch.randn(3, 37, D, generator=g, dtype=torch.float64)
    r = torch.randn(3, 37, D, generator=g, dtype=torch.float64)
    sd = encoder_state_dict(int(z["wseed"]), D, 12, F, 1, K)
    return z, x.float(), r.float(), sd


def sub_state(sd, prefix):
    return {k[len(prefix):]: v for k, v in sd.items() if k.startswith(prefix)}


def rel_err(a, ref):
    ref = torch.as_tensor(np.asarray(ref)).double()
    return (a.double().cpu() - ref).abs().max().item() / max(ref.abs().max().item(), 1e-30)


def check_param_grads(module, z, prec, what):
    for n, p in module.named_parameters():
        assert p.grad is not None, n
        key = "grad_" + n
        if key in z.files and np.abs(z[key]).max() < 1e-9:
            # mathematically zero (a bias in front of BatchNorm: the batch mean removes it): absolute check against the
            # scale of the other gradients instead of a ratio of rounding noise
            e = p.grad.abs().max().item()
            record("backward_" + what, (prec, n, "abs"), e, 1e-4)
            assert e < 1e-4, (what, n, e)
            continue
        if key in z.files:
            e = rel_err(p.grad, z[key])
        else:                                    # big matrices: every 8th row + checksums (oracle/make_golden_train.py)
            step = int(z[key + "__step"]) if key + "__step" in z.files else 8
            e = rel_err(p.grad[::step], z[key + "__rows8"])
            cs = z[key + "__checksum"]
            g = p.grad.double().cpu()
            got = np.array([g.sum().item(), g.abs().sum().item(), (g ** 2).sum().item()])
            assert abs(got[1] - cs[1]) <= 2e-3 * cs[1] and abs(got[2] - cs[2]) <= 4e-3 * cs[2], (what, n, got, cs)
        record("backward_" + what, (prec, n), e, TOL_GRAD[prec])
        assert e < TOL_GRAD[prec], (what, n, prec, e)


@pytest.mark.parametrize("prec", PRECS)
def test_gpu_backward_layernorm(dev, prec):
    from auto_avsr_b200 import LayerNorm
    z, x, r, sd = load("train_ln")
    m = LayerNorm(D)
    m.load_state_dict(sub_state(sd, "encoders.0.norm_ff."))
    m = m.to(dev).train()
    xg = x.to(dev).requires_grad_(True)
    y = m(xg)
    (y * r.to(dev)).sum().backward()
    assert rel_err(y, z["y"]) < 5e-6
    e = rel_err(xg.grad, z["dx"])
    record("backward_ln", (prec, "dx"), e, 2e-5)
    assert e < 2e-5, e                                           # LayerNorm backward is fp32 in every mode
    for n, key in (("weight", "grad_weight"), ("bias", "grad_bias")):
        e = rel_err(getattr(m, n).grad, z[key])
        record("backward_ln", (prec, n), e, 2e-5)
        assert e < 2e-5, (n, e)


@pytest.mark.parametrize("prec", PRECS)
def test_gpu_backward_feed_forward(dev, prec):
    from auto_avsr_b200 import PositionwiseFeedForward
    z, x, r, sd = load("train_ffn")
    m = PositionwiseFeedForward(D, F, 0.0)
    m.load_state_dict(sub_state(sd, "encoders.0.feed_forward."))
    m = m.to(dev).train()
    m.precision = prec
    xg = x.to(dev).requires_grad_(True)
    y = m(xg)
    (y * r.to(dev)).sum().backward()
    e = rel_err(y, z["y"])
    record("backward_ffn", (prec, "y"), e, TOL_FWD[prec])
    assert e < TOL_FWD[prec], e
    if prec == "fp32":
        e = rel_err(xg.grad, z["dx"])
        record("backward_ffn", (prec, "dx"), e, TOL_GRAD[prec])
        assert e < TOL_GRAD[prec], e
        check_param_grads(m, z, prec, "ffn")
        return
    # Tensor-core forward: hidden units whose pre-activation is smaller than the operand rounding (|h| < ~1e-3) can land
    # on the other side of the ReLU than in the float64 reference; each such unit moves dx by one full term (a
    # derivative discontinuity, not an arithmetic error: the fp32 path above matches the reference to 2e-5).  So the
    # reference gradients are restated in float64 with the mask the GPU forward actually used (the FFN backward is
    # three lines: positionwise_feed_forward.py:28-30), and the reference-autograd fixture is checked with a loose bound.
    w1, b1 = m.w_1.weight.detach().double().cpu(), m.w_1.bias.detach().double().cpu()
    w2 = m.w_2.weight.detach().double().cpu()
    from auto_avsr_b200 import ops
    h_gpu = ops.linear(x.to(dev), m.w_1.weight, m.w_1.bias, relu=True, precision=prec).double().cpu().reshape(-1, F)
    mask = (h_gpu > 0).double()
    x2, r2 = x.double().reshape(-1, D), r.double().reshape(-1, D)
    h = torch.relu(x2 @ w1.T + b1) * mask
    dh = (r2 @ w2) * mask
    ref = {"dx": (dh @ w1).reshape(x.shape), "w_1.weight": dh.T @ x2, "w_1.bias": dh.sum(0), "w_2.weight": r2.T @ h,
           "w_2.bias": r2.sum(0)}
    e = rel_err(xg.grad, ref["dx"])
    record("backward_ffn_same_mask", (prec, "dx"), e, TOL_GRAD[prec])
    assert e < TOL_GRAD[prec], e
    for n, p in m.named_parameters():
        e = rel_err(p.grad, ref[n])
        record("backward_ffn_same_mask", (prec, n), e, TOL_GRAD[prec])
        assert e < TOL_GRAD[prec], (n, e)
    e = rel_err(xg.grad, z["dx"])
    record("backward_ffn_vs_reference_autograd", (prec, "dx"), e, 1e-1)
    assert e < 1e-1, e


@pytest.mark.parametrize("prec", PRECS)
def test_gpu_backward_conv_module(dev, prec):
    from auto_avsr_b200 import ConvolutionModule
    z, x, r, sd = load("train_conv")
    m = ConvolutionModule(D, K)
    m.load_state_dict(sub_state(sd, "encoders.0.conv_module."))
    m = m.to(dev).train()
    m.precision = prec
    xg = x.to(dev).requires_grad_(True)
    y = m(xg)
    (y * r.to(dev)).sum().backward()
    e = rel_err(y, z["y"])
    record("backward_conv", (prec, "y"), e, TOL_FWD[prec])
    assert e < TOL_FWD[prec], e
    e = rel_err(xg.grad, z["dx"])
    record("backward_conv", (prec, "dx"), e, TOL_GRAD[prec])
    assert e < TOL_GRAD[prec], e
    check_param_grads(m, z, prec, "conv")
    # BatchNorm1d bookkeeping exactly like torch's: running statistics (momentum 0.1, unbiased variance) and the counter
    assert int(m.norm.num_batches_tracked) == int(z["buf_norm.num_batches_tracked"])      # the loaded counter + 1
    for n in ("running_mean", "running_var"):
        e = rel_err(getattr(m.norm, n), z["buf_norm." + n])
        record("backward_conv", (prec, n), e, TOL_FWD[prec])
        assert e < TOL_FWD[prec], (n, e)


@pytest.mark.parametrize("prec", PRECS)
def test_gpu_backward_relpos_attention(dev, prec):
    """RelPositionMultiHeadedAttention in train() on a ragged batch: the fused forward kernel of the precision, the
    recomputing fp32 backward kernels, q/k/v/pos/out projections through LinearFn -- against the reference module's
    autograd (output, dx, all 11 parameter gradients incl. pos_bias_u / pos_bias_v and linear_pos)."""
    from auto_avsr_b200 import RelPositionMultiHeadedAttention, ops
    from oracle import conformer_oracle as O
    z, x, r, sd = load("train_attn")
    lengths = [int(v) for v in z["lengths"]]
    m = RelPositionMultiHeadedAttention(12, D, 0.0)
    m.load_state_dict(sub_state(sd, "encoders.0.self_attn."))
    m = m.to(dev).train()
    m.precision = prec
    mask = O.non_pad_mask(lengths).unsqueeze(1).to(dev)
    pos_emb = ops.rel_sinusoid_table(x.size(1), D, dev).unsqueeze(0)
    xg = x.to(dev).requires_grad_(True)
    y = m(xg, None, None, pos_emb, mask)
    (y * r.to(dev)).sum().backward()
    e = rel_err(y, z["y"])
    record("backward_attn", (prec, "y"), e, TOL_FWD[prec])
    assert e < TOL_FWD[prec], e
    tol = TOL_GRAD[prec] if prec == "fp32" else 8e-3       # forward probabilities come from fp16 / tf32 operands
    e = rel_err(xg.grad, z["dx"])
    record("backward_attn", (prec, "dx"), e, tol)
    assert e < tol, e
    for n, p in m.named_parameters():
        key = "grad_" + n
        if key in z.files and np.abs(z[key]).max() < 1e-9:
            # linear_k.bias: a constant added to every key shifts all scores of a row alike -- softmax ignores it, the
            # gradient is mathematically zero; absolute check against the scale of the other gradients
            scale = float(np.abs(z["grad_linear_q.bias"]).max())
            e = p.grad.abs().max().item() / scale
            record("backward_attn", (prec, n, "abs / |d linear_q.bias|"), e, tol)
            assert e < tol, (n, e)
            continue
        if key in z.files:
            e = rel_err(p.grad, z[key])
        else:
            e = rel_err(p.grad[::int(z[key + "__step"])], z[key + "__rows8"])
        record("backward_attn", (prec, n), e, tol)
        assert e < tol, (n, e)


@pytest.mark.parametrize("prec", ["fp32", "f16"])
def test_gpu_backward_whole_encoder_train_mode(dev, prec):
    """The drop-in ConformerEncoder (2 layers) in train() with every dropout rate 0: forward output, input gradient,
    every parameter gradient (checksums; rows of the big matrices; small ones in full) and the BatchNorm running
    statistics against the reference encoder's autograd -- what train.py's training_step drives (lightning.py:86-94)."""
    from auto_avsr_b200 import ConformerEncoder
    from oracle import conformer_oracle as O
    z = np.load(os.path.join(GOLDEN, "train_enc2.npz"))
    g = torch.Generator().manual_seed(int(z["seed"]))
    x = torch.randn(3, 37, D, generator=g, dtype=torch.float64).float()
    r = torch.randn(3, 37, D, generator=g, dtype=torch.float64).float()
    lengths = [int(v) for v in z["lengths"]]
    enc = ConformerEncoder(num_blocks=2, dropout_rate=0.0, positional_dropout_rate=0.0, attention_dropout_rate=0.0)
    enc.load_state_dict(encoder_state_dict(int(z["wseed"]), D, 12, F, 2, K), strict=True)
    enc = enc.to(dev).train()
    enc.precision = prec
    mask = O.non_pad_mask(lengths).unsqueeze(1).to(dev)
    xg = x.to(dev).requires_grad_(True)
    y, m_out = enc(xg, mask)
    assert m_out is mask
    (y * r.to(dev)).sum().backward()
    tf, tg = (3e-5, 1e-4) if prec == "fp32" else (8e-3, 4e-2)
    e = rel_err(y, z["y"])
    record("backward_enc2", (prec, "y"), e, tf)
    assert e < tf, e
    e = rel_err(xg.grad, z["dx"])
    record("backward_enc2", (prec, "dx"), e, tg)
    assert e < tg, e
    worst = 0.0
    for n, p in enc.named_parameters():
        assert p.grad is not None and torch.isfinite(p.grad).all(), n
        cs = z["cs_" + n]
        gd = p.grad.double().cpu()
        got = np.array([gd.sum().item(), gd.abs().sum().item(), (gd ** 2).sum().item()])
        e = 0.0
        if cs[1] > 1e-6:                         # (a bias in front of BatchNorm has a mathematically zero gradient)
            e = max(e, abs(got[1] - cs[1]) / cs[1], abs(got[2] - cs[2]) / cs[2])
        # element-wise only where the gradient is a smooth function of the forward: a hidden unit whose pre-activation
        # sits within the operand rounding of zero flips its ReLU against the float64 reference and moves its whole row
        # of d w_1 (the same-mask FFN test above pins that arithmetic); the checksums still cover w_1
        elementwise = prec == "fp32" or ".w_1." not in n
        if elementwise and "rows64_" + n in z.files:
            e = max(e, rel_err(p.grad[::64], z["rows64_" + n]))
        elif elementwise and "grad_" + n in z.files and np.abs(z["grad_" + n]).max() > 1e-9:
            e = max(e, rel_err(p.grad, z["grad_" + n]))
        record("backward_enc2_param", (prec, n), e, tg)
        worst = max(worst, e)
    record("backward_enc2", (prec, "worst parameter gradient"), worst, tg)
    assert worst < tg, worst
    for n, b in enc.named_buffers():
        if "running" in n:
            e = rel_err(b, z["buf_" + n])
            assert e < (1e-5 if prec == "fp32" else 5e-3), (n, e)


def test_train_mode_scope_and_optimizer_step(dev):
    """Gradients land on the original Parameters (AdamW steps them); what is not in the slice refuses loudly."""
    from auto_avsr_b200 import ConformerEncoder, PositionwiseFeedForward
    m = PositionwiseFeedForward(D, F, 0.1).to(dev).train()           # dropout active: just has to run and be finite
    opt = torch.optim.AdamW(m.parameters(), lr=1e-3)
    before = [p.detach().clone() for p in m.parameters()]
    x = torch.randn(2, 50, D, device=dev)
    for _ in range(2):
        opt.zero_grad()
        loss = m(x).pow(2).mean()
        loss.backward()
        torch.nn.utils.clip_grad_norm_(m.parameters(), 10.0)        # train.py:41
        opt.step()
    assert all(torch.isfinite(p).all() for p in m.parameters())
    assert all(not torch.equal(a, p.detach()) for a, p in zip(before, m.parameters()))
    enc = ConformerEncoder(num_blocks=1, attention_dropout_rate=0.1).to(dev).train()
    with pytest.raises(NotImplementedError):                          # dropout on attention probabilities: not built
        enc(torch.randn(1, 20, D, device=dev), None)
    enc = ConformerEncoder(num_blocks=1).to(dev).train()             # the reference's rates (0.1 / 0.1 / 0.0)
    opt = torch.optim.AdamW(enc.parameters(), lr=1e-4)
    out, _ = enc(torch.randn(2, 30, D, device=dev), None)
    out.pow(2).mean().backward()
    torch.nn.utils.clip_grad_norm_(enc.parameters(), 10.0)
    opt.step()
    assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in enc.parameters())


def test_ddp_gradient_allreduce_two_ranks(dev):
    """Two NCCL ranks (both on cuda:0 when the box has a single GPU is not possible -> needs 2 GPUs; skipped otherwise):
    DistributedDataParallel over a stack of the slice's modules -- every gradient is produced by libavsr_b200's backward
    and all-reduced by DDP's hooks on the original Parameters (train.py:37)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                        "127.0.0.1", "--master-port", "29533", os.path.join(root, "tests", "ddp_worker.py")],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "DDP-OK" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]
    # train.py:31 sync_batchnorm=True: conv_module.norm converted to SyncBatchNorm -- cross-rank batch statistics
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                        "127.0.0.1", "--master-port", "29534", os.path.join(root, "tests", "ddp_worker.py")],
                       capture_output=True, text=True, timeout=600, env=dict(os.environ, AVSR_DDP_SYNCBN="1", AVSR_DDP_BLOCKS="2"))
    assert r.returncode == 0 and "DDP-OK syncbn" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]
