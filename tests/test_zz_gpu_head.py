"""GPU parity of the steps either side of the encoder (SURVEY.md section 8f #1): proj_encoder in front, the CTC head
(ctc_lo GEMM + row-wise log-softmax / argmax) behind -- through the C ABI, against the oracle and the golden vectors
generated from the reference's own modules (tests/golden/head_*.npz).

Each test runs in a child process (its own CUDA context and its own environment switches).  First B200 run: round 2
(10 passed); the bounds below are <= 4x the errors observed there (gpurun_out/parity_observed.jsonl ->
profiles/r02_parity_observed.txt)."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))

pytestmark = pytest.mark.gpu

PRELUDE = f"""
import sys, math, torch
sys.path.insert(0, {ROOT!r}); sys.path.insert(0, {HERE!r})
from helpers import err_stats, load_head_case, record
from auto_avsr_b200 import ops, ConformerEncoder, CTC, ProjEncoder
from oracle import conformer_oracle as O
from oracle import head_oracle as HO
dev = torch.device("cuda:0")
# <= 4x the errors observed on B200 (round 2): encoder features, CTC log-probs (max-abs, rms), proj (relative max)
TOL = {{"fp32": (2.5e-5, 2.4e-6), "tf32": (9e-3, 1.3e-3), "f16": (9e-3, 1.3e-3)}}
TOL_LOGP = {{"fp32": (1.4e-5, 2.4e-6), "tf32": (5e-3, 1.1e-3), "f16": (5e-3, 1.1e-3)}}
TOL_PROJ = {{"fp32": 3e-6, "tf32": 1.1e-3, "f16": 1.1e-3}}

def build(c, prec):
    cfg = c["cfg"]
    enc = ConformerEncoder(attention_dim=cfg["d_model"], attention_heads=cfg["n_heads"], linear_units=cfg["linear_units"],
                           num_blocks=cfg["num_blocks"], cnn_module_kernel=cfg["cnn_kernel"])
    enc.load_state_dict(c["enc_sd"], strict=True)
    proj = ProjEncoder(cfg["idim"], cfg["d_model"])
    proj.load_state_dict({{"weight": c["head_sd"]["proj_encoder.weight"], "bias": c["head_sd"]["proj_encoder.bias"]}})
    ctc = CTC(cfg["odim"], cfg["d_model"], 0.1)
    ctc.load_state_dict({{"ctc_lo.weight": c["head_sd"]["ctc.ctc_lo.weight"], "ctc_lo.bias": c["head_sd"]["ctc.ctc_lo.bias"]}})
    mods = [m.to(dev).eval() for m in (proj, enc, ctc)]
    for m in mods:
        m.precision = prec
    enc.graph_after = 1
    return mods
"""


def run_child(body, timeout=600):
    r = subprocess.run([sys.executable, "-c", PRELUDE + body], capture_output=True, text=True, timeout=timeout,
                       cwd=ROOT)
    assert r.returncode == 0 and "CHILD-OK" in r.stdout, r.stdout[-1500:] + r.stderr[-2500:]


def test_log_softmax_and_argmax_rows():
    run_child("""
g = torch.Generator().manual_seed(5)
for rows, n, ld in [(37, 5049, 5120), (1, 1, 128), (3, 37, 128), (1600, 5049, 5120), (5, 130, 130), (2, 5049, 5049)]:
    x = torch.randn(rows, ld, generator=g) * 3.0
    x[:, n:] = 1e4                                   # padding columns must be ignored
    if rows >= 3 and n > 8:
        x[1, 5] = x[1, 2] = x[1, :n].max() + 1.0      # tie: the first maximal index wins
    ref = torch.log_softmax(x[:, :n].double(), dim=-1)
    y, best = ops.log_softmax(x.to(dev), n, want_argmax=True)
    mx, _ = err_stats(y.cpu(), ref)
    assert y.shape == (rows, n) and mx < 2e-5, (rows, n, ld, mx)
    assert torch.equal(best.cpu(), x[:, :n].argmax(-1)), (rows, n)
    assert torch.equal(ops.argmax_rows(x.to(dev), n).cpu(), x[:, :n].argmax(-1))
    lse = torch.logsumexp(y.double().cpu(), -1)
    assert lse.abs().max() < 1e-4
print("CHILD-OK")
""")


@pytest.mark.parametrize("prec", ["fp32", "tf32", "f16"])
@pytest.mark.parametrize("name", ["head_tiny", "head_full"])
def test_features_to_log_probs_match_reference_golden(name, prec):
    run_child(f"""
c = load_head_case({name!r})
proj, enc, ctc = build(c, {prec!r})
mask = O.non_pad_mask(c["lengths"]).unsqueeze(1).to(dev)
with torch.no_grad():
    x = proj(c["feats"].to(dev))
    hs, _ = enc(x, mask)
    logp = ctc.log_softmax(hs)
    prob = ctc.softmax(hs)
    best = ctc.argmax(hs)
z = c["z"]
mx, rms = err_stats(x.cpu(), torch.from_numpy(z["proj_f64"]))
scale = float(torch.from_numpy(z["proj_f64"]).abs().max())
record("head_proj", ({name!r}, {prec!r}), mx / max(1.0, scale), TOL_PROJ[{prec!r}])
assert mx < TOL_PROJ[{prec!r}] * max(1.0, scale), ("proj", mx)
mx, rms = err_stats(logp.cpu(), torch.from_numpy(z["logp_f64"]))
record("head_logp", ({name!r}, {prec!r}), [mx, rms], list(TOL_LOGP[{prec!r}]))
assert mx < TOL_LOGP[{prec!r}][0] and rms < TOL_LOGP[{prec!r}][1], ("logp", mx, rms)
assert logp.shape == tuple(z["logp_f64"].shape)
assert (prob.sum(-1).cpu() - 1).abs().max() < 1e-4 and ctc.probs is prob
agree = (best.cpu() == torch.from_numpy(z["argmax_f64"])).float().mean().item()
record("head_argmax_agree", ({name!r}, {prec!r}), agree, 0.99 if {prec!r} == "fp32" else 0.9)
assert agree >= (0.99 if {prec!r} == "fp32" else 0.9), agree
print("CHILD-OK")
""")


def test_full_size_s2_features_to_log_probs_against_oracle():
    run_child("""
from auto_avsr_b200.synthetic import SHAPES, encoder_state_dict, frontend_features, head_state_dict
lengths = list(SHAPES["S2"])
c = dict(cfg=dict(idim=512, d_model=768, n_heads=12, linear_units=3072, num_blocks=12, cnn_kernel=31, odim=5049),
         enc_sd=encoder_state_dict(0), head_sd=head_state_dict(0))
feats = frontend_features(lengths, 512, 4321)
proj, enc, ctc = build(c, "f16")
mask = O.non_pad_mask(lengths).unsqueeze(1).to(dev)
with torch.no_grad():
    hs, _ = enc(proj(feats.to(dev)), mask)
    logp = ctc.log_softmax(hs).cpu()
ref = HO.features_to_log_probs(c["head_sd"], c["enc_sd"], feats.float(), lengths, 12)
mx, rms = err_stats(logp, ref)
record("head_full_s2_logp", ("f16",), [mx, rms], [7e-3, 1.1e-3])
assert torch.isfinite(logp).all() and mx < 7e-3 and rms < 1.1e-3, (mx, rms)
assert torch.logsumexp(logp.double(), -1).abs().max() < 1e-4          # every frame's distribution is normalised
print("CHILD-OK")
""", timeout=900)


@pytest.mark.parametrize("prec", ["fp32", "tf32", "f16"])
@pytest.mark.parametrize("name", ["head_tiny", "head_full"])
def test_fused_features_to_log_probs_match_reference_golden(name, prec):
    """ONE library call (avsr_features_to_logprobs): proj_encoder with the embed scale folded in writing the residual
    stream, the encoder, after_norm emitting ctc_lo's operand, ctc_lo with log-sum-exp partials -- against the fixtures
    generated from the reference's own proj_encoder / ConformerEncoder / CTC modules."""
    run_child(f"""
from auto_avsr_b200.head import features_to_log_probs
c = load_head_case({name!r})
proj, enc, ctc = build(c, {prec!r})
mask = O.non_pad_mask(c["lengths"]).unsqueeze(1).to(dev)
with torch.no_grad():
    hs, logp, best = features_to_log_probs(proj, enc, ctc, c["feats"].to(dev), mask, want_argmax=True)
    hs2, logp2, _ = features_to_log_probs(proj, enc, ctc, c["feats"].to(dev), mask, want_features=False)
z = c["z"]
assert hs2 is None and torch.equal(logp, logp2)
keep = logp.clone()
for _ in range(3):                                    # graph_after = 1 in build(): these replay the captured plan
    hs3, logp3, best3 = features_to_log_probs(proj, enc, ctc, c["feats"].to(dev), mask, want_argmax=True)
assert torch.equal(logp3, keep) and torch.equal(hs3, hs) and torch.equal(best3, best)
mx, rms = err_stats(hs.cpu(), torch.from_numpy(z["enc_f64"]))
record("fused_enc", ({name!r}, {prec!r}), [mx, rms], list(TOL[{prec!r}]))
assert mx < TOL[{prec!r}][0] and rms < TOL[{prec!r}][1], ("enc", mx, rms)
mx, rms = err_stats(logp.cpu(), torch.from_numpy(z["logp_f64"]))
record("fused_logp", ({name!r}, {prec!r}), [mx, rms], list(TOL_LOGP[{prec!r}]))
assert mx < TOL_LOGP[{prec!r}][0] and rms < TOL_LOGP[{prec!r}][1], ("logp", mx, rms)
assert torch.logsumexp(logp.double().cpu(), -1).abs().max() < 1e-4
assert torch.equal(best.cpu(), logp.argmax(-1).cpu())
agree = (best.cpu() == torch.from_numpy(z["argmax_f64"])).float().mean().item()
assert agree >= (0.99 if {prec!r} == "fp32" else 0.9), agree
assert len(enc._fused_head.plans) == 2                # one per (want_features, want_argmax) combination used above
enc.refresh_weights()                                 # the encoder's prepared weights go, and the fused plans baking them
assert len(enc._fused_head.plans) == 0
print("CHILD-OK")
""")


def test_fused_full_size_s2_matches_module_path_and_oracle():
    """BASELINE.json configs[2] at full size (4 x 400 frames, idim 512, odim 5049): the fused call (two-SM ctc_lo GEMM
    with the log-sum-exp epilogue: M = 1600 >= 256) against the module-by-module path and the CPU oracle."""
    run_child("""
from auto_avsr_b200.head import features_to_log_probs
from auto_avsr_b200.synthetic import SHAPES, encoder_state_dict, frontend_features, head_state_dict
lengths = list(SHAPES["S2r"])
c = dict(cfg=dict(idim=512, d_model=768, n_heads=12, linear_units=3072, num_blocks=12, cnn_kernel=31, odim=5049),
         enc_sd=encoder_state_dict(0), head_sd=head_state_dict(0))
feats = frontend_features(lengths, 512, 4321)
proj, enc, ctc = build(c, "f16")
mask = O.non_pad_mask(lengths).unsqueeze(1).to(dev)
with torch.no_grad():
    hs, logp, best = features_to_log_probs(proj, enc, ctc, feats.to(dev), mask, want_argmax=True)
    hs_m, _ = enc(proj(feats.to(dev)), mask)
    logp_m = ctc.log_softmax(hs_m)
    best_m = ctc.argmax(hs_m)
mx, rms = err_stats(hs.cpu(), hs_m.cpu())
record("fused_vs_modules_enc", ("S2r",), [mx, rms], [1.8e-2, 1.2e-3])
assert mx < 1.8e-2 and rms < 1.2e-3, (mx, rms)          # proj rounding differs (scale folded before fp16 rounding)
mx, rms = err_stats(logp.cpu(), logp_m.cpu())
record("fused_vs_modules_logp", ("S2r",), [mx, rms], [5.2e-3, 1e-3])
assert mx < 5.2e-3 and rms < 1e-3, (mx, rms)
assert torch.logsumexp(logp.double().cpu(), -1).abs().max() < 1e-4
assert torch.equal(best.cpu(), logp.argmax(-1).cpu()) and torch.equal(best_m.cpu(), logp_m.argmax(-1).cpu())
ref = HO.features_to_log_probs(c["head_sd"], c["enc_sd"], feats.float(), lengths, 12)
mx, rms = err_stats(logp.cpu(), ref)
record("fused_full_logp_vs_oracle", ("S2r",), [mx, rms], [6e-3, 1.1e-3])
assert torch.isfinite(logp).all() and mx < 6e-3 and rms < 1.1e-3, (mx, rms)
print("CHILD-OK")
""", timeout=900)
