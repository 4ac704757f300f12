#!/usr/bin/env python3
"""Benchmark of the hot path: Conformer encoder forward, frames/sec at max-frames=1600 (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--precision tf32|fp32]
                    [--dump-outputs DIR]

A step = one ConformerEncoder.forward (embed + 12 layers + after_norm, eval) over one synthetic max-frames=1600
bucket per GPU (workload S2 = 4 utterances x 400 frames, d=768, BASELINE.json configs[1]); weak scaling: every
rank gets its own bucket, no collective on the data path; value = all ranks' valid frames / max-over-ranks time.
Prints ONE JSON line (rank 0).  `--impl reference` times the reference's own CPU implementation on the host cores
instead: the unmodified espnet modules copied into the git-ignored oracle/_ref by oracle/build_ref.py (kind
"reference"; the copy travels to the GPU box with the snapshot), or, when that copy is absent, the CPU restatement
oracle/conformer_oracle.py (kind "port", pinned to the reference by tests/test_oracle_golden.py).
`--dump-outputs DIR` writes what the timed path returned in its last timed step (rank 0) as DIR/<name>.npy in float32,
so that two builds run with the same arguments, hence the same seeded inputs, can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from auto_avsr_b200.synthetic import SHAPES, encoder_input, encoder_state_dict  # noqa: E402

WORKLOAD = "S2"
CFG = dict(d_model=768, n_heads=12, linear_units=3072, num_blocks=12, cnn_kernel=31)
METRIC = "conformer_encoder_frames_per_sec_max_frames_1600"


def workload_string(name=None):
    """ONE description of the workload for both arms (the driver compares the two `config.workload` strings)."""
    name = name or WORKLOAD
    return (f"{name}: lengths={list(SHAPES[name])} (max-frames=1600 per GPU), d=768 H=12 ff=3072 L=12 k=31, eval forward, "
            "BASELINE.json configs[1]")


def non_pad_mask(lengths, device):
    """make_non_pad_mask(lengths).unsqueeze(-2) (e2e_asr_conformer.py:67) built with torch on the device."""
    ln = torch.tensor(list(lengths), device=device)
    return (torch.arange(int(max(lengths)), device=device)[None, :] < ln[:, None]).unsqueeze(1)


def algorithmic_flops(lengths, warm_pos_cache=False):
    """SURVEY.md 8d: 326,154,240*sum(L) + 55,296*sum(L^2) + 14,155,776*(2*Tmax-1) (valid frames only)."""
    s1 = sum(lengths)
    s2 = sum(v * v for v in lengths)
    pos = 0 if warm_pos_cache else 14_155_776 * (2 * max(lengths) - 1)
    return 326_154_240 * s1 + 55_296 * s2 + pos


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(bf16_tflops=p["bf16_tflops"], bf16_tflops_sustained=p.get("bf16_tflops_sustained"),
                    hbm_gbs=p["hbm_gbs"], source="measured")
    return dict(bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, hbm_gbs=6650.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "50"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = [v for v in sm if mx and v > 0.3 * mx] or sm
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def dump_outputs(directory, arrays):
    """arrays: name -> tensor; written as directory/<name>.npy in float32."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), t.detach().float().cpu().numpy())
    log(f"outputs of the last timed step written to {directory}: {', '.join(sorted(arrays))}")


def log(msg):
    sys.stderr.write(f"[bench +{time.perf_counter() - _T0:7.2f}s] {msg}\n")
    sys.stderr.flush()


_T0 = time.perf_counter()


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


# ------------------------------------------------------------------------------------------------ CPU arm
class CpuEncoder:
    """The reference's own CPU implementation of the path when oracle/_ref was built (kind "reference": the unmodified
    espnet modules, copied by oracle/build_ref.py), else the CPU restatement oracle/conformer_oracle.py (kind "port").
    Same synthetic weights and inputs as the GPU arm; eval mode, no_grad, fp32."""

    def __init__(self, cfg):
        self.cfg = cfg
        self.sd = encoder_state_dict(0, **cfg)
        self.kind = "port"
        self.enc = None
        try:
            from oracle.build_ref import available, import_reference_encoder
            if available():
                Ref, _ = import_reference_encoder()
                enc = Ref(attention_dim=cfg["d_model"], attention_heads=cfg["n_heads"], linear_units=cfg["linear_units"],
                          num_blocks=cfg["num_blocks"], cnn_module_kernel=cfg["cnn_kernel"])
                enc.load_state_dict(self.sd, strict=True)
                self.enc = enc.eval()
                self.kind = "reference"
        except Exception as e:      # noqa: BLE001 -- any import problem falls back to the port, loudly
            log(f"oracle/_ref unusable ({type(e).__name__}: {e}); timing the CPU port instead")
        if self.enc is None:
            from oracle import conformer_oracle as O
            self.O = O

    def forward(self, xs, lengths):
        with torch.no_grad():
            if self.enc is not None:
                mask = non_pad_mask(lengths, "cpu")
                return self.enc(xs, mask)[0]
            return self.O.encoder_forward(self.sd, xs, lengths, self.cfg["n_heads"])


def pick_threads(lengths):
    """Both CPU implementations are many mid-sized torch ops; on a many-core host all-threads is far from optimal (128
    threads were 30x slower than 32 on the first B200 box).  Probe a 1-layer forward at a few thread counts and keep
    the fastest: 'all the host threads it can use' productively."""
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (4, 8, 16, 32, 64, ncpu) if c <= ncpu})
    cpu1 = CpuEncoder(dict(CFG, num_blocks=1))
    xs = encoder_input(lengths, CFG["d_model"], 1234)
    best, best_t, worse = cands[0], float("inf"), 0
    for c in cands:
        torch.set_num_threads(c)
        cpu1.forward(xs, lengths)
        t0 = time.perf_counter()
        cpu1.forward(xs, lengths)
        dt = time.perf_counter() - t0
        log(f"cpu probe ({cpu1.kind}): {c} threads -> {dt * 1e3:.0f} ms / layer")
        if dt < best_t:
            best, best_t, worse = c, dt, 0
        else:
            worse += 1
            if worse >= 2:
                break
    return best


def cpu_time(lengths, repeats, threads):
    """Best-of-`repeats` wall time of one full forward on `threads` host threads -> (seconds, kind)."""
    torch.set_num_threads(threads)
    cpu = CpuEncoder(CFG)
    xs = encoder_input(lengths, CFG["d_model"], 1234)
    t0 = time.perf_counter()
    cpu.forward(xs, lengths)                                        # warm-up
    warm = time.perf_counter() - t0
    best = float("inf")
    for _ in range(repeats if warm < 8 else 1):                     # bounded: ~10-30 s of CPU work in total
        t0 = time.perf_counter()
        cpu.forward(xs, lengths)
        best = min(best, time.perf_counter() - t0)
    return best, cpu.kind


def run_reference(args):
    rank, _, world = dist_env()
    if rank != 0:
        return
    lengths = list(SHAPES[WORKLOAD])
    threads = pick_threads(lengths)
    torch.set_num_threads(threads)
    cpu = CpuEncoder(CFG)
    xs = encoder_input(lengths, CFG["d_model"], 1234)
    cpu.forward(xs, lengths)                                        # warm-up (1 forward; each is a full S2 bucket)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = cpu.forward(xs, lengths)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"encoder_out": out, "masks": non_pad_mask(lengths, "cpu")})
    fps = sum(lengths) * args.steps / dt
    note = ("the reference's own espnet ConformerEncoder (oracle/_ref: unmodified copy made by oracle/build_ref.py)"
            if cpu.kind == "reference" else
            "CPU restatement of the reference encoder (oracle/, pinned to reference golden vectors)")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_string(), "impl_note": note + "; rank 0 only, host cores"},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "host_cpus": os.cpu_count(), "kind": cpu.kind,
                         "sample": f"{args.steps} full forwards of workload {WORKLOAD} (1600 frames each)"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------------ GPU arm
def kernel_roofline(dev, peaks, precision):
    """Dominant kernel = the tcgen05 GEMM (92% of the forward's algorithmic FLOPs).  Times its largest instance, the
    FFN w_1 projection (1600 x 3072 x 768, bias+ReLU epilogue, operand-typed output; 24 launches per forward), over
    24 distinct weight matrices back to back with CUDA events on the launch stream, operands already in operand
    storage exactly as inside the encoder; achieved = algorithmic 2*M*N*K per launch / mean launch duration."""
    import ctypes as C
    from auto_avsr_b200 import _cabi
    from auto_avsr_b200.engine import PRECISIONS
    M, N, K = 1600, 3072, 768
    tdt = torch.float16 if precision == "f16" else torch.float32
    g = torch.Generator().manual_seed(7)
    x = torch.randn(M, K, generator=g).to(dev).to(tdt)
    ws = [((torch.rand(N, K, generator=g) - 0.5) * 0.07).to(dev).to(tdt) for _ in range(24)]
    b = torch.zeros(N, device=dev)
    y = torch.empty(M, N, device=dev, dtype=tdt)
    st = torch.cuda.current_stream(dev).cuda_stream

    def launch(w):
        nonlocal st
        _cabi.check(_cabi.lib.avsr_linear_operands(x.data_ptr(), w.data_ptr(), b.data_ptr(), None, 0.0, y.data_ptr(),
                                                   M, N, K, 1, 1, PRECISIONS[precision], st))
    for w in ws[:3]:
        launch(w)
    torch.cuda.synchronize(dev)
    # replay the 24 launches from a CUDA graph (as the encoder does): the python/ctypes launch path (~10 us) would
    # otherwise be what is timed, not the kernel
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        st = torch.cuda.current_stream(dev).cuda_stream
        for w in ws:
            launch(w)
    graph.replay()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 4
    e0.record()
    for _ in range(reps):
        graph.replay()
    e1.record()
    torch.cuda.synchronize(dev)
    per_launch_s = e0.elapsed_time(e1) * 1e-3 / (reps * len(ws))
    flops = 2.0 * M * N * K
    achieved = flops / per_launch_s / 1e12
    peak = peaks["bf16_tflops"]
    prof = os.path.join(ROOT, "profiles", "gemm_traffic.json")
    traffic = None
    if os.path.exists(prof):
        try:
            traffic = json.load(open(prof)).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    kind = "kind::f16, fp16 operands" if precision == "f16" else "kind::tf32"
    kname = ("gemm_tc2_kernel<EPI_LINEAR,384> (cta_group::2 pair tile 256x384, 56 clusters)" if precision == "f16"
             else "gemm_tc_kernel<EPI_LINEAR> (persistent, 1-CTA)")
    out = {"bound": "tensor", "kernel": f"{kname} FFN w_1 1600x3072x768 (tcgen05 {kind}, fp32 accumulate)",
           "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
           "peak_source": f"MEASURED_PEAKS.json bf16_tflops ({peaks['source']}, cuBLAS bf16 8192^3 burst)",
           "us_per_launch": per_launch_s * 1e6, "algorithmic_flops_per_launch": flops, "traffic": traffic}
    if precision == "tf32":
        out["frac_of_tf32_nominal"] = achieved / (0.5 * peak)
    return out


def time_forward(enc, xs, mask, steps, warm=6):
    """ms per forward of `enc` on device-resident inputs (CUDA events on the launch stream, after warm-up)."""
    with torch.no_grad():
        for _ in range(warm):
            enc(xs, mask)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            enc(xs, mask)
        e1.record()
        torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def extras(dev, enc, args, peaks):
    """Numbers that explain / frame the headline (none of them is the headline):
    shapes      device-resident frames/s of the other SURVEY.md section 8d shapes in the product arithmetic
    precisions  S2 in tf32 and fp32 modes (the fp32-class accuracy paths) next to f16
    sustained   S2 replayed back to back for >= 3 s, against MEASURED_PEAKS' sustained bf16 figure
    gpu_eager_baseline   the same op sequence in stock eager PyTorch on this GPU (cuBLAS / ATen kernels): the torch
                restatement oracle/conformer_oracle.py moved to cuda, fp32 with and without allow_tf32 -- SURVEY.md
                section 2b's per-kernel bar ("beat eager PyTorch-on-B200 of the same op sequence")."""
    out = {"shapes": {}, "precisions": {}}
    prec0 = enc.precision
    for name in ("S1", "S2r", "S3", "S4"):
        lengths = list(SHAPES[name])
        xs = encoder_input(lengths, CFG["d_model"], 1234).to(dev)
        mask = None if name == "S1" else non_pad_mask(lengths, dev)
        ms = time_forward(enc, xs, mask, 20)
        fl = algorithmic_flops(lengths)
        out["shapes"][name] = {"lengths": lengths if len(lengths) <= 5 else f"[{lengths[0]}]x{len(lengths)}",
                               "frames_per_s": sum(lengths) / (ms * 1e-3), "ms_per_step": ms,
                               "frac_of_bf16_peak": fl / (ms * 1e-3) / 1e12 / peaks["bf16_tflops"]}
        log(f"extras: {name} {ms:.3f} ms")
    lengths = list(SHAPES[WORKLOAD])
    xs = encoder_input(lengths, CFG["d_model"], 1234).to(dev)
    mask = non_pad_mask(lengths, dev)
    for prec, steps in (("tf32", 10), ("fp32", 3)):
        enc.precision = prec
        ms = time_forward(enc, xs, mask, steps, warm=3)
        out["precisions"][prec] = {"frames_per_s": sum(lengths) / (ms * 1e-3), "ms_per_step": ms}
        log(f"extras: S2 {prec} {ms:.3f} ms")
    enc.precision = prec0
    # sustained: >= 3 s of back-to-back replays (clocks settle to the sustained point)
    ms1 = time_forward(enc, xs, mask, 20)
    n = max(50, int(3200.0 / ms1))
    ms = time_forward(enc, xs, mask, n, warm=3)
    fl = algorithmic_flops(lengths)
    out["sustained"] = {"seconds": n * ms * 1e-3, "steps": n, "frames_per_s": sum(lengths) / (ms * 1e-3), "ms_per_step": ms,
                        "frac_of_bf16_sustained_peak": (fl / (ms * 1e-3) / 1e12 / peaks["bf16_tflops_sustained"])
                        if peaks.get("bf16_tflops_sustained") else None}
    log(f"extras: sustained {ms:.3f} ms/step over {n * ms * 1e-3:.1f} s")
    # BASELINE.json configs[2]: front-end features -> proj_encoder -> encoder -> CTC log-probs (the fused call of
    # auto_avsr_b200.head, SURVEY.md 8f #1); frames/s of the whole chain, device-resident synthetic features
    try:
        from auto_avsr_b200 import CTC, ProjEncoder
        from auto_avsr_b200.head import features_to_log_probs
        from auto_avsr_b200.synthetic import frontend_features, head_state_dict
        hsd = head_state_dict(0)
        proj = ProjEncoder(512, CFG["d_model"])
        proj.load_state_dict({"weight": hsd["proj_encoder.weight"], "bias": hsd["proj_encoder.bias"]})
        ctc = CTC(5049, CFG["d_model"], 0.1)
        ctc.load_state_dict({"ctc_lo.weight": hsd["ctc.ctc_lo.weight"], "ctc_lo.bias": hsd["ctc.ctc_lo.bias"]})
        proj, ctc = proj.to(dev).eval(), ctc.to(dev).eval()
        feats = frontend_features(lengths, 512, 4321).to(dev)
        with torch.no_grad():
            for _ in range(5):
                features_to_log_probs(proj, enc, ctc, feats, mask)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(20):
                features_to_log_probs(proj, enc, ctc, feats, mask)
            e1.record()
            torch.cuda.synchronize()
            ms_f = e0.elapsed_time(e1) / 20
            for _ in range(3):
                ctc.log_softmax(enc(proj(feats), mask)[0])
            torch.cuda.synchronize()
            e0.record()
            for _ in range(20):
                ctc.log_softmax(enc(proj(feats), mask)[0])
            e1.record()
            torch.cuda.synchronize()
            ms_m = e0.elapsed_time(e1) / 20
        out["configs2_features_to_ctc_logprobs"] = {
            "what": "BASELINE.json configs[2] (ASR Conformer-base encoder fwd + CTC head): synthetic (4, 400, 512) front-end "
                    "features -> proj_encoder -> 12-layer encoder -> ctc_lo (5049) + log_softmax; both paths replay CUDA graphs",
            "fused_call": {"frames_per_s": sum(lengths) / (ms_f * 1e-3), "ms_per_step": ms_f,
                           "api": "auto_avsr_b200.head.features_to_log_probs -> avsr_features_to_logprobs"},
            "module_by_module": {"frames_per_s": sum(lengths) / (ms_m * 1e-3), "ms_per_step": ms_m,
                                 "api": "ctc.log_softmax(encoder(proj_encoder(x), mask)[0]) (drop-in modules, encoder from its CUDA graph)"}}
        log(f"extras: configs[2] fused {ms_f:.3f} ms, module-by-module {ms_m:.3f} ms")
    except Exception as e:          # noqa: BLE001
        out["configs2_features_to_ctc_logprobs"] = {"error": f"{type(e).__name__}: {e}"}
    # config 1 caller replay (lightning.py:69-72): B = 1, masks None, a new T per utterance -> direct launches
    try:
        from auto_avsr_b200.shim import E2EShell, test_step_encoder
        shell = E2EShell()
        shell.encoder, shell.proj_encoder = enc, proj
        Ts = [100, 37, 251, 64, 180, 99, 33, 400, 12, 77, 313, 58, 129, 240, 91, 17, 365, 204, 146, 63]
        fs = [frontend_features([T], 512, 1000 + T)[0].to(dev) for T in Ts]
        with torch.no_grad():
            for f in fs[:3]:
                test_step_encoder(shell, f)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for f in fs:
                test_step_encoder(shell, f)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
        out["config1_eval_path"] = {"what": "ModelModule.test_step replay (proj_encoder -> encoder(x, None)), 20 utterances with 20 "
                                            "distinct lengths (12..400 frames), B = 1, wall clock incl. host overhead",
                                    "utterances_per_s": len(Ts) / dt, "frames_per_s": sum(Ts) / dt,
                                    "ms_per_utterance": dt / len(Ts) * 1e3,
                                    "engine_stats": dict(enc._engine.stats)}
        log(f"extras: config-1 replay {dt / len(Ts) * 1e3:.3f} ms / utterance")
    except Exception as e:          # noqa: BLE001
        out["config1_eval_path"] = {"error": f"{type(e).__name__}: {e}"}
    # training step of the encoder alone (SURVEY.md 8f #2): forward + backward in train() mode, reference dropout rates
    try:
        enc.train()
        xt = xs.clone().requires_grad_(False)
        for _ in range(2):
            enc.zero_grad(set_to_none=True)
            enc(xt, mask)[0].pow(2).mean().backward()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(3):
            enc.zero_grad(set_to_none=True)
            enc(xt, mask)[0].pow(2).mean().backward()
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / 3
        enc.zero_grad(set_to_none=True)
        enc.eval()
        out["train_step_encoder"] = {"what": "ConformerEncoder.train(): forward + backward of workload S2 (dropout 0.1, batch-stat "
                                             "BatchNorm), every module's forward and backward in libavsr_b200; correctness-first "
                                             "slice (fp32 CUDA-core attention backward, unfused module-by-module schedule)",
                                     "ms_per_step": dt * 1e3, "frames_per_s": sum(lengths) / dt}
        log(f"extras: train step {dt * 1e3:.1f} ms")
    except Exception as e:          # noqa: BLE001
        enc.eval()
        out["train_step_encoder"] = {"error": f"{type(e).__name__}: {e}"}
    # eager-PyTorch comparator on the same GPU (cuBLAS / ATen), same weights and inputs: the UNMODIFIED reference
    # modules moved to cuda when oracle/_ref was built, else the torch restatement (oracle/conformer_oracle.py)
    try:
        cpu = CpuEncoder(CFG)                          # baseline leg only: the comparator, never the product path
        if cpu.enc is not None:
            ref = cpu.enc.to(dev)
            run = lambda: ref(xs, mask)[0]             # noqa: E731
            what = "the reference's own espnet ConformerEncoder (oracle/_ref, unmodified) .to('cuda')"
        else:
            sd = {k: v.to(dev) for k, v in cpu.sd.items()}
            run = lambda: cpu.O.encoder_forward(sd, xs, lengths, CFG["n_heads"])   # noqa: E731
            what = "oracle/conformer_oracle.py (torch restatement of the reference encoder) on cuda"
        eager = {}
        for tf32 in (False, True):
            torch.backends.cuda.matmul.allow_tf32 = tf32
            torch.backends.cudnn.allow_tf32 = tf32
            with torch.no_grad():
                for _ in range(3):
                    run()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(10):
                    run()
                e1.record()
                torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / 10
            eager["tf32" if tf32 else "fp32"] = {"frames_per_s": sum(lengths) / (ms * 1e-3), "ms_per_step": ms}
            log(f"extras: eager PyTorch allow_tf32={tf32} {ms:.3f} ms")
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = False
        eager["what"] = what + ": stock eager PyTorch kernels (cuBLAS / cuDNN / ATen), device-resident inputs"
        out["gpu_eager_baseline"] = eager
    except Exception as e:          # noqa: BLE001
        out["gpu_eager_baseline"] = {"error": f"{type(e).__name__}: {e}"}
    # BASELINE.json configs[4] flavour (SURVEY.md 8f #3): beam-search decoding of one utterance on the drop-in scorers vs
    # the unmodified reference on the same GPU.  Runs LAST and in a CHILD process with its own CUDA context and timeout
    # (scripts/bench_decode.py): whatever happens there cannot touch the headline measurement above.
    try:
        import subprocess
        torch.cuda.synchronize()
        r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "bench_decode.py"), "100", "40"], capture_output=True,
                           text=True, timeout=150, cwd=ROOT)
        rows = [ln for ln in r.stdout.splitlines() if ln.startswith("DECODE-JSON ")]
        out["decode_beam_search"] = json.loads(rows[-1][len("DECODE-JSON "):]) if rows else \
            {"error": f"child rc={r.returncode}: {(r.stderr or r.stdout)[-400:]}"}
        log("extras: decode child done")
    except Exception as e:          # noqa: BLE001
        out["decode_beam_search"] = {"error": f"{type(e).__name__}: {e}"}
    return out


def run_ours(args):
    rank, local_rank, world = dist_env()
    assert torch.cuda.is_available(), "bench.py needs a GPU (the encoder path has no CPU fallback)"
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from auto_avsr_b200 import ConformerEncoder, _cabi

    lengths = list(SHAPES[WORKLOAD])
    B, T, D = len(lengths), max(lengths), CFG["d_model"]
    enc = ConformerEncoder(attention_dim=D, attention_heads=CFG["n_heads"], linear_units=CFG["linear_units"],
                           num_blocks=CFG["num_blocks"], cnn_module_kernel=CFG["cnn_kernel"])
    enc.load_state_dict(encoder_state_dict(0, **CFG), strict=True)
    enc = enc.to(dev).eval()
    enc.precision = args.precision
    enc.assume_frozen = True
    mask = non_pad_mask(lengths, dev)
    nbuf = 4     # rotating inputs; the 682 MB of weights streamed every step already exceed the 126 MB L2
    host_in = [encoder_input(lengths, D, 1234 + rank * 100 + i).pin_memory() for i in range(nbuf)]
    dev_in = [h.to(dev) for h in host_in]
    host_out = torch.empty(B, T, D).pin_memory()
    host_len = torch.tensor(lengths, dtype=torch.int32).pin_memory()

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize(dev)

    log("model + inputs on device")
    # clocks / throttle reasons are sampled from before the warm-up until after the e2e region: the timed regions are
    # a few hundred ms, shorter than nvidia-smi's start-up, so the sampler must already be running when they begin
    sampler = ClockSampler(local_rank)
    sampler.start()
    with torch.no_grad():
        t_w = time.perf_counter()
        i = 0
        while i < max(args.warmup, 3) or (time.perf_counter() - t_w < 0.6 and len(sampler.rows) < 4):
            enc(dev_in[i % nbuf], mask)
            i += 1
            if i % 16 == 0:
                torch.cuda.synchronize(dev)
        barrier()
        n_warm = i
        log(f"warm-up done ({n_warm} untimed steps)")
        # ---- device-resident timing: CUDA events on the launch stream
        l0 = _cabi.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(args.steps):
            out = enc(dev_in[i % nbuf], mask)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        launches = _cabi.launch_count() - l0
        log(f"device-timed region done: {ms / args.steps:.3f} ms/step")
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, {"encoder_out": out[0], "masks": out[1]})
        # ---- end to end through the public API: every step copies its inputs from pinned host memory (H2D), runs
        # ConformerEncoder.forward, and copies the features back to pinned host memory (D2H).  PipelinedEncoder
        # (auto_avsr_b200/pipeline.py) overlaps the copies of neighbouring steps with the forward on 3 streams.
        from auto_avsr_b200.pipeline import PipelinedEncoder
        pipe = PipelinedEncoder(enc, B, T, depth=2, device=dev)
        host_outs = [torch.empty(B, T, D).pin_memory() for _ in range(2)]
        ins = [host_in[i % nbuf] for i in range(args.steps)]
        lens = [host_len for _ in range(args.steps)]
        outs = [host_outs[i % 2] for i in range(args.steps)]
        pipe.run(ins[:3], lens[:3], outs[:3])
        pipe.synchronize()
        barrier()
        t0 = time.perf_counter()
        pipe.run(ins, lens, outs)
        pipe.synchronize()
        e2e_s = time.perf_counter() - t0
        barrier()
        clocks = sampler.stop()
        log(f"e2e region done: {e2e_s / args.steps * 1e3:.3f} ms/step")

    t_ms = torch.tensor([ms, e2e_s * 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_max, e2e_ms_max = t_ms.tolist()
    frames = sum(lengths) * args.steps * world
    value = frames / (ms_max * 1e-3)
    e2e_value = frames / (e2e_ms_max * 1e-3)

    if rank == 0:
        peaks = measured_peaks()
        line = {
            "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": {"f16": "f16 operands, f32 accumulate (f32 residual/LN/softmax)", "tf32": "tf32 operands, f32 accumulate",
                      "fp32": "f32"}[args.precision], "data": "synthetic",
            "config": {"workload": workload_string(),
                       "global_frames_per_step": sum(lengths) * world, "parallelism": f"dp{world} (one bucket per GPU, "
                                                                                       "no data-path collective)",
                       "l2": "682 MB of weights streamed per step > 126 MB L2; 4 rotating input buffers",
                       "pos_cache": "cold: linear_pos(pos_emb) recomputed every step", "precision": args.precision,
                       "assume_frozen": True, "graph_after": enc._engine.graph_after,
                       "untimed_steps_before_timing": n_warm},
            "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": B * T * D * 4 + B * 4,
                    "d2h_bytes_per_step": B * T * D * 4, "ms_per_step": e2e_ms_max / args.steps,
                    "api": "auto_avsr_b200.pipeline.PipelinedEncoder.run -> ConformerEncoder.forward(xs, masks) -> "
                           "avsr_plan_forward (C ABI); H2D / D2H of neighbouring steps overlap the forward"},
            "gpu_launches": int(launches), "clocks": clocks,
            "forward_model": {"algorithmic_gflop_per_step": algorithmic_flops(lengths) / 1e9,
                              "achieved_tflops": algorithmic_flops(lengths) / (ms_max / args.steps * 1e-3) / 1e12,
                              "frac_of_bf16_peak": algorithmic_flops(lengths) / (ms_max / args.steps * 1e-3) / 1e12
                              / peaks["bf16_tflops"]},
        }
        if args.precision != "fp32":
            line["roofline"] = kernel_roofline(dev, peaks, args.precision)
            log("kernel roofline done")
        if world == 1 and not args.no_extras:
            line["extras"] = extras(dev, enc, args, peaks)
        if world == 1 and not args.no_cpu:
            threads = pick_threads(lengths)
            best, kind = cpu_time(lengths, repeats=3, threads=threads)
            log(f"cpu baseline ({kind}) done: {best:.3f} s/forward on {threads} threads")
            line["cpu_baseline"] = {"value": sum(lengths) / best, "unit": "frames/s", "cores": threads, "host_cpus": os.cpu_count(),
                                    "kind": kind, "sample": f"best of 3 full forwards of workload {WORKLOAD} (1600 frames), fp32, "
                                              "after 1 warm-up"}
        print(json.dumps(line))
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("AVSR_B200_PRECISION", "f16"),
                    choices=["f16", "tf32", "fp32"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extras", action="store_true", help="skip the extras (other shapes / precisions, sustained "
                                                               "loop, eager-PyTorch GPU comparator)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy "
                                                           "(float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
