"""Host-side / boundary checks that need no GPU: the C-ABI library loads and exports every symbol the header
declares, the drop-in modules honour the reference's state-dict contract, install() shadows the reference's
import path, and the product refuses to run on the CPU instead of falling back."""
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "avsr_b200.h")


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()
    return g.LIB


def _header_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(avsr_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol(built):
    syms = _header_symbols()
    assert len(syms) >= 17
    out = subprocess.run(["nm", "-D", "--defined-only", built], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r" T (avsr_[a-z0-9_]+)", out))
    assert set(syms) <= exported, sorted(set(syms) - exported)
    from auto_avsr_b200 import _cabi
    assert set(_cabi.SIGNATURES) == set(syms)
    assert _cabi.lib.avsr_abi_version() == _cabi.ABI_VERSION == 10
    assert _cabi.launch_count() == 0


def test_sizes_and_argument_errors_without_gpu(built):
    import ctypes as C
    from auto_avsr_b200 import _cabi
    cfg = _cabi.EncoderConfig(768, 12, 3072, 12, 31)
    pb = _cabi.lib.avsr_prepared_bytes(C.byref(cfg))
    assert pb >= 170_451_456 * 4 - 12 * 768 * 4 * 8          # >= the fp32 parameter bytes it re-lays out
    assert _cabi.lib.avsr_workspace_bytes(C.byref(cfg), 4, 400) > 0
    assert _cabi.lib.avsr_workspace_bytes(C.byref(cfg), 0, 400) == 256
    bad = _cabi.EncoderConfig(768, 8, 3072, 12, 31)           # d_k != 64
    assert _cabi.lib.avsr_prepared_bytes(C.byref(bad)) == 0
    assert b"d_model" in _cabi.lib.avsr_last_error()
    with pytest.raises(_cabi.AvsrError):
        _cabi.check(_cabi.lib.avsr_layernorm(None, None, None, None, 4, 768, None))
    # log-softmax entry: NULL input, row stride shorter than the row, and the empty batch (a no-op, no launch)
    with pytest.raises(_cabi.AvsrError):
        _cabi.check(_cabi.lib.avsr_log_softmax(None, 8, None, 8, None, 1, 8, None))
    with pytest.raises(_cabi.AvsrError, match="ldx"):
        _cabi.check(_cabi.lib.avsr_log_softmax(0x1000, 4, 0x2000, 8, None, 1, 8, None))
    before = _cabi.launch_count()
    _cabi.check(_cabi.lib.avsr_log_softmax(0x1000, 8, 0x2000, 8, None, 0, 8, None))
    assert _cabi.launch_count() == before


def test_state_dict_contract(built, golden_dir):
    from auto_avsr_b200 import ConformerEncoder
    enc = ConformerEncoder()
    want = [l.split() for l in open(os.path.join(golden_dir, "encoder_state_keys.txt"))]
    got = enc.state_dict()
    assert [w[0] for w in want] == list(got.keys())
    assert len(got) == 482
    for w in want:
        assert tuple(int(v) for v in w[1:]) == tuple(got[w[0]].shape), w[0]
    assert sum(p.numel() for p in enc.parameters()) == 170_451_456
    assert isinstance(enc.encoders[0].conv_module.norm, torch.nn.BatchNorm1d)
    # legacy checkpoint key renames (conformer_encoder.py:173-183)
    sd = {("norm." + k[len("after_norm."):] if k.startswith("after_norm.") else k): v for k, v in got.items()}
    enc2 = ConformerEncoder()
    enc2.load_state_dict(sd, strict=True)


def test_no_cpu_fallback(built):
    from auto_avsr_b200 import ConformerEncoder
    from auto_avsr_b200.espnet_dropin import LayerNorm, PositionwiseFeedForward
    enc = ConformerEncoder(num_blocks=1).eval()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        enc(torch.zeros(1, 8, 768), None)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        LayerNorm(768)(torch.zeros(2, 768))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        PositionwiseFeedForward(768, 3072, 0.1).eval()(torch.zeros(2, 768))
    enc.train()                                   # training runs in the library too (round 2): still no CPU path
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        enc(torch.zeros(1, 8, 768), None)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        PositionwiseFeedForward(768, 3072, 0.1).train()(torch.zeros(2, 768))


def test_missing_library_fails_loudly(built):
    """Without the built CUDA library the package must not import (AVSR_B200_LIB points the loader at another
    build of the same library; a path that does not exist is the 'extension missing' case)."""
    r = subprocess.run([sys.executable, "-c", "import auto_avsr_b200._cabi"], cwd=ROOT, capture_output=True, text=True,
                       env=dict(os.environ, AVSR_B200_LIB="/nonexistent/libavsr_b200.so"), timeout=120)
    assert r.returncode != 0
    assert "ImportError" in r.stderr and "no CPU / PyTorch fallback" in r.stderr


def test_trace_hooks_are_absent_from_the_product_build(built):
    """The phase-trace instrumentation (scripts/build_trace.py, -DAVSR_TRACE) is a separate diagnostic build."""
    import ctypes
    lib = ctypes.CDLL(built)
    assert not hasattr(lib, "avsr_trace_set")


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "auto_avsr_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                txt = open(os.path.join(dp, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), f
                assert "/root/reference" not in txt.replace("(``/root/reference``", ""), f


def test_install_shadows_reference_import_path(built):
    """install() answers the reference's import paths with the drop-in (e2e_asr_conformer.py:12 and the north_star spelling),
    re-points an E2E module imported before it, and the encoder part of the reference E2E(5049, "audio") state dict
    (tests/golden/reference_surfaces.json) loads strictly, also with lightning.py:41-42's 'encoder.' prefix stripped."""
    code = f"""
import json, sys, types
sys.path.insert(0, {ROOT!r})
import torch
import auto_avsr_b200
early = types.ModuleType("espnet.nets.pytorch_backend.e2e_asr_conformer"); early.ConformerEncoder = object
sys.modules[early.__name__] = early                 # an E2E module imported before install()
auto_avsr_b200.install()
from espnet.nets.pytorch_backend.encoder.conformer_encoder import ConformerEncoder
from espnet.nets.pytorch_backend.conformer.encoder import Encoder
assert ConformerEncoder.__module__ == "auto_avsr_b200.espnet_dropin.conformer_encoder", ConformerEncoder.__module__
assert Encoder is ConformerEncoder is early.ConformerEncoder is auto_avsr_b200.ConformerEncoder
from auto_avsr_b200.install import is_installed
assert is_installed()
golden = json.load(open({os.path.join(ROOT, "tests", "golden", "reference_surfaces.json")!r}))["e2e_audio"]
enc = {{k[len("encoder."):]: s for k, s in golden["state"] if k.startswith("encoder.")}}
e = ConformerEncoder()
e.load_state_dict({{k: torch.zeros(s) for k, s in enc.items()}}, strict=True)
buffers = ("running_mean", "running_var", "num_batches_tracked")
assert sum(p.numel() for p in e.parameters()) == sum(torch.Size(s).numel() for k, s in enc.items() if not k.endswith(buffers))
print("OK", golden["n_parameters"])
"""
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "OK 243049202" in r.stdout      # audio E2E parameter count, README.md:124-125 / BASELINE.md section 2


# ------------------------------------------------------------------ steps either side of the encoder (8f #1)
def test_head_dropins_keep_the_reference_state_dict_keys_and_refuse_cpu(built):
    from auto_avsr_b200 import CTC, ProjEncoder
    from auto_avsr_b200.synthetic import head_state_dict
    sd = head_state_dict(3)
    ctc = CTC(5049, 768, 0.1, reduce=True)
    proj = ProjEncoder(512, 768)
    ctc.load_state_dict({"ctc_lo.weight": sd["ctc.ctc_lo.weight"], "ctc_lo.bias": sd["ctc.ctc_lo.bias"]}, strict=True)
    proj.load_state_dict({"weight": sd["proj_encoder.weight"], "bias": sd["proj_encoder.bias"]}, strict=True)
    assert list(ctc.state_dict()) == ["ctc_lo.weight", "ctc_lo.bias"]
    assert (ctc.reduce, ctc.ignore_id, ctc.dropout_rate, ctc.ctc_loss.reduction) == (True, -1, 0.1, "sum")
    ctc.eval(); proj.eval()
    for call in (lambda: ctc.log_softmax(torch.zeros(1, 3, 768)), lambda: ctc.softmax(torch.zeros(1, 3, 768)),
                 lambda: ctc.argmax(torch.zeros(1, 3, 768)), lambda: proj(torch.zeros(1, 3, 512))):
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            call()
    with pytest.raises(NotImplementedError):
        ctc(torch.zeros(1, 3, 768), torch.tensor([3]), torch.zeros(1, 2, dtype=torch.long))
    ctc.train()
    with pytest.raises(NotImplementedError, match="inference"):
        ctc.log_softmax(torch.zeros(1, 3, 768))
    # the prepared (padded, operand-typed) copy lives in the library and is rebuilt when a parameter's version moves
    from auto_avsr_b200.head import PreparedHead
    w = ctc.ctc_lo.weight
    fp0 = PreparedHead._fp(w, ctc.ctc_lo.bias)
    with torch.no_grad():
        w.add_(1.0)
    assert PreparedHead._fp(w, ctc.ctc_lo.bias) != fp0
    from auto_avsr_b200 import _cabi
    import ctypes as C
    cfg = _cabi.EncoderConfig(768, 12, 3072, 12, 31)
    need = _cabi.lib.avsr_head_prepared_bytes(C.byref(cfg), 512, 5049)
    assert need >= (2 * 768 * 512 + 5120 * 768) * 2          # two proj copies + ctc_lo padded to 5120 rows
    assert _cabi.lib.avsr_head_workspace_bytes(C.byref(cfg), 4, 400, 512, 5049) > 1600 * 5120 * 4
    assert _cabi.lib.avsr_ctc_workspace_bytes(C.byref(cfg), 1600, 5049) > 1600 * 5120 * 4


def test_install_head_rehomes_the_reference_modules(built):
    """install_head on a shell with the two members E2E.__init__ builds; the reference CTC module is stood in for by a
    module with its state dict and the attributes install_head reads (tests/golden/reference_surfaces.json)."""
    code = f"""
import json, sys
sys.path.insert(0, {ROOT!r})
import torch
import auto_avsr_b200
golden = json.load(open({os.path.join(ROOT, "tests", "golden", "reference_surfaces.json")!r}))["ctc"]

class RefCTC(torch.nn.Module):         # the reference CTC's state dict and the attributes install_head reads
    def __init__(self):
        super().__init__()
        (_, (odim, adim)), _ = golden["state"]
        self.ctc_lo = torch.nn.Linear(adim, odim)
        self.dropout_rate, self.reduce = golden["dropout_rate"], golden["reduce"]

class Shell(torch.nn.Module):          # the two members E2E.__init__ builds (e2e_asr_conformer.py:31, :56)
    def __init__(self):
        super().__init__()
        self.proj_encoder = torch.nn.Linear(512, 768)
        self.ctc = RefCTC()

m = Shell().eval()
before = {{k: v.data_ptr() for k, v in m.state_dict().items()}}
params = {{id(p) for p in m.parameters()}}
auto_avsr_b200.install_head(m)
assert type(m.proj_encoder).__module__ == "auto_avsr_b200.espnet_dropin.ctc"
assert type(m.ctc).__module__ == "auto_avsr_b200.espnet_dropin.ctc"
after = {{k: v.data_ptr() for k, v in m.state_dict().items()}}
assert before == after, (before.keys(), after.keys())
assert params == {{id(p) for p in m.parameters()}}
assert not m.ctc.training and not m.proj_encoder.training
assert [[k, list(v.shape)] for k, v in m.ctc.state_dict().items()] == golden["state"]
assert (m.ctc.dropout_rate, m.ctc.reduce) == (golden["dropout_rate"], golden["reduce"])
print("OK")
"""
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout + r.stderr[-2000:]


def test_mask_to_lengths_prefix_check():
    """ADVICE r01: a key mask that is not prefix-contiguous cannot be expressed as lengths; check=True raises."""
    import torch
    from auto_avsr_b200.espnet_dropin.attention import mask_to_lengths
    ok = torch.tensor([[[1, 1, 1, 0, 0]], [[1, 1, 1, 1, 1]]], dtype=torch.bool)
    assert mask_to_lengths(ok, 2, 5, check=True).tolist() == [3, 5]
    bad = torch.tensor([[[1, 0, 1, 0, 0]], [[1, 1, 1, 1, 1]]], dtype=torch.bool)
    assert mask_to_lengths(bad, 2, 5).tolist() == [2, 5]            # unchecked: silently a prefix of 2 (documented)
    with pytest.raises(NotImplementedError):
        mask_to_lengths(bad, 2, 5, check=True)
