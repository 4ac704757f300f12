"""Host logic of row 8f #3 on the CPU: the TransformerDecoder / CTCPrefixScorer drop-ins and the device beam loop keep
the reference's surface (state-dict keys, scorer API, n-best of the search) -- driven through tests/emu's host replay of
the library schedule, against the reference-generated fixtures; and the reference's OWN BatchBeamSearch (oracle/_ref,
unmodified) drives the drop-in scorers to the same n-best.  The product path refuses CPU tensors."""
import os
import subprocess
import sys

import pytest
import torch

from helpers import load_decoder_case

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_COPY = os.path.join(ROOT, "oracle", "_ref")
HAVE_NVCC = os.path.exists("/usr/local/cuda/bin/nvcc")
needs_emu = pytest.mark.skipif(not HAVE_NVCC, reason="nvcc is needed to build the host replay")


class CpuCTC(torch.nn.Module):
    """stands in for the CTC module in front of the prefix scorer in the emulated runs (ctc.py:77-84)"""

    def __init__(self, head_sd):
        super().__init__()
        w, b = head_sd["ctc.ctc_lo.weight"], head_sd["ctc.ctc_lo.bias"]
        self.ctc_lo = torch.nn.Linear(w.shape[1], w.shape[0])
        self.ctc_lo.load_state_dict({"weight": w, "bias": b})

    @torch.no_grad()
    def log_softmax(self, hs):
        return torch.log_softmax(self.ctc_lo(hs), dim=-1)


def _dropin_decoder(c, lib=None):
    from auto_avsr_b200 import TransformerDecoder
    cfg = c["cfg"]
    dec = TransformerDecoder(cfg["odim"], cfg["d_model"], cfg["n_heads"], cfg["linear_units"], cfg["num_blocks"])
    dec.load_state_dict(c["dec_sd"], strict=True)
    dec.eval()
    dec.precision = "fp32"
    dec._lib = lib
    return dec


def test_decoder_dropin_state_dict_contract_and_cpu_refusal():
    from auto_avsr_b200 import CTCPrefixScorer, TransformerDecoder
    from auto_avsr_b200.synthetic import decoder_state_dict
    dec = TransformerDecoder(odim=5049, attention_dim=768, attention_heads=12, linear_units=3072, num_blocks=6)   # e2e_asr_conformer.py:41-47
    sd = decoder_state_dict(0)
    assert list(dec.state_dict().keys()) == list(sd.keys())
    assert len(sd) == 6 * 26 + 5 and sum(v.numel() for v in sd.values()) == sum(p.numel() for p in dec.parameters())
    dec.load_state_dict(sd, strict=True)
    # the pre-3d422f6 spelling of after_norm is renamed on load (transformer_decoder.py:143-156)
    old = {k.replace("after_norm.", "output_norm."): v for k, v in sd.items()}
    dec.load_state_dict(old, strict=True)
    dec.eval()
    ys = torch.tensor([[5048]])
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        dec.batch_score(ys, [None], torch.zeros(1, 7, 768))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        dec.score(ys[0], None, torch.zeros(7, 768))
    for call in (lambda: dec(ys, None, torch.zeros(1, 7, 768), None), lambda: dec.forward_one_step(ys, None, torch.zeros(1, 7, 768))):
        with pytest.raises(NotImplementedError):
            call()
    dec.train()
    with pytest.raises(NotImplementedError, match="inference"):
        dec.batch_score(ys, [None], torch.zeros(1, 7, 768))
    with pytest.raises(NotImplementedError):
        TransformerDecoder(10, 64, 1, 64, 1, concat_after=True)
    sc = CTCPrefixScorer(torch.nn.Identity(), 9)
    assert sc.select_state(None, 0) is None and sc.select_state([1, 2, 3], 1) == 2
    with pytest.raises(RuntimeError, match="before batch_init_state"):
        sc.batch_score_partial(torch.zeros(1, 1, dtype=torch.long), torch.zeros(1, 2, dtype=torch.long), [None], None)
    with pytest.raises(NotImplementedError):
        sc.init_state(torch.zeros(3, 4))


def _check_nbest(nbest, z, tag, tol):
    """same hypotheses in the same order as the reference's n-best (fixture keeps the first 10), scores within tol"""
    assert len(nbest) == int(z[f"nbest_count_{tag}"])
    for i in range(len(z[f"nbest_len_{tag}"])):
        L = int(z[f"nbest_len_{tag}"][i])
        h = nbest[i]
        assert h["yseq"] == z[f"nbest_yseq_{tag}"][i, :L].tolist(), i
        assert abs(h["score"] - float(z[f"nbest_score_{tag}"][i])) < tol
        assert abs(h["scores"]["decoder"] - float(z[f"nbest_dec_{tag}"][i])) < tol
        assert abs(h["scores"]["ctc"] - float(z[f"nbest_ctc_{tag}"][i])) < tol


@needs_emu
def test_device_beam_search_reproduces_the_reference_nbest_on_the_host_replay():
    from auto_avsr_b200.beam_search import DeviceBeamSearch
    from emu import build
    c = load_decoder_case("decoder_tiny")
    cfg = c["cfg"]
    dec = _dropin_decoder(c, build.load())
    bs = DeviceBeamSearch(dec, CpuCTC(c["head_sd"]), beam_size=cfg["beam"], vocab_size=cfg["odim"])
    nbest = [h.asdict() for h in bs(c["memory"])]
    _check_nbest(nbest, c["z"], "f32", 2e-3)
    assert bs.stats["utterances"] == 1 and dec.engine().stats["begin"] == 1
    assert dec.engine().stats["step"] == bs.stats["steps"] <= cfg["T"]
    # a second utterance re-uses the prepared weights and the session
    nbest2 = [h.asdict() for h in bs(c["memory"])]
    assert [h["yseq"] for h in nbest2] == [h["yseq"] for h in nbest]
    assert dec.engine().stats["prepare"] == 1 and dec.engine().stats["begin"] == 2
    # no CTC scorer (ctc_weight 0): pure attention-decoder search still terminates with <eos>-closed hypotheses
    plain = DeviceBeamSearch(dec, None, beam_size=3, vocab_size=cfg["odim"], ctc_weight=0.0)(c["memory"][:6])
    assert plain and all(int(h.yseq[-1]) == cfg["odim"] - 1 for h in plain)


@needs_emu
@pytest.mark.skipif(not os.path.isdir(os.path.join(REF_COPY, "espnet")), reason="oracle/_ref not built")
def test_reference_batch_beam_search_drives_the_dropin_scorers():
    """The UNMODIFIED reference BatchBeamSearch (oracle/_ref copy), configured like get_beam_search_decoder
    (lightning.py:126-157), with the drop-in TransformerDecoder + CTCPrefixScorer as its scorers."""
    code = f"""
import sys
sys.path.insert(0, {ROOT!r}); sys.path.insert(0, {os.path.join(ROOT, "tests")!r})
from oracle import build_ref
ref = build_ref.import_reference_search()
import torch
from helpers import load_decoder_case
from test_decoder_dropin_cpu import CpuCTC, _dropin_decoder, _check_nbest
from auto_avsr_b200 import CTCPrefixScorer, TransformerDecoder
from auto_avsr_b200.espnet_dropin import scorer_interface
from espnet.nets.scorer_interface import BatchPartialScorerInterface, BatchScorerInterface
assert scorer_interface.rebind()
assert issubclass(TransformerDecoder, BatchScorerInterface) and issubclass(CTCPrefixScorer, BatchPartialScorerInterface)
from emu import build
c = load_decoder_case("decoder_tiny")
cfg = c["cfg"]
lib = build.load()
dec = _dropin_decoder(c, lib)
ctc = CTCPrefixScorer(CpuCTC(c["head_sd"]), cfg["odim"] - 1)
ctc._lib = lib
token_list = [str(i) for i in range(cfg["odim"])]
scorers = dict(decoder=dec, ctc=ctc, lm=None, length_bonus=ref["LengthBonus"](len(token_list)))
weights = dict(decoder=0.9, ctc=0.1, lm=0.0, length_bonus=0)
bs = ref["BatchBeamSearch"](beam_size=cfg["beam"], vocab_size=len(token_list), weights=weights, scorers=scorers,
                            sos=cfg["odim"] - 1, eos=cfg["odim"] - 1, token_list=token_list, pre_beam_score_key="decoder")
with torch.no_grad():
    nbest = [h.asdict() for h in bs(c["memory"])]
_check_nbest(nbest, c["z"], "f32", 2e-3)
print("OK", len(nbest), dec.engine().stats)
"""
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]


def _module_from_parameter_names(named_shapes):
    """A module tree with exactly these parameter names and shapes (numbered children in a Sequential)."""
    root = torch.nn.Module()
    for name, shape in named_shapes:
        *path, leaf = name.split(".")
        mod = root
        for i, part in enumerate(path):
            if part not in mod._modules:
                nxt = path[i + 1] if i + 1 < len(path) else leaf
                mod.add_module(part, torch.nn.Sequential() if nxt.isdigit() else torch.nn.Module())
            mod = mod._modules[part]
        mod.register_parameter(leaf, torch.nn.Parameter(torch.randn(shape)))
    return root


def test_install_decoder_rehomes_the_reference_decoder():
    """install_decoder on a shell with the members of E2E the decoding path touches (e2e_asr_conformer.py:41-59); the
    reference TransformerDecoder(odim=37, attention_dim=128, attention_heads=2, linear_units=256, num_blocks=2) is stood in
    for by a module with its parameter names and shapes and the attributes install_decoder reads
    (tests/golden/reference_surfaces.json)."""
    import json
    import auto_avsr_b200
    from auto_avsr_b200.espnet_dropin import scorer_interface
    with open(os.path.join(ROOT, "tests", "golden", "reference_surfaces.json")) as f:
        golden = json.load(f)["decoder"]
    ref_dec = _module_from_parameter_names(golden["parameters"])
    emb = ref_dec.embed[0]
    emb.num_embeddings, emb.embedding_dim = emb.weight.shape
    ref_dec.decoders[0].self_attn.h = golden["attention_heads"]
    ref_dec.decoders[0].feed_forward.w_1.out_features = ref_dec.decoders[0].feed_forward.w_1.weight.shape[0]
    m = torch.nn.Module()
    m.decoder = ref_dec
    m.ctc = CpuCTC({"ctc.ctc_lo.weight": torch.randn(37, 128), "ctc.ctc_lo.bias": torch.randn(37)})
    m.eval()
    before = {k: v.data_ptr() for k, v in m.state_dict().items()}
    params = {id(p) for p in m.parameters()}
    auto_avsr_b200.install_decoder(m)
    assert type(m.decoder).__module__ == "auto_avsr_b200.espnet_dropin.transformer_decoder"
    assert {k: v.data_ptr() for k, v in m.state_dict().items()} == before
    assert params == {id(p) for p in m.parameters()} and not m.decoder.training
    assert [[k, list(v.shape)] for k, v in m.decoder.state_dict().items()] == golden["parameters"]
    assert isinstance(m.decoder, scorer_interface.BatchScorerInterface)


@needs_emu
def test_bench_decode_child_dry_run_agrees_with_the_reference_decoder():
    """scripts/bench_decode.py (the child bench.py's extras start) on the CPU: full-size decoder (d 768, 6 layers, odim 5049),
    the drop-in scorers on the host replay under DeviceBeamSearch: the best hypothesis and score of the reference's own
    decoder + CTCPrefixScorer + BatchBeamSearch on the same inputs (tests/golden/reference_surfaces.json)."""
    import json
    with open(os.path.join(ROOT, "tests", "golden", "reference_surfaces.json")) as f:
        golden = json.load(f)["decode_dryrun_T6_beam4"]
    env = dict(os.environ, AVSR_BENCH_DECODE_DRYRUN="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "bench_decode.py"), "6", "4"], capture_output=True, text=True,
                       timeout=600, env=env, cwd=ROOT)
    rows = [ln for ln in r.stdout.splitlines() if ln.startswith("DECODE-JSON ")]
    assert r.returncode == 0 and rows, r.stdout[-1000:] + r.stderr[-2000:]
    out = json.loads(rows[-1][len("DECODE-JSON "):])
    dev = out["device_beam_search"]
    assert "error" not in dev, dev
    assert dev["best_yseq"] == golden["best_yseq"]
    assert abs(dev["best_score"] - golden["best_score"]) < 1e-3
    assert dev["steps"] == 6
    # where the reference copy was built (oracle/build_ref.py) the script also runs the reference's arms
    for arm, tol in (("reference_loop_dropins", 1e-4), ("reference_eager", 1e-3)):
        if arm in out:
            assert "error" not in out[arm], out[arm]
            assert out[arm]["best_yseq"] == golden["best_yseq"]
            assert abs(out[arm]["best_score"] - dev["best_score"]) < tol


@needs_emu
def test_shim_replays_test_step_through_the_beam_search():
    """lightning.py:69-76 (after the front-end) on an E2EShell whose encoder side is stubbed out (it needs the GPU; its own
    replay is tests/test_gpu_callers.py): proj_encoder -> encoder(x, None) -> beam search over model.scorers() -> token ids."""
    from auto_avsr_b200 import shim
    from auto_avsr_b200.beam_search import DeviceBeamSearch
    from emu import build
    c = load_decoder_case("decoder_tiny")
    cfg = c["cfg"]
    model = shim.E2EShell(odim=cfg["odim"], idim=cfg["d_model"], adim=cfg["d_model"], aheads=cfg["n_heads"], eunits=cfg["linear_units"],
                          elayers=1)
    assert set(model.scorers()) == {"decoder", "ctc"} and model.eos == cfg["odim"] - 1
    # the tiny fixture's decoder has 2 layers: swap the shell's 6-layer decoder for it, stub the encoder side
    model.decoder = _dropin_decoder(c, build.load())
    model.ctc = CpuCTC(c["head_sd"])
    model.proj_encoder = torch.nn.Identity()
    class _PassThrough(torch.nn.Module):
        def forward(self, x, masks):
            return x, masks
    model.encoder = _PassThrough()
    bs = shim.get_beam_search_decoder(model, beam_size=cfg["beam"])
    assert isinstance(bs, DeviceBeamSearch) and bs.weights == {"decoder": 0.9, "ctc": 0.1} and bs.pre_beam_size == 7
    ids = shim.test_step_decode(model, c["memory"], bs)
    z = c["z"]
    L = int(z["nbest_len_f32"][0])
    assert ids.tolist() == z["nbest_yseq_f32"][0, 1:L].tolist()            # best hypothesis of the reference, <sos> dropped


@needs_emu
@pytest.mark.parametrize("T,beam,odim,seed", [(1, 3, 11, 0), (2, 1, 9, 1), (5, 4, 8, 2), (9, 6, 23, 3), (14, 2, 37, 4), (7, 5, 6, 5)])
def test_device_beam_search_corner_shapes_against_the_oracle_loop(T, beam, odim, seed):
    """Corner shapes of the search (T = 1: the first step is also the last; beam 1; pre-beam >= vocabulary -> no pre-beam;
    vocabularies so small that hypotheses end early and the beam runs dry) against the oracle's restatement of
    BatchBeamSearch, on a random 1-layer decoder through the host replay."""
    from auto_avsr_b200 import TransformerDecoder
    from auto_avsr_b200.beam_search import DeviceBeamSearch
    from auto_avsr_b200.synthetic import decoder_state_dict, encoder_input, head_state_dict
    from emu import build
    from oracle import decoder_oracle as DO
    from oracle import head_oracle as HO
    d, H, ff = 64, 1, 64
    sd = decoder_state_dict(100 + seed, odim, d, H, ff, 1)
    hsd = head_state_dict(100 + seed, 64, d, odim)
    mem = encoder_input([T], d, 200 + seed)[0]
    dec = TransformerDecoder(odim, d, H, ff, 1)
    dec.load_state_dict(sd, strict=True)
    dec.eval()
    dec.precision, dec._lib = "fp32", build.load()
    got = [h.asdict() for h in DeviceBeamSearch(dec, CpuCTC(hsd), beam_size=beam, vocab_size=odim)(mem)]
    want = DO.beam_search(lambda ys: DO.decoder_logp(sd, ys, mem.double(), H), HO.ctc_log_softmax(mem.double(), hsd), odim, beam,
                          maxlen=T)
    assert len(got) == len(want) >= 1
    assert got[0]["yseq"] == want[0]["yseq"] and got[0]["yseq"][0] == got[0]["yseq"][-1] == odim - 1
    assert abs(got[0]["score"] - want[0]["score"]) < 2e-3
    # same multiset of ended hypotheses (order may swap between near-ties in fp32 vs fp64)
    key = lambda h: tuple(h["yseq"])            # noqa: E731
    assert sorted(map(key, got)) == sorted(map(key, want))
    by = {key(h): h for h in want}
    for h in got:
        assert abs(h["score"] - by[key(h)]["score"]) < 2e-3
        assert abs(h["scores"]["decoder"] - by[key(h)]["scores"]["decoder"]) < 2e-3
        assert abs(h["scores"]["ctc"] - by[key(h)]["scores"]["ctc"]) < 2e-3


@needs_emu
def test_decoder_refuses_states_of_a_replaced_utterance():
    """The session holds one utterance: hypotheses of an earlier utterance must not be scored against the new K/V."""
    from emu import build
    c = load_decoder_case("decoder_tiny")
    cfg = c["cfg"]
    dec = _dropin_decoder(c, build.load())
    sos = cfg["odim"] - 1
    xs = c["memory"].unsqueeze(0)
    _, st_a = dec.batch_score(torch.tensor([[sos]]), [None], xs)
    _, st_a2 = dec.batch_score(torch.tensor([[sos, 3]]), st_a, xs)                 # same utterance: fine
    assert st_a2[0][0] == st_a[0][0] and len(st_a2[0]) == 3
    _, st_b = dec.batch_score(torch.tensor([[sos]]), [None], xs[:, :7])            # a new utterance replaces the session
    assert st_b[0][0] == st_a[0][0] + 1
    with pytest.raises(ValueError, match="session was replaced"):
        dec.batch_score(torch.tensor([[sos, 3, 4]]), st_a2, xs)
    with pytest.raises(ValueError, match="same prefix length"):
        dec.batch_score(torch.tensor([[sos, 3, 4]]), st_b, xs[:, :7])
    dec.batch_score(torch.tensor([[sos, 5]]), st_b, xs[:, :7])
