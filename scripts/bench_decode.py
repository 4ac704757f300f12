#!/usr/bin/env python3
"""bench.py extras, BASELINE.json configs[4] flavour (SURVEY.md 8f #3): one utterance's encoder output -> beam-search
decoding (attention decoder + CTC prefix scorer, beam 40, ctc_weight 0.1 as lightning.py:126-157 builds it), timed three
ways on the same GPU with the same synthetic weights:

  device_beam_search      auto_avsr_b200.beam_search.DeviceBeamSearch over the drop-in scorers (libavsr_b200)
  reference_loop_dropins  the UNMODIFIED reference BatchBeamSearch (oracle/_ref) driving the drop-in scorers
  reference_eager         the UNMODIFIED reference decoder + CTCPrefixScorer + BatchBeamSearch moved to cuda (stock
                          eager PyTorch): the baseline leg

Runs as a CHILD of bench.py (own CUDA context, own timeout) and prints one JSON object; wall-clock per utterance with
a synchronize on both sides (the search is host-driven: its host time is part of what is being measured)."""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    T = int(sys.argv[1]) if len(sys.argv) > 1 else 100
    beam = int(sys.argv[2]) if len(sys.argv) > 2 else 40
    out = {"what": f"beam-search decoding of ONE utterance: encoder output ({T}, 768) -> n-best; 6-layer d=768 attention decoder + "
                   f"CTC prefix scorer (pre-beam {int(1.5 * beam)}), beam {beam}, odim 5049, synthetic weights (the search runs to "
                   "its length limit: T steps)", "T": T, "beam": beam}
    ref = None
    try:
        from oracle import build_ref
        ref = build_ref.import_reference_search()            # before the drop-ins: they then derive from ITS interfaces
    except Exception as e:                                   # noqa: BLE001
        out["reference_unavailable"] = f"{type(e).__name__}: {e}"
    import torch
    from auto_avsr_b200 import CTC, CTCPrefixScorer, TransformerDecoder
    from auto_avsr_b200.beam_search import DeviceBeamSearch
    from auto_avsr_b200.espnet_dropin import scorer_interface
    from auto_avsr_b200.synthetic import decoder_state_dict, encoder_input, head_state_dict

    # AVSR_BENCH_DECODE_DRYRUN=1: CPU dry run of THIS SCRIPT's plumbing on the tests' host replay (no measurement value)
    dry = os.environ.get("AVSR_BENCH_DECODE_DRYRUN") == "1"
    dev = torch.device("cpu" if dry else "cuda:0")
    lib = None
    if dry:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from emu import build as emu_build
        lib = emu_build.load()
    sync = (lambda: None) if dry else torch.cuda.synchronize
    dsd, hsd = decoder_state_dict(4), head_state_dict(4)
    ctc_sd = {"ctc_lo.weight": hsd["ctc.ctc_lo.weight"], "ctc_lo.bias": hsd["ctc.ctc_lo.bias"]}
    x = encoder_input([T], 768, 9)[0].to(dev)
    odim, eos = 5049, 5048

    def timed(fn, reps):
        fn()                                                  # warm-up (weight preparation, allocations)
        sync()
        t0 = time.perf_counter()
        for _ in range(reps):
            res = fn()
        sync()
        return (time.perf_counter() - t0) / reps, res

    dec = TransformerDecoder(odim=odim, attention_dim=768, attention_heads=12, linear_units=3072, num_blocks=6)
    dec.load_state_dict(dsd, strict=True)
    ctc = CTC(odim, 768, 0.1)
    ctc.load_state_dict(ctc_sd)
    dec, ctc = dec.to(dev).eval(), ctc.to(dev).eval()
    if dry:
        class _CpuCTC(torch.nn.Module):                       # the drop-in CTC refuses CPU tensors
            def __init__(self, lo):
                super().__init__()
                self.ctc_lo = lo

            @torch.no_grad()
            def log_softmax(self, hs):
                return torch.log_softmax(self.ctc_lo(hs), dim=-1)
        ctc = _CpuCTC(ctc.ctc_lo)
        dec._lib, dec.precision = lib, "fp32"
    best = {}
    try:
        bs = DeviceBeamSearch(dec, ctc, beam_size=beam)
        s0 = bs.stats["steps"]
        dt, nb = timed(lambda: bs(x), 3)
        steps = (bs.stats["steps"] - s0) // 4
        best["device"] = (nb[0].yseq.tolist(), float(nb[0].score))
        out["device_beam_search"] = {"ms_per_utterance": dt * 1e3, "steps": steps, "ms_per_step": dt * 1e3 / max(steps, 1),
                                     "utterances_per_s": 1.0 / dt, "nbest": len(nb), "best_score": float(nb[0].score),
                                     "best_yseq": best["device"][0], "precision": dec.precision or "f16",
                                     "api": "auto_avsr_b200.beam_search.DeviceBeamSearch -> avsr_decoder_step / avsr_ctc_prefix_*"}
    except Exception as e:                                   # noqa: BLE001
        out["device_beam_search"] = {"error": f"{type(e).__name__}: {e}"}
    if ref is not None:
        token_list = [str(i) for i in range(odim)]
        weights = dict(decoder=0.9, ctc=0.1, lm=0.0, length_bonus=0)

        def build(decoder, scorer):
            scorers = dict(decoder=decoder, ctc=scorer, lm=None, length_bonus=ref["LengthBonus"](len(token_list)))
            return ref["BatchBeamSearch"](beam_size=beam, vocab_size=len(token_list), weights=weights, scorers=scorers,
                                          sos=eos, eos=eos, token_list=token_list, pre_beam_score_key="decoder")
        try:
            scorer_interface.rebind()
            scorer = CTCPrefixScorer(ctc, eos)
            scorer._lib = lib
            bs2 = build(dec, scorer)
            with torch.no_grad():
                dt, nb = timed(lambda: bs2(x), 2)
            best["ref_loop"] = (nb[0].yseq.tolist(), float(nb[0].score))
            out["reference_loop_dropins"] = {"ms_per_utterance": dt * 1e3, "utterances_per_s": 1.0 / dt, "nbest": len(nb),
                                             "best_score": float(nb[0].score), "best_yseq": best["ref_loop"][0],
                                             "api": "espnet BatchBeamSearch (unmodified) over the drop-in scorers"}
        except Exception as e:                               # noqa: BLE001
            out["reference_loop_dropins"] = {"error": f"{type(e).__name__}: {e}"}
        try:
            rdec = ref["TransformerDecoder"](odim=odim, attention_dim=768, attention_heads=12, linear_units=3072, num_blocks=6)
            rdec.load_state_dict(dsd, strict=True)
            rctc = ref["CTC"](odim, 768, 0.1, reduce=True)
            rctc.load_state_dict(ctc_sd)
            rdec, rctc = rdec.to(dev).eval(), rctc.to(dev).eval()
            bs3 = build(rdec, ref["CTCPrefixScorer"](rctc, eos))
            with torch.no_grad():
                dt, nb = timed(lambda: bs3(x), 1)
            best["ref_eager"] = (nb[0].yseq.tolist(), float(nb[0].score))
            out["reference_eager"] = {"ms_per_utterance": dt * 1e3, "utterances_per_s": 1.0 / dt, "nbest": len(nb),
                                      "best_score": float(nb[0].score), "best_yseq": best["ref_eager"][0],
                                      "api": "the reference's own decoder + CTCPrefixScorer + BatchBeamSearch .to('cuda'), fp32 eager"}
        except Exception as e:                               # noqa: BLE001
            out["reference_eager"] = {"error": f"{type(e).__name__}: {e}"}
    if "device" in best and "ref_eager" in best:
        out["same_best_hypothesis_as_reference_eager"] = best["device"][0] == best["ref_eager"][0]
        out["best_score_gap_vs_reference_eager"] = abs(best["device"][1] - best["ref_eager"][1])
    print("DECODE-JSON " + json.dumps(out))


if __name__ == "__main__":
    main()
