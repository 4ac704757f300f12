#!/usr/bin/env python3
"""Golden module surfaces of the reference (tests/golden/reference_surfaces.json): what the install tests and the
decode-bench dry run compare against, so that they run without the reference tree.

TEST INFRASTRUCTURE ONLY.  Run where the reference tree is importable (after oracle/build_ref.py has made oracle/_ref):
    PYTHONPATH=<reference tree> python oracle/make_golden_surfaces.py

Stores
  e2e_audio    state-dict keys and shapes of E2E(5049, "audio") (e2e_asr_conformer.py) and its parameter count
  ctc          state-dict keys / shapes and the attributes install_head reads of CTC(5049, 768, 0.1, reduce=True)
  decoder      parameter names / shapes and the attributes install_decoder reads of
               TransformerDecoder(odim=37, attention_dim=128, attention_heads=2, linear_units=256, num_blocks=2)
  decode_dryrun_T6_beam4   best hypothesis and score of the reference's own decoder + CTCPrefixScorer + BatchBeamSearch
               in scripts/bench_decode.py's CPU dry run (T = 6, beam 4, fp32)
"""
import json
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
OUT = os.path.join(ROOT, "tests", "golden", "reference_surfaces.json")


def shapes(named):
    return [[k, list(v.shape)] for k, v in named]


def main():
    from espnet.nets.pytorch_backend.ctc import CTC
    from espnet.nets.pytorch_backend.decoder.transformer_decoder import TransformerDecoder
    from espnet.nets.pytorch_backend.e2e_asr_conformer import E2E

    m = E2E(5049, "audio")
    e2e = {"state": shapes(m.state_dict().items()), "n_parameters": sum(p.numel() for p in m.parameters())}
    ctc = CTC(5049, 768, 0.1, reduce=True)
    ctc_s = {"state": shapes(ctc.state_dict().items()), "dropout_rate": ctc.dropout_rate, "reduce": ctc.reduce}
    d = TransformerDecoder(odim=37, attention_dim=128, attention_heads=2, linear_units=256, num_blocks=2)
    dec = {"parameters": shapes(d.named_parameters()), "attention_heads": d.decoders[0].self_attn.h}

    # the child imports the reference from oracle/_ref: with the reference tree on PYTHONPATH too, two espnets would meet
    env = {k: v for k, v in os.environ.items() if k != "PYTHONPATH"}
    env["AVSR_BENCH_DECODE_DRYRUN"] = "1"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "bench_decode.py"), "6", "4"], capture_output=True,
                       text=True, env=env, cwd=ROOT, check=True)
    run = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("DECODE-JSON ")][-1][len("DECODE-JSON "):])
    eager = run["reference_eager"]
    decode = {"best_yseq": eager["best_yseq"], "best_score": eager["best_score"]}

    with open(OUT, "w") as f:
        json.dump({"e2e_audio": e2e, "ctc": ctc_s, "decoder": dec, "decode_dryrun_T6_beam4": decode}, f, indent=0)
        f.write("\n")
    print("wrote", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
