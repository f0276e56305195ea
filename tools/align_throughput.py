"""Diagnostic (not the bench contract): what option "align" costs.

Runs bench.py's c3 and c2 models on a synthetic sequence with records staying in HBM, alternating three arms: MAF
(align 0), SAM alignment lines (align 1) and BAM alignment records (align 1, align_bam 1), and once more each with
"deflate" on host delivery.  Reports per run the generated Gbp/s,
the pass-2 seconds (the ABI's emit_seconds, which include k_aln_*), and the bytes per base of the second stream, with
the card's name, power limit and clocks.  Prints one JSON line.  GLEN_MBP (default 500) sets the sequence length."""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def _card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], stdout=subprocess.PIPE,
                         text=True).stdout.strip().split("\n")[0]
    return dict(zip(q.split(","), [x.strip() for x in out.split(",")]))


ARMS = (("maf", 0, 0), ("sam", 1, 0), ("align_bam", 1, 1))


def _run(eng, glen, depth, seq, arm, deflate):
    from pbsim_b200 import capi
    name, align, align_bam = arm
    eng.set_option("align", align)
    eng.set_option("align_bam", align_bam)
    eng.set_option("deflate", deflate)
    eng.set_synthetic_sequence(glen, seq, 20240601 + seq)
    if align:
        eng.set_sequence_name("chr%d" % seq)
    eng.timer_start()
    eng.begin(int(depth * glen), rng_mode=capi.RNG_PHILOX, seed=1)
    bases = second = text = 0
    while True:
        c = eng.next_chunk(device=not deflate)
        if c is None:
            break
        bases += c.bases
        second += c.maf_bytes
        text += c.maf_text_bytes
    st = eng.end()
    ms = eng.timer_stop()
    return dict(arm=name, deflate=deflate, bases=bases, seconds=ms / 1e3, gbps=bases / ms / 1e6,
                pass2_seconds=st.emit_seconds, second_stream_bytes_per_base=(text if deflate else second) / bases,
                compressed_bytes_per_base=second / bases if deflate else None)


def main():
    import torch
    from bench import WORKLOADS
    from pbsim_b200 import capi, simulator
    from tests.golden_util import model_path
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: the engine has no CPU fallback")
    glen = int(os.environ.get("GLEN_MBP", "500")) * 1000000
    L = capi.load()
    out = dict(diagnostic="option align: MAF vs SAM lines vs BAM records, synthetic sequence of %d bp" % glen, card=_card(),
               runs=[])
    for key in ("c3", "c2"):
        w = WORKLOADS[key]
        eng = simulator.Engine(0)
        try:
            eng.set_model(capi.HostModel(L, capi.host_params(w["method"], **w["params"]), model_path(w["model"])))
            eng.set_option("pipeline", 1)
            for arm in ARMS:  # warm-up: modules, buffers
                _run(eng, glen, w["depth"], 1, arm, 0)
            for rep in range(2):
                for arm in ARMS:
                    r = _run(eng, glen, w["depth"], 2 + rep, arm, 0)
                    r["workload"] = key
                    out["runs"].append(r)
            for arm in ARMS:
                r = _run(eng, glen, w["depth"], 5, arm, 1)
                r["workload"] = key
                out["runs"].append(r)
        finally:
            eng.close()
    out["card_after"] = _card()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
