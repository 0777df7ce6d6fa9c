"""Cost of the per-hit detail: engine.rank at TVR shape (10,895 queries x 2,179 videos, L = 128, D = 384, two
branches, two-scale head, bf16 + exact rescoring of 128 candidates, top-100) with and without return_detail, the two
interleaved call by call in one process, each call bracketed by CUDA events.  Prints the card name and power limit
beside the numbers and one JSON line (also written to --out when given).

    python tools/detail_probe.py [--reps 30] [--out results/detail_probe.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as ge  # noqa: E402

ge.load_package()
from dkd_b200 import engine  # noqa: E402
from tests import synth  # noqa: E402

Nq, Nv, L, D, K, KC = 10895, 2179, 128, 384, 100, 128


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in out.split(",")]
    except Exception:   # noqa: BLE001 — the timings stand without it
        name, power = torch.cuda.get_device_name(0), "unknown"
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda")
    frames, mask, _ = synth.encoded_corpus(Nv, L, D, seed=1, shared=1.5)
    frames2 = synth.encoded_corpus(Nv, L, D, seed=2, shared=1.5)[0] * mask[:, :, None]
    g = torch.Generator().manual_seed(3)
    params = [tuple(t.to(dev) for t in (0.05 * torch.randn(D, D, generator=g), torch.zeros(D),
                                        0.05 * torch.randn(D, D, generator=g), torch.zeros(D))) for _ in range(2)]
    pc = engine.prepare_corpus([frames.to(dev), frames2.to(dev)], mask.to(dev), params, heads=("two_scale",),
                               precisions=("exact", "bf16"))
    pq = engine.prepare_queries([synth.encoded_queries(Nq, D, seed=4).to(dev), synth.encoded_queries(Nq, D, seed=5).to(dev)])
    del frames, frames2

    def call(detail):
        return engine.rank(pc, pq, K=K, head="two_scale", precision="bf16", Kc=KC, certify="deferred",
                           return_detail=detail)

    for _ in range(args.warmup):
        call(False)
        call(True)
    engine.finish()
    torch.cuda.synchronize()
    times = {False: [], True: []}
    same = True
    for r in range(args.reps):
        for detail in ((False, True) if r % 2 == 0 else (True, False)):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            out = call(detail)
            b.record()
            b.synchronize()
            engine.finish()
            times[detail].append(a.elapsed_time(b))
            if detail:
                s1, i1 = out[0], out[1]
            else:
                s0, i0 = out
        same = same and torch.equal(s0, s1) and torch.equal(i0, i1)
    name, power = card()
    med = {k: statistics.median(v) for k, v in times.items()}
    res = dict(probe="detail_probe", card=name, power_limit=power, shape=dict(Nq=Nq, Nv=Nv, L=L, D=D, K=K, Kc=KC),
               reps=args.reps, rank_ms_median=med[False], rank_detail_ms_median=med[True],
               rank_ms_min=min(times[False]), rank_detail_ms_min=min(times[True]),
               extra_ms_median=med[True] - med[False], extra_pct_median=100.0 * (med[True] / med[False] - 1.0),
               identical_scores_ids=bool(same), certify_fallback_queries=engine.STATS["certify_fallback_queries"])
    print(f"{name}, power limit {power}: rank {med[False]:.3f} ms, rank + detail {med[True]:.3f} ms "
          f"(median of {args.reps} interleaved calls each; +{res['extra_pct_median']:.2f} %)")
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(dict(res, times_ms={"rank": times[False], "rank_detail": times[True]}), f, indent=1)


if __name__ == "__main__":
    main()
