"""Cost of moment localization: engine.rank at TVR shape (10,895 queries x 2,179 videos, L = 128, D = 384, two
branches, two-scale head, bf16 + exact rescoring of 128 candidates, top-100), then engine.localize of the returned ids
(m = 5, iou = 0.5).  rank and localize calls are interleaved in one process; every call is bracketed by CUDA events,
and inside localize so is every C-ABI call (the CSR build, one dots pass per branch, the NMS).  Prints the card name
and power limit beside the numbers, E and the bytes of the dots, a checksum of the moments, and one JSON line (also
written to --out when given).

    python tools/moment_probe.py [--reps 30] [--out results/moment_probe.json]
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
from dkd_b200 import _lib, engine  # noqa: E402
from tests import synth  # noqa: E402

Nq, Nv, L, D, K, KC, MOMENTS, IOU = 10895, 2179, 128, 384, 100, 128, 5, 0.5


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

    # per-entry-point events inside localize only (rank's own calls are not bracketed)
    real_call = _lib.call
    inner = {"on": False, "calls": []}

    def call(name, *a):
        if not inner["on"]:
            return real_call(name, *a)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        real_call(name, *a)
        e.record()
        inner["calls"].append((name, s, e))

    _lib.call = call

    def rank():
        return engine.rank(pc, pq, K=K, head="two_scale", precision="bf16", Kc=KC, certify="deferred")

    def localize(ids):
        inner["on"] = True
        try:
            return engine.localize(pc, pq, ids, m=MOMENTS, iou=IOU)
        finally:
            inner["on"] = False

    for _ in range(args.warmup):
        _, ids = rank()
        localize(ids)
    engine.finish()
    torch.cuda.synchronize()
    inner["calls"].clear()
    times = {"rank": [], "localize": []}
    parts = {}
    mo = ids = None
    for _ in range(args.reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        _, ids = rank()
        b.record()
        b.synchronize()
        engine.finish()
        times["rank"].append(a.elapsed_time(b))
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        mo = localize(ids)
        b.record()
        b.synchronize()
        times["localize"].append(a.elapsed_time(b))
        seen = {}
        for name, s, e in inner["calls"]:
            i = seen.get(name, 0)
            seen[name] = i + 1
            parts.setdefault(f"{name}[{i}]" if name == "dkd_clip_dots_list" else name, []).append(s.elapsed_time(e))
        inner["calls"].clear()
    name, power = card()
    E = int((ids >= 0).sum())
    live = mo.arg >= 0
    med = {k: statistics.median(v) for k, v in times.items()}
    res = dict(probe="moment_probe", card=name, power_limit=power,
               shape=dict(Nq=Nq, Nv=Nv, L=L, D=D, K=K, Kc=KC, m=MOMENTS, iou=IOU, branches=2), reps=args.reps,
               rank_ms_median=med["rank"], rank_ms_min=min(times["rank"]),
               localize_ms_median=med["localize"], localize_ms_min=min(times["localize"]),
               localize_over_rank=med["localize"] / med["rank"],
               parts_ms_median={k: statistics.median(v) for k, v in parts.items()},
               parts_ms_min={k: min(v) for k, v in parts.items()},
               entries_per_branch=E, dots_bytes_per_branch=E * 32 * 4,
               moments_per_hit_mean=float(live.sum()) / max(E, 1),
               checksum_arg=int(mo.arg.long().sum()), checksum_score=float(mo.score[live].double().sum()),
               certify_fallback_queries=engine.STATS["certify_fallback_queries"])
    print(f"{name}, power limit {power}: rank {med['rank']:.3f} ms, localize {med['localize']:.3f} ms "
          f"(median of {args.reps} interleaved calls each); E = {E} per branch, {E * 128 / 1e6:.1f} MB of dots per branch")
    for k, v in res["parts_ms_median"].items():
        print(f"  {k}: median {v:.3f} ms, min {res['parts_ms_min'][k]:.3f} ms")
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(dict(res, times_ms=times, parts_ms=parts), f, indent=1)


if __name__ == "__main__":
    main()
