"""Cost of a video filter: engine.rank at TVR shape (10,895 queries x 2,179 videos, L = 128, D = 384, two branches,
two-scale head, bf16 + exact rescoring of 128 candidates, top-100) without a filter and with three per-query filters
(all ones; 50 % of the videos at random; a 100-id deny list), the four interleaved call by call in one process, each
call bracketed by CUDA events.  Also times dkd_build_video_filter for the deny lists, and the candidate selection
kernel alone (dkd_select_topk vs dkd_select_topk_filtered on the same fused matrix), where the filter is read.
Prints the card name and power limit beside the numbers and one JSON line (also written to --out when given).

    python tools/filter_probe.py [--reps 30] [--out results/filter_probe.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as ge  # noqa: E402

ge.load_package()
from dkd_b200 import engine, ops  # noqa: E402
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


def timed(fn, reps):
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b))
    return out


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

    rng = np.random.default_rng(6)
    deny = [rng.integers(0, Nv, 100) for _ in range(Nq)]
    W = (Nv + 31) // 32
    filters = {
        "none": None,
        "all_ones": engine.make_video_filter(Nv, deny=[]).expand(Nq, W).contiguous(),
        "half_random": torch.randint(-2 ** 31, 2 ** 31, (Nq, W), dtype=torch.int32, device=dev,
                                     generator=torch.Generator(device=dev).manual_seed(7)),
        "deny_100": engine.make_video_filter(Nv, deny=deny),
    }

    def call(vf):
        return engine.rank(pc, pq, K=K, head="two_scale", precision="bf16", Kc=KC, certify="deferred",
                           video_filter=vf)

    for _ in range(args.warmup):
        for vf in filters.values():
            call(vf)
    engine.finish()
    torch.cuda.synchronize()
    engine.STATS["certify_fallback_queries"] = 0
    times = {k: [] for k in filters}
    names = list(filters)
    same_all_ones = True
    for r in range(args.reps):
        order = names if r % 2 == 0 else names[::-1]
        outs = {}
        for name in order:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            outs[name] = call(filters[name])
            b.record()
            b.synchronize()
            engine.finish()
            times[name].append(a.elapsed_time(b))
        same_all_ones = same_all_ones and torch.equal(outs["none"][0], outs["all_ones"][0]) and \
            torch.equal(outs["none"][1], outs["all_ones"][1])

    # the builder alone (CSR already on the device), and the selection kernel alone on the fused matrix
    ptr = torch.from_numpy(np.arange(0, 100 * Nq + 1, 100, dtype=np.int32)).to(dev)
    ids = torch.from_numpy(np.concatenate(deny).astype(np.int32)).to(dev)
    build_ms = timed(lambda: ops.build_video_filter(ptr, ids, Nv, deny=True), args.reps)
    assert torch.equal(ops.build_video_filter(ptr, ids, Nv, deny=True), filters["deny_100"])
    fused, _ = engine.score_two_scale_head(pc, pq, "bf16")
    sel = {"select_topk": timed(lambda: ops.select_topk(fused, KC), args.reps)}
    for name in names[1:]:
        sel[f"select_topk_filtered_{name}"] = timed(lambda: ops.select_topk_filtered(fused, KC, filters[name]),
                                                    args.reps)

    name, power = card()
    med = {k: statistics.median(v) for k, v in times.items()}
    res = dict(probe="filter_probe", card=name, power_limit=power, shape=dict(Nq=Nq, Nv=Nv, L=L, D=D, K=K, Kc=KC),
               reps=args.reps, rank_ms_median=med, rank_ms_min={k: min(v) for k, v in times.items()},
               extra_pct_median={k: 100.0 * (med[k] / med["none"] - 1.0) for k in names[1:]},
               build_deny_100_ms_median=statistics.median(build_ms), build_deny_100_ms_min=min(build_ms),
               select_ms_median={k: statistics.median(v) for k, v in sel.items()},
               select_ms_min={k: min(v) for k, v in sel.items()},
               all_ones_identical=bool(same_all_ones),
               certify_fallback_queries=engine.STATS["certify_fallback_queries"])
    print(f"{name}, power limit {power}: rank medians (ms, {args.reps} interleaved calls each): "
          + ", ".join(f"{k} {v:.3f}" for k, v in med.items()))
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(dict(res, times_ms=times, build_ms=build_ms, select_ms=sel), f, indent=1)


if __name__ == "__main__":
    main()
