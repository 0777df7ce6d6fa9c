"""Cost of deep rankings: engine.rank at K = 100, 1,000 and 4,096 on 4,096 queries x 16,384 synthetic videos (TVR frame
shape L = 128, D = 384, two branches, two-scale head, bf16 + exact rescoring of candidate_depth(K, 128) candidates,
certify=True), the three depths interleaved call by call.  Every call is bracketed by CUDA events, and so is every
C-ABI call inside it; calls made by the certificate's exact re-rank are reported apart ("fallback:").  Then a deep merge
of G = 8 lists of K = 4,096 for 16,384 queries, with and without a 6-word payload.  Prints the card name and power
limit beside the numbers, the queries that failed the certificate per depth, the C-ABI calls of each depth, and one
JSON line (also written to --out when given).

    python tools/deepk_probe.py [--reps 30] [--out results/deepk_probe.json]
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
from dkd_b200 import _lib, engine, ops  # noqa: E402

Nq, Nv, L, D, KC = 4096, 16384, 128, 384, 128
DEPTHS = (100, 1000, 4096)
MERGE_G, MERGE_M, MERGE_K = 8, 16384, 4096


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in out.split(",")]
    except Exception:   # noqa: BLE001 — the timings stand without it
        name, power = torch.cuda.get_device_name(0), "unknown"
    return name, power


def corpus(dev, seed):
    """Encoded-frame stand-in on the device (synth.encoded_corpus's recipe): ragged lengths L/2 .. L, a per-video
    shared component, zero padding."""
    g = torch.Generator(device=dev).manual_seed(seed)
    lengths = torch.randint(L // 2, L + 1, (Nv,), generator=g, device=dev)
    mask = (torch.arange(L, device=dev)[None, :] < lengths[:, None]).float()
    x = 1.5 * torch.randn(Nv, 1, D, generator=g, device=dev) + torch.randn(Nv, L, D, generator=g, device=dev)
    return (x * mask[:, :, None]).contiguous(), mask


def ev():
    e = torch.cuda.Event(enable_timing=True)
    e.record()
    return e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda")
    f0, mask = corpus(dev, 1)
    f1 = corpus(dev, 2)[0] * mask[:, :, None]
    g = torch.Generator(device=dev).manual_seed(3)
    params = [(0.05 * torch.randn(D, D, generator=g, device=dev), torch.zeros(D, device=dev),
               0.05 * torch.randn(D, D, generator=g, device=dev), torch.zeros(D, device=dev)) for _ in range(2)]
    pc = engine.prepare_corpus([f0, f1], mask, params, heads=("two_scale",), precisions=("exact", "bf16"))
    del f0, f1
    q = [torch.randn(Nq, D, generator=g, device=dev) for _ in range(2)]
    pq = engine.prepare_queries(q)

    # every C-ABI call bracketed by events; calls inside the certificate's re-rank are tagged
    real_call, real_fallback = _lib.call, engine._apply_fallback
    state = {"fallback": False, "calls": []}

    def call(name, *a):
        s = ev()
        real_call(name, *a)
        state["calls"].append((("fallback:" if state["fallback"] else "") + name, s, ev()))

    def fallback(*a, **kw):
        state["fallback"] = True
        try:
            return real_fallback(*a, **kw)
        finally:
            state["fallback"] = False

    _lib.call, engine._apply_fallback = call, fallback

    def rank(K):
        return engine.rank(pc, pq, K=K, head="two_scale", precision="bf16", Kc=KC, certify=True)

    for _ in range(args.warmup):
        for K in DEPTHS:
            rank(K)
    torch.cuda.synchronize()
    state["calls"].clear()
    times = {K: [] for K in DEPTHS}
    parts = {K: {} for K in DEPTHS}
    fails = {K: 0 for K in DEPTHS}
    sequence = {}
    out = {}
    for _ in range(args.reps):
        for K in DEPTHS:
            before = engine.STATS["certify_fallback_queries"]
            a = ev()
            out[K] = rank(K)
            b = ev()
            b.synchronize()
            times[K].append(a.elapsed_time(b))
            fails[K] += engine.STATS["certify_fallback_queries"] - before
            per = {}
            for name, s, e in state["calls"]:
                per[name] = per.get(name, 0.0) + s.elapsed_time(e)
            for name, v in per.items():
                parts[K].setdefault(name, []).append(v)
            sequence.setdefault(K, [name for name, _, _ in state["calls"] if not name.startswith("fallback:")])
            state["calls"].clear()
    _lib.call, engine._apply_fallback = real_call, real_fallback
    # the top-100 of every depth is the K = 100 ranking
    prefix_equal = all(torch.equal(out[K][1][:, :100], out[100][1]) and torch.equal(out[K][0][:, :100], out[100][0])
                       for K in DEPTHS)
    del pc, pq, out
    torch.cuda.empty_cache()

    # deep merge: G sorted lists of K per query, distinct ids across the lists
    gm = torch.Generator(device=dev).manual_seed(5)
    ms = torch.sort(torch.rand(MERGE_G, MERGE_M, MERGE_K, generator=gm, device=dev), dim=-1, descending=True).values
    mi = (torch.arange(MERGE_G, device=dev, dtype=torch.int32)[:, None, None] * MERGE_K
          + torch.arange(MERGE_K, device=dev, dtype=torch.int32)).expand(MERGE_G, MERGE_M, MERGE_K).contiguous()
    mw = torch.randint(0, 1 << 30, (MERGE_G, MERGE_M, MERGE_K, 6), generator=gm, device=dev, dtype=torch.int32)
    pad = torch.full((6,), -1, dtype=torch.int32, device=dev)
    merge_t = {"plain": [], "payload6": []}
    for i in range(args.warmup + 10):
        a = ev()
        ops.merge_topk_deep(ms, mi)
        b = ev()
        ops.merge_topk_deep(ms, mi, payload=mw, pad=pad)
        c = ev()
        c.synchronize()
        if i >= args.warmup:
            merge_t["plain"].append(a.elapsed_time(b))
            merge_t["payload6"].append(b.elapsed_time(c))

    name, power = card()
    res = dict(probe="deepk_probe", card=name, power_limit=power,
               shape=dict(Nq=Nq, Nv=Nv, L=L, D=D, branches=2, head="two_scale", precision="bf16", Kc_arg=KC),
               reps=args.reps,
               candidates={K: engine.candidate_depth(K, KC) for K in DEPTHS},
               rank_ms_median={K: statistics.median(v) for K, v in times.items()},
               rank_ms_min={K: min(v) for K, v in times.items()},
               parts_ms_median={K: {n: statistics.median(v) for n, v in p.items()} for K, p in parts.items()},
               parts_calls_with={K: {n: len(v) for n, v in p.items()} for K, p in parts.items()},
               certify_fallback_queries=fails, certify_checked_queries=Nq * args.reps,
               c_abi_sequence=sequence, top100_prefix_equal=prefix_equal,
               merge=dict(G=MERGE_G, M=MERGE_M, K=MERGE_K,
                          ms_median={k: statistics.median(v) for k, v in merge_t.items()},
                          ms_min={k: min(v) for k, v in merge_t.items()}))
    print(f"{name}, power limit {power}; {Nq} queries x {Nv} videos, two branches, two-scale, bf16")
    for K in DEPTHS:
        print(f"K = {K} (Kc = {res['candidates'][K]}): median {res['rank_ms_median'][K]:.3f} ms, "
              f"min {res['rank_ms_min'][K]:.3f} ms, certificate failures {fails[K]} of {Nq * args.reps}")
        for n, v in sorted(res["parts_ms_median"][K].items(), key=lambda kv: -kv[1]):
            print(f"    {n}: median {v:.3f} ms per call (in {res['parts_calls_with'][K][n]} of {args.reps} calls)")
    print(f"merge G = {MERGE_G}, K = {MERGE_K}, {MERGE_M} queries: plain {res['merge']['ms_median']['plain']:.3f} ms, "
          f"6-word payload {res['merge']['ms_median']['payload6']:.3f} ms (median)")
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(dict(res, times_ms=times), f, indent=1)


if __name__ == "__main__":
    main()
