#!/usr/bin/env python
"""bench.py — query-video pairs scored+ranked per second on the TVR-shaped synthetic eval.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload tvr_two_scale]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over the whole query set: encoded query vectors (resident in
HBM) -> L2-normalise/bf16 cast -> tcgen05 scoring GEMM with fused max/argmax (both branches) ->
frame-scale gather + fusion -> warp top-128 -> exact fp32 rescoring -> per-query top-100
[-> NCCL all-gather + merge for N > 1].  The corpus is prepared once (untimed, reported as
`prep_ms`).  Prints ONE JSON line on rank 0.

Workloads (BASELINE.json configs[1]): TVR shape, 2,179 videos x 128 frames x 3072-d, 10,895 queries
x <=30 words x 768-d, random-init DL-DKD++ (hidden 384, two branches), synthetic features.
  tvr_two_scale  north_star head (clip proposals + key-clip frame attention)        [default, headline]
  tvr_frame      the head the reference ships (max over frames), same kernels
N > 1: weak scaling — every rank owns its own 2,179-video shard of an N x 2,179-video corpus,
queries replicated, local top-100 merged through one NCCL all-gather.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TVR = dict(Nv=2179, L=128, Dv=3072, Nq=10895, Lq=30, Dq=768, H=384, T=32)
K_TOP = 100
K_CAND = 128


_T0 = time.perf_counter()


def log(msg):
    """Progress on stderr (stdout carries the one JSON line): which leg every rank is in, with a wall-clock stamp."""
    print(f"[bench rank {os.environ.get('RANK', '0')} +{time.perf_counter() - _T0:6.1f}s] {msg}", file=sys.stderr, flush=True)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(bf16_burst=d.get("bf16_tflops", 1590.0), bf16_sustained=d.get("bf16_tflops_sustained", 1400.0),
                    hbm=d.get("hbm_gbs", 6650.0), source="measured")
    return dict(bf16_burst=1590.0, bf16_sustained=1400.0, hbm=6650.0, source="fallback")


DUMP_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """--dump-outputs: every named array as <path>/<name>.npy, floating point as float32, integers as float64 (exact),
    so that two builds can be compared output for output.  Above DUMP_BYTES in all, every array of rank >= 1 keeps the
    same fraction of its rows, a fixed, seeded sample (arrays with as many rows keep the same rows), listed in
    <name>_rows.npy; scalars are kept."""
    out = {}
    for name, t in arrays.items():
        t = t.detach().cpu()
        out[name] = (t.float() if t.is_floating_point() else t.double()).numpy()
    if sum(a.nbytes for a in out.values()) > DUMP_BYTES:
        big = [name for name, a in out.items() if a.ndim >= 1]
        room = DUMP_BYTES - sum(a.nbytes for name, a in out.items() if name not in big)
        frac = room / sum(out[name].nbytes + 8 * len(out[name]) for name in big)   # the row lists count too
        for name in big:
            n = len(out[name])
            rows = np.sort(np.random.default_rng(0).choice(n, int(n * frac), replace=False))
            out[name] = out[name][rows]
            out[name + "_rows"] = rows.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons, self.max_mhz = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.02)

    def result(self):
        self.stop_flag = True
        self.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml_unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------
def model_config(shape):
    from dkd_b200.config import model_config as mc, options
    cfg = mc(shape["Dv"], shape["Dq"], hidden=shape["H"], n_heads=4, max_ctx_l=shape["L"], max_desc_l=shape["Lq"])
    return cfg, options()


def synth_encoded(shape, device, shard_seed, dkd_model_cls, want_queries=True):
    """Synthetic raw features of the named shapes -> random-init DL-DKD++ encoders (PyTorch) -> encoded
    frames per branch + mask, encoded query vectors per branch.  Setup only (untimed)."""
    cfg, opt = model_config(shape)
    torch.manual_seed(0)
    model = dkd_model_cls(cfg, opt).to(device).eval()
    Nv, L, Dv, Nq, Lq, Dq = (shape[k] for k in ("Nv", "L", "Dv", "Nq", "Lq", "Dq"))
    g = torch.Generator(device=device).manual_seed(1000 + shard_seed)
    inher, explore = [], []
    mask = torch.ones(Nv, L, device=device)  # "x 128 frames" headline: every video has all 128 frames
    with torch.no_grad():
        for lo in range(0, Nv, 200):  # eval_context_bsz = 200 (method/config.py:48)
            n = min(200, Nv - lo)
            x = torch.randn(n, L, Dv, device=device, generator=g)
            x = x / (x.norm(dim=-1, keepdim=True) + 1e-5)          # l2_normalize_np_array, data_provider.py:71
            a, b = model.encode_context(x, mask[lo: lo + n])
            inher.append(a)
            explore.append(b)
        if not want_queries:
            return model, [torch.cat(inher), torch.cat(explore)], mask, None
        gq = torch.Generator(device=device).manual_seed(5_000_000)  # queries identical on every rank
        qlen = torch.randint(5, Lq + 1, (Nq,), device=device, generator=gq)
        qi, qe = [], []
        for lo in range(0, Nq, 500):
            n = min(500, Nq - lo)
            x = torch.randn(n, Lq, Dq, device=device, generator=gq)
            x = x / (x.norm(dim=-1, keepdim=True) + 1e-5)
            qm = (torch.arange(Lq, device=device)[None] < qlen[lo: lo + n, None]).float()
            x = x * qm[:, :, None]
            a, b = model.encode_query(x, qm)
            qi.append(a)
            qe.append(b)
    return model, [torch.cat(inher), torch.cat(explore)], mask, [torch.cat(qi), torch.cat(qe)]


def synth_c4(shape, device, shard_seed, nq=None):
    """BASELINE.json configs[3] (SURVEY §8d C4): clip features generated directly at D = H on the device, N(0,1),
    seed = shard id; queries N(0,1) identical on every rank; key/value projections N(0, 0.02) like
    reset_parameters (method/model.py:80-93).  The 32 downsampled frames ARE the frames (L = T = 32)."""
    Nv, L, H = shape["Nv"], shape["L"], shape["H"]
    nq = shape["Nq"] if nq is None else nq
    g = torch.Generator(device=device).manual_seed(1000 + shard_seed)
    frames = [torch.empty(Nv, L, H, device=device).normal_(generator=g) for _ in range(2)]
    mask = torch.ones(Nv, L, device=device)
    gq = torch.Generator(device=device).manual_seed(5_000_000)
    qs = [torch.empty(nq, H, device=device).normal_(generator=gq) for _ in range(2)]
    gp = torch.Generator(device=device).manual_seed(7)
    params = [(torch.empty(H, H, device=device).normal_(0.0, 0.02, generator=gp), torch.zeros(H, device=device),
               torch.empty(H, H, device=device).normal_(0.0, 0.02, generator=gp), torch.zeros(H, device=device))
              for _ in range(2)]
    return frames, mask, qs, params


# ------------------------------------------------------------------------------------------------
class CpuBaseline:
    """The oracle port of the reference's CPU eval loop on a bounded sample of the same workload:
    `sample_queries` queries x the full corpus, all host threads.  Setup (corpus-side preparation) happens once in
    the constructor and is not timed.  `tensors` = (frames_by_branch, mask, queries_by_branch, attn_params) on the
    host: the SAME encoded tensors the GPU arm scores (so the two results can be compared, `vs_oracle`); without
    it (the --impl reference arm, which must not touch the GPU) the same synthetic workload is generated on the CPU."""

    def __init__(self, shape, workload, max_queries, threads=None, tensors=None):
        from oracle import oracle as O
        self.O, self.shape, self.workload = O, shape, workload
        self.threads = threads or os.cpu_count()
        torch.set_num_threads(self.threads)
        if tensors is not None:
            self.frames, self.mask, self.qs, params = tensors
        else:
            from dkd_b200.model import DLDKD
            sub = dict(shape)
            sub["Nq"] = max_queries
            if workload == "c4_stream":
                self.frames, self.mask, self.qs, params = synth_c4(sub, torch.device("cpu"), 0)
            else:
                model, self.frames, self.mask, self.qs = synth_encoded(sub, torch.device("cpu"), 0, DLDKD)
                params = model.attention_params()
        if workload != "tvr_frame":
            with torch.no_grad():
                self.props, self.keys, self.vals = O.two_scale_corpus(self.frames, self.mask, params, shape["T"])

    def run(self, sample_queries, keep=False):
        """One timed pass -> dict for the JSON line (keep: also the fused matrix and the oracle's top-K ids)."""
        O = self.O
        qs = [q[:sample_queries] for q in self.qs]
        with torch.no_grad():
            t0 = time.perf_counter()
            if self.workload != "tvr_frame":
                fused, order = O.cpu_eval_two_scale(qs, self.props, self.keys, self.vals, self.mask, bsz=50, K=K_TOP)
            else:
                fused, order = O.cpu_eval_frame_head(qs, self.frames, self.mask, bsz=50, K=K_TOP)
            dt = time.perf_counter() - t0
        nv = self.mask.shape[0]
        pairs = sample_queries * nv
        out = {"value": pairs / dt, "unit": "pairs/s", "cores": self.threads, "kind": "port",
               "sample": f"{sample_queries} queries x {nv} videos ({self.workload}, oracle/oracle.py "
                         f"cpu_eval loop, batches of 50, torch {torch.__version__} CPU, {dt:.1f} s)",
               "seconds": dt}
        if keep:
            out["_fused"], out["_order"] = fused, order
        return out

    def detail(self, n):
        """Untimed: fused scores + key clips + fp32 key-clip tie mask of the first n queries (two-scale head), or the
        fused scores with an empty tie mask (frame head)."""
        O = self.O
        qs = [q[:n] for q in self.qs]
        with torch.no_grad():
            if self.workload != "tvr_frame":
                return O.two_scale_eval_detail(qs, self.props, self.keys, self.vals, self.mask, bsz=50)
            fused, _ = O.cpu_eval_frame_head(qs, self.frames, self.mask, bsz=50, K=K_TOP)
            return dict(fused=fused, tie=np.zeros_like(fused, dtype=bool))


class ReferenceBaseline:
    """The UNMODIFIED reference (baseline/_ref, staged by oracle/install_ref.py; imported through oracle/ref_shim.py)
    timed on the host cores for the head it ships: compute_query2ctx_info (method/eval.py:177-219: encode_query +
    get_sim_scores x 2 branches per batch of 50 + the dense D2H-style concatenation) -> 0.7/0.3 fusion (:254) ->
    eval_q2m (:59-94), on `sample_queries` raw queries x the full TVR-shaped corpus.  Setup (random-init reference
    model, synthetic raw features, the reference's own compute_context_info) is not timed."""

    def __init__(self, shape, max_queries, threads=None):
        staged = os.path.join(ROOT, "baseline", "_ref")
        if os.path.isdir(os.path.join(staged, "method")):
            os.environ["DKD_REFERENCE_ROOT"] = staged          # the staged copy, here and on the GPU box
        from oracle import ref_shim
        from oracle.datasets import QuerySet, VideoSet
        if os.environ.get("DKD_REFERENCE_ROOT"):
            ref_shim.REF_ROOT = os.environ["DKD_REFERENCE_ROOT"]
        if not ref_shim.available():
            raise RuntimeError("the reference is not staged: run `python oracle/install_ref.py` where /root/reference exists")
        self.rm, self.re, _ = ref_shim.load()
        self.shape, self.threads = shape, threads or os.cpu_count()
        torch.set_num_threads(self.threads)
        cfg = ref_shim.model_config(shape["Dv"], shape["Dq"], hidden=shape["H"], max_ctx_l=shape["L"], max_desc_l=shape["Lq"])
        self.opt = ref_shim.options()
        torch.manual_seed(0)
        self.model = self.rm.DLDKD(cfg, self.opt).eval()
        g = torch.Generator().manual_seed(1000)
        Nv, L, Dv, Lq, Dq = (shape[k] for k in ("Nv", "L", "Dv", "Lq", "Dq"))
        vids = []
        for _ in range(Nv):
            x = torch.randn(L, Dv, generator=g)
            vids.append(x / (x.norm(dim=-1, keepdim=True) + 1e-5))
        gq = torch.Generator().manual_seed(5_000_000)
        qlen = torch.randint(5, Lq + 1, (max_queries,), generator=gq)
        qs = []
        for n in range(max_queries):
            x = torch.randn(int(qlen[n]), Dq, generator=gq)
            qs.append(x / (x.norm(dim=-1, keepdim=True) + 1e-5))
        self.qset_cls, self.qs, self.Nv = QuerySet, qs, Nv
        with torch.no_grad():
            self.ctx = self.re.compute_context_info(self.model, VideoSet(vids), self.opt)
        self.root = ref_shim.REF_ROOT

    def run(self, sample_queries):
        qset = self.qset_cls(self.qs[:sample_queries], self.Nv)
        t2v = {q: [q % self.Nv] for q in range(sample_queries)}
        with torch.no_grad():
            t0 = time.perf_counter()
            inher, explore, _, metas = self.re.compute_query2ctx_info(self.model, qset, self.opt, self.ctx)
            fused = 0.7 * inher + 0.3 * explore
            order = {m: i for i, m in enumerate(metas)}
            gts = {order[qset.ids[q]]: t2v[q] for q in range(sample_queries)}
            metrics = self.re.eval_q2m(-1 * fused, gts)
            dt = time.perf_counter() - t0
        pairs = sample_queries * self.Nv
        return {"value": pairs / dt, "unit": "pairs/s", "cores": self.threads, "kind": "reference",
                "sample": f"{sample_queries} raw queries x {self.Nv} videos: unmodified reference compute_query2ctx_info + "
                          f"fusion + eval_q2m ({self.root}, torch {torch.__version__} CPU, {dt:.1f} s; R@1/5/10/100 = "
                          f"{[round(float(x), 2) for x in metrics[:4]]})",
                "seconds": dt}


def run_cpu_baseline(shape, workload, sample_queries, threads=None):
    return CpuBaseline(shape, workload, sample_queries, threads).run(sample_queries)


def parity_vs_oracle(cpu, n, dense_exact, dense_approx, top_ids, id_base=0):
    """The device results for the first n queries against the CPU oracle ON THE SAME TENSORS (north_star tolerances:
    fused scores 1e-3 for the bf16 path, 5e-6 for the exact path, outside the oracle's own fp32 key-clip ties; top-K
    ids identical up to swaps of oracle scores closer than 1e-5)."""
    O = cpu.O
    det = cpu.detail(n)
    tie = det["tie"]
    ref = det["fused"]
    d_ex = np.abs(dense_exact.float().cpu().numpy() - ref)[~tie].max()
    d_ap = np.abs(dense_approx.float().cpu().numpy() - ref)[~tie].max()
    rk = O.compare_ranking(ref, tie, top_ids.cpu().numpy() - id_base, top_ids.shape[1])
    ok = bool(d_ex <= 5e-6 and d_ap <= 1e-3 and rk["mismatches"] == 0)
    return {"queries": int(n), "videos": int(ref.shape[1]), "max_abs_err_exact_path": float(d_ex),
            "max_abs_err_timed_path": float(d_ap), "tol_exact": 5e-6, "tol_timed": 1e-3,
            "key_clip_tie_pairs": int(tie.sum()), "ranking": rk, "ok": ok,
            "what": "oracle/oracle.py two_scale_eval_detail (CPU fp32) on the encoded tensors the GPU scored"}


# ------------------------------------------------------------------------------------------------
def bench_c5_train(args, rank, world, dev):
    """BASELINE.json configs[4] from the encoded vectors on: batch 128 videos x 128 frames, 5 captions each (640
    queries), D = 384 (teacher 512): in-batch similarity x3 + triplet / soft-NCE / KL losses, forward + backward
    (train.losses_from_encoded).  value = (query, video) pairs per second through the whole step."""
    import types
    from dkd_b200 import train, _lib
    from tests import synth
    N, L, D, Dt, caps = 128, 128, 384, 512, 5
    M = N * caps
    labels = [i // caps for i in range(M)]
    ci, mask, _ = synth.encoded_corpus(N, L, D, seed=51 + rank)
    ce, ct = synth.encoded_corpus(N, L, D, seed=152 + rank)[0] * mask[:, :, None], \
        synth.encoded_corpus(N, L, Dt, seed=253 + rank)[0] * mask[:, :, None]
    qi, qe, qt = (synth.encoded_queries(M, d, seed=54 + k) for k, d in enumerate((D, D, Dt)))
    qi, qe, qt = qi + 0.5 * ci[labels, 0], qe + 0.5 * ce[labels, 0], qt + 0.5 * ct[labels, 0]
    host = [t.contiguous().pin_memory() for t in (qt, ct, qi, ci, qe, ce)]
    keys = ("teacher_q", "teacher_ctx", "inher_q", "inher_ctx", "explore_q", "explore_ctx")
    model = types.SimpleNamespace(
        config=types.SimpleNamespace(label_style="soft", margin=0.1, use_hard_negative=True, hard_pool_size=1),
        double_branch=True, weight=1, kl_intra_weight=0.1, inher_nce_weight=0.04, explore_nce_weight=0.04,
        alpha=0.8, belta=0.8)
    mask_d = mask.to(dev)
    last = {}                     # the leaves of the latest step: their gradients are what the step returns besides the loss

    def step(tensors):
        enc = {k: (t.detach().requires_grad_(k.startswith(("inher", "explore")))) for k, t in zip(keys, tensors)}
        loss, _ = train.losses_from_encoded(model, enc, labels, mask_d)
        loss.backward()
        last.update(enc)
        return loss.detach()

    resident = [t.to(dev) for t in host]
    for _ in range(max(args.warmup, 3)):
        step(resident)
    _lib.reset_counters()
    step(resident)
    launches = _lib.launch_count()
    torch.cuda.synchronize()
    sampler = ClockSampler(dev.index or 0)
    sampler.start()
    timed = ("dkd_train_sim_fwd", "dkd_train_sim_bwd", "dkd_kl_curve_loss", "dkd_row_inv_norms", "dkd_score_max_exact",
             "dkd_pack_rows_tf32", "dkd_normalize_rows", "dkd_train_curve", "dkd_train_losses")
    _lib.set_timed(set(timed))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss = step(resident)
    e1.record()
    torch.cuda.synchronize()
    clocks = sampler.result()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(loss=loss, **{"grad_" + k: last[k].grad for k in keys if last[k].requires_grad}))
    ms_step = e0.elapsed_time(e1) / args.steps
    tr = _lib.timed_results()
    fwd_ms = tr.get("dkd_score_max_exact", []) or tr.get("dkd_train_sim_fwd", [])
    kernels_ms = {k: {"calls_per_step": len(v) // max(args.steps, 1), "ms_per_step": float(np.sum(v)) / max(args.steps, 1)}
                  for k, v in tr.items() if v}
    _lib.set_timed(set())
    out_loss = torch.empty((), dtype=torch.float32).pin_memory()
    e0.record()
    for _ in range(args.steps):
        out_loss.copy_(step([t.to(dev, non_blocking=True) for t in host]), non_blocking=True)
    e1.record()
    torch.cuda.synchronize()
    e2e_ms = e0.elapsed_time(e1) / args.steps
    # CPU baseline: the oracle's loop-for-loop restatement of the reference, forward + backward, all threads
    from oracle import oracle as O
    torch.set_num_threads(os.cpu_count())
    cpu_s = []
    for _ in range(3):
        leaves = {k: t.clone().requires_grad_(k.startswith(("inher", "explore"))) for k, t in zip(keys, (qt, ct, qi, ci, qe, ce))}
        t0 = time.perf_counter()
        ref, _ = O.train_losses(leaves, labels, mask, use_hard_negative=True, hard_pool_size=1, label_style="soft")
        ref.backward()
        cpu_s.append(time.perf_counter() - t0)
    cpu_t = float(np.median(cpu_s))
    got = float(step(resident))
    pk = peaks()
    flops = 2.0 * M * N * L * (D + D + Dt) / 3.0      # average launch of the three similarity passes
    avg = float(np.mean(fwd_ms)) if fwd_ms else None
    line = {"metric": "query-video pairs scored fwd+bwd/sec (training step, from encoded vectors)",
            "value": M * N / (ms_step * 1e-3), "unit": "pairs/s", "n_gpus": 1, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "c5_train", "videos": N, "frames": L, "queries": M, "hidden": D, "teacher_dim": Dt,
                       "label_style": "soft", "hard_negative_pool": 1, "l2": "working set 60 MB, L2 resident (one batch)"},
            "clocks": clocks,
            "e2e": {"value": M * N / (e2e_ms * 1e-3), "unit": "pairs/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": int(sum(t.numel() * 4 for t in host)), "d2h_bytes_per_step": 4},
            "gpu_launches": launches * args.steps, "gpu_launches_per_step": launches,
            "roofline": {"bound": "tensor", "kernel": "exact_umma_kernel<1> (tcgen05 kind::tf32 x 3: in-batch cosine / raw maxima)"
                                                      if tr.get("dkd_score_max_exact") else "train_sim_fwd_kernel (fp32 SIMT dots)",
                         "achieved": flops / (avg * 1e-3) / 1e12 if avg else None, "peak": pk["bf16_burst"],
                         "unit": "TFLOP/s", "frac": flops / (avg * 1e-3) / 1e12 / pk["bf16_burst"] if avg else None,
                         "avg_launch_ms": avg, "launches_timed": len(fwd_ms), "traffic": None,
                         "note": "fp32-grade contraction: 3 tf32 MMAs per product, so its own ceiling is 1/6 of the bf16 peak; "
                                 "at 640 x 128 x 128 the launch is latency bound (5 tiles per CTA)"},
            "kernels_ms": kernels_ms,
            "parity": {"loss": got, "oracle_loss": float(ref), "abs_diff": abs(got - float(ref))},
            "cpu_baseline": {"value": M * N / cpu_t, "unit": "pairs/s", "cores": os.cpu_count(), "kind": "port",
                             "sample": f"the same batch, oracle.train_losses forward+backward, median of 3 ({cpu_t:.2f} s)"}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="dkd_b200", choices=["dkd_b200", "reference"])
    ap.add_argument("--workload", default="tvr_two_scale", choices=["tvr_two_scale", "tvr_frame", "c4_stream", "c5_train"])
    ap.add_argument("--c4-videos", type=int, default=125_000, help="c4_stream: videos per GPU (1 M / 8)")
    ap.add_argument("--c4-queries", type=int, default=100_000)
    ap.add_argument("--chunk-videos", type=int, default=8192, help="c4_stream: videos per streamed chunk")
    ap.add_argument("--query-batch", type=int, default=16384, help="c4_stream: queries per scoring call")
    ap.add_argument("--cpu-sample-queries", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-reference-leg", action="store_true", help="skip timing the unmodified reference's frame head")
    ap.add_argument("--no-eval-epoch", action="store_true", help="skip the wall-clock run of the reference-named eval_epoch entry")
    ap.add_argument("--no-encoder", action="store_true", help="skip timing encode_context (PyTorch mirror vs fused kernels)")
    ap.add_argument("--no-c4", action="store_true", help="skip the reduced c4_stream sub-measurement")
    ap.add_argument("--c4-sub-videos", type=int, default=32768)
    ap.add_argument("--c4-sub-queries", type=int, default=16384)
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling measurement (fixed 17,432-video corpus)")
    ap.add_argument("--strong-shards", type=int, default=8, help="strong scaling: corpus = this many 2,179-video shards")
    ap.add_argument("--profile", action="store_true", help="short run for ncu: no e2e / parity / cpu legs")
    ap.add_argument("--operand", default="bf16", choices=["bf16", "fp16", "shortcut"],
                    help="approximate pass: bf16 GEMM operands (north_star, default); IEEE-half operands (reported "
                         "variant: same tensor rate and bytes, 8 x smaller rounding error -> 8 x fewer ambiguous "
                         "pairs); shortcut (reported variant: no dense GEMM — exact clip scores for every pair "
                         "through 32 per-clip dots + window scan, approximate fp16 frame gather)")
    ap.add_argument("--candidates", type=int, default=K_CAND)
    ap.add_argument("--no-variants", action="store_true", help="skip the variants.shortcut measurement")
    ap.add_argument("--variants-multi-gpu", action="store_true", help=argparse.SUPPRESS)   # accepted, now the default
    ap.add_argument("--e2e-steps", type=int, default=None, help="timed steps of the e2e leg (default max(3, steps/2))")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (float32 / float64, <= 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "dkd_b200":
        ap.error("--dump-outputs writes the outputs of the dkd_b200 arm")
    if args.impl == "dkd_b200" and not args.profile:
        args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    stream = args.workload == "c4_stream"
    if stream:
        # BASELINE.json configs[3]: 1 M videos x 32 downsampled frames over 8 GPUs = 125 k videos per GPU
        shape = dict(Nv=args.c4_videos, L=32, Dv=None, Nq=args.c4_queries, Lq=None, Dq=None, H=384, T=32)
    else:
        shape = dict(TVR)
    head = "frame" if args.workload == "tvr_frame" else "two_scale"
    cfg_common = {"workload": args.workload, "videos_per_gpu": shape["Nv"], "frames": shape["L"],
                  "visual_dim": shape["Dv"], "queries": shape["Nq"], "hidden": shape["H"], "branches": 2,
                  "top_k": K_TOP, "l2": "inputs larger than L2 (bf16 corpus operand 884 MB/branch)"}
    if stream:
        cfg_common.update(chunk_videos=args.chunk_videos, query_batch=args.query_batch,
                          l2="inputs larger than L2 (resident clips 6.1 GB/branch; 3.3 GB bf16 operand per chunk)")
    # the CPU legs run a bounded sample: a corpus slice for the streamed config (the full shard's proposals
    # would need 100 GB of host memory), the full corpus otherwise
    cpu_shape = dict(shape, Nv=min(shape["Nv"], 2048)) if stream else shape

    import __graft_entry__ as ge
    ge.load_package()

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        nq = args.cpu_sample_queries or (1000 if head == "two_scale" else 4000)
        # the head the reference ships runs the UNMODIFIED reference (kind "reference"); the two-scale head does not
        # exist in the reference (SURVEY section 8 a-NS), so that workload times the oracle port of its eval loop
        use_ref = args.workload == "tvr_frame"
        cpu = ReferenceBaseline(cpu_shape, nq) if use_ref else CpuBaseline(cpu_shape, args.workload, nq)
        first = cpu.run(50)                                     # untimed: also sizes the sample
        for _ in range(max(args.warmup - 1, 0)):
            cpu.run(50)
        # keep the whole run within a few minutes: K steps x sample <= ~200 s of CPU work
        budget_q = int(first["value"] * (200.0 / max(args.steps, 1)) / cpu_shape["Nv"]) // 50 * 50
        nq = max(50, min(nq, budget_q))
        vals, last = [], None
        for _ in range(max(args.steps, 1)):
            last = cpu.run(nq)
            vals.append(last["value"])
        v = float(np.mean(vals))
        sec = float(np.mean([nq * cpu_shape["Nv"] / x for x in vals]))
        line = {"impl": "reference", "metric": "query-video pairs scored+ranked/sec", "value": v, "unit": "pairs/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "config": cfg_common,
                "cpu_baseline": {"value": v, "unit": "pairs/s", "cores": last["cores"], "kind": last["kind"],
                                 "sample": last["sample"]},
                "e2e": {"value": v, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------ dkd_b200 arm
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if args.workload == "c5_train":          # single-GPU secondary workload (replicas only: one batch per GPU)
        if rank == 0:
            bench_c5_train(args, rank, world, dev)
        return
    import torch.distributed as dist
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"      # keep stdout to the one JSON line (NCCL prints its version there)
        dist.init_process_group("nccl", device_id=dev)
    from dkd_b200 import engine, ops, _lib
    from dkd_b200.model import DLDKD
    _lib.load()

    Nq, Nv = shape["Nq"], shape["Nv"]
    cert_mode = ["deferred"]     # how engine.rank's candidate certificate is read: see step() below
    if stream:
        # the shard stays resident as encoded clips; operands are rebuilt chunk by chunk INSIDE the step
        frames, mask, qs, attn = synth_c4(shape, dev, rank)
        torch.cuda.synchronize()
        prep_ms, pc = None, None

        def step(q_dev, precision=args.operand):
            pqs = engine.split_queries(q_dev, args.query_batch)
            chunks = engine.iter_chunks(frames, mask, args.chunk_videos, id_base=rank * Nv)
            s, i = engine.rank_streamed(chunks, pqs, attn, K=K_TOP, T=shape["T"], precision=precision, Kc=args.candidates)
            if world > 1:
                s, i = engine.merge_shards(s, i)
            return s, i
    else:
        model, frames, mask, qs = synth_encoded(shape, dev, rank, DLDKD)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        pc = engine.prepare_corpus(frames, mask, [tuple(t.detach() for t in p) for p in model.attention_params()],
                                   T=shape["T"], heads=(head,), precisions=("exact", args.operand),
                                   id_base=rank * shape["Nv"])
        e1.record()
        torch.cuda.synchronize()
        prep_ms = e0.elapsed_time(e1)
        attn_cpu = [tuple(t.detach().float().cpu() for t in p) for p in model.attention_params()]
        host_tensors = None
        if rank == 0 and not args.no_cpu_baseline and not args.profile:   # the oracle scores these very tensors
            host_tensors = ([f.float().cpu() for f in frames], mask.float().cpu(), None, attn_cpu)
        del frames
        qs = [q.contiguous() for q in qs]

        def step(q_dev, precision=args.operand, corpus=None, cert=None):
            # no host synchronisation inside: the candidate certificate of every call is queued on the device and
            # resolved by engine.finish() before the lists are consumed (after the timed loop / one step later in e2e)
            pq = engine.prepare_queries(q_dev)
            s, i = engine.rank(corpus or pc, pq, K=K_TOP, head=head, precision=precision, rescore=True, Kc=args.candidates,
                               certify=cert_mode[0] if cert is None else cert)
            if world > 1:
                s, i = engine.merge_shards(s, i)
            return s, i

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def any_rank(flag):
        """True on every rank if `flag` is true on any rank (decisions that change the sequence of collectives must
        be taken together)."""
        if world == 1:
            return bool(flag)
        t = torch.tensor([1 if flag else 0], device=dev, dtype=torch.int32)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return bool(t.item())

    log("corpus prepared; warm-up")
    # warm-up (also: one pass to count kernel launches per step)
    for _ in range(args.warmup):
        step(qs)
    _lib.reset_counters()
    step(qs)
    launches_per_step = _lib.launch_count()
    barrier()

    log("timed region")
    # ---- timed region: device-resident inputs
    sampler = ClockSampler(local_rank)
    sampler.start()
    # the dominant kernel's entry point: the two-scale head calls the GEMM through dkd_score_max_bf16_lists (ambiguous
    # pairs listed by the epilogue), the frame head through dkd_score_max_bf16 / _f16
    if args.operand == "shortcut":
        gemm_entry = "dkd_clip_score_f32"
    elif head == "two_scale":
        gemm_entry = "dkd_score_max_bf16_lists"
    else:
        gemm_entry = "dkd_score_max_f16" if args.operand == "fp16" else "dkd_score_max_bf16"
    _lib.set_timed({gemm_entry})
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    barrier()
    engine.finish()
    fallbacks_before = engine.STATS["certify_fallback_queries"]
    ev[0].record()
    for _ in range(args.steps):
        top_s, top_i = step(qs)
    ev[1].record()
    barrier()
    # deferred certificates of the timed steps: a fallback (never observed at these shapes) would have been applied
    # AFTER the timed region, so in that case the steps are timed again with the certificate read back inside each step
    engine.finish()
    if any_rank(engine.STATS["certify_fallback_queries"] > fallbacks_before) and not stream:
        cert_mode[0] = True
        _lib.set_timed({gemm_entry})
        barrier()
        ev[0].record()
        for _ in range(args.steps):
            top_s, top_i = step(qs)
        ev[1].record()
        barrier()
    clocks = sampler.result()
    timed_fallbacks = engine.STATS["certify_fallback_queries"] - fallbacks_before   # 0: nothing was re-ranked
    ms_total = ev[0].elapsed_time(ev[1])
    gemm_ms = _lib.timed_results().get(gemm_entry, [])
    _lib.set_timed(set())
    if args.dump_outputs and rank == 0:   # the lists of the last timed step (merged over the ranks for N > 1)
        dump_outputs(args.dump_outputs, {"top_scores": top_s, "top_ids": top_i})
    if world > 1:
        t = torch.tensor([ms_total], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    ms_step = ms_total / args.steps
    pairs_step = Nq * Nv * world
    value = pairs_step / (ms_step * 1e-3)

    if args.profile:
        if rank == 0:
            print(json.dumps({"profile_run": True, "ms_per_step": ms_step, "value": value}))
        return
    # ---- step budget: 3 more steps with EVERY C-ABI entry bracketed by CUDA events (not part of the timed region:
    # the brackets serialise the launches a little); per entry: calls per step and ms per step
    kernels_ms = None
    if not stream:                       # every rank runs the steps (they contain the merge collectives); rank 0 reports
        _lib.set_timed(set(_lib.PROTOTYPES))
        for _ in range(3):
            step(qs)
        engine.finish()
        kernels_ms = {k: {"calls_per_step": len(v) // 3, "ms_per_step": round(float(np.sum(v)) / 3, 4)}
                      for k, v in _lib.timed_results().items() if v}
        _lib.set_timed(set())
        barrier()
    log("e2e leg")
    # ---- e2e: host buffers in, host buffers out, through the same public entry (engine.rank)
    q_host = [q.cpu().pin_memory() for q in qs]
    out_s = torch.empty((Nq, K_TOP), dtype=torch.float32).pin_memory()
    out_i = torch.empty((Nq, K_TOP), dtype=torch.int32).pin_memory()

    copy_stream = torch.cuda.Stream(dev)

    e2e_fb = [0]

    def run_e2e(n_steps):
        """n_steps passes, each fed from pinned host memory and drained to pinned host memory.  The copies of
        step i+1 (H2D) and step i-1 (D2H) run on a copy stream under the kernels of step i."""
        main = torch.cuda.current_stream()
        engine.finish()
        e2e_fb[0] = engine.STATS["certify_fallback_queries"]

        def upload():
            with torch.cuda.stream(copy_stream):
                qd = [q.to(dev, non_blocking=True) for q in q_host]
                ev = torch.cuda.Event()
                ev.record(copy_stream)
            return qd, ev

        nxt = upload()
        for i in range(n_steps):
            qd, ev = nxt
            if i + 1 < n_steps:
                nxt = upload()
            main.wait_event(ev)
            for t in qd:
                t.record_stream(main)
            s, ids = step(qd)
            done = torch.cuda.Event()
            done.record(main)
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(done)
                out_s.copy_(s, non_blocking=True)
                out_i.copy_(ids, non_blocking=True)
            s.record_stream(copy_stream)
            ids.record_stream(copy_stream)
        main.wait_stream(copy_stream)          # the last result has reached host memory
        # the steps' certificates are looked at once here (no host synchronisation inside the loop); a fallback would
        # have patched lists that were already copied out, so in that case the leg is timed again with the certificate
        # read back inside every step
        engine.finish()
        if engine.STATS["certify_fallback_queries"] > e2e_fb[0]:
            cert_mode[0] = True

    run_e2e(1 if stream else 2)
    barrier()
    e2e_steps = args.e2e_steps or max(3, args.steps // 2)
    ev2 = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev2[0].record()
    run_e2e(e2e_steps)
    ev2[1].record()
    barrier()
    if any_rank(cert_mode[0] is True) and not stream:      # see run_e2e: time it again with the in-step certificate
        cert_mode[0] = True
        ev2[0].record()
        run_e2e(e2e_steps)
        ev2[1].record()
        barrier()
    e2e_ms = ev2[0].elapsed_time(ev2[1]) / e2e_steps
    if world > 1:
        t = torch.tensor([e2e_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    e2e = {"value": pairs_step / (e2e_ms * 1e-3), "unit": "pairs/s",
           "h2d_bytes_per_step": int(sum(q.numel() * 4 for q in q_host)),
           "d2h_bytes_per_step": int(out_s.numel() * 4 + out_i.numel() * 4), "ms_per_step": e2e_ms,
           "boundary": "encoded query vectors in pinned host memory -> engine.rank -> top-100 (score, id) in host memory; "
                       "copies on a side stream, overlapped with the neighbouring steps' kernels"}

    log("parity vs exact path")
    # ---- parity of the timed result: bf16+rescore top-100 == exact fp32 path top-100, EVERY query (in slices of
    # 2,048 to bound the exact path's dense temporaries)
    same_ids = same_scores = True
    nchk = min(512, Nq)
    n_par = nchk if stream else Nq          # streamed config: the all-exact pass over 125 k videos is bounded to 512 queries
    for lo in range(0, n_par, 2048):
        hi = min(lo + 2048, n_par)
        s_ex, i_ex = step([q[lo:hi] for q in qs], precision="exact")
        same_ids &= bool(torch.equal(i_ex, top_i[lo:hi]))
        same_scores &= bool(torch.equal(s_ex, top_s[lo:hi]))
    if n_par != nchk:
        s_ex, i_ex = step([q[:nchk] for q in qs], precision="exact")
    parity = {"queries_checked": n_par, "top100_ids_identical_to_exact_fp32": same_ids,
              "top100_scores_identical": same_scores}

    log("variants")
    # ---- reported variant, same run / same box: the linearity-shortcut pass (exact clip scale for every pair, no dense
    # GEMM; DESIGN.md section 4).  Not the headline: north_star specifies the dense bf16 GEMM.
    variants = None
    if head == "two_scale" and args.operand != "shortcut" and not stream and not args.no_variants:
        for _ in range(2):
            step(qs, precision="shortcut")
        barrier()
        vsteps = max(3, args.steps // 4)
        engine.finish()
        v_fb = engine.STATS["certify_fallback_queries"]
        ev3 = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev3[0].record()
        for _ in range(vsteps):
            v_s, v_i = step(qs, precision="shortcut")
        ev3[1].record()
        barrier()
        engine.finish()
        if any_rank(engine.STATS["certify_fallback_queries"] > v_fb):   # a deferred certificate failed somewhere
            v_s, v_i = step(qs, precision="shortcut", cert=True)
        v_ms = ev3[0].elapsed_time(ev3[1]) / vsteps
        if world > 1:
            t = torch.tensor([v_ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            v_ms = float(t.item())
        variants = {"shortcut": {"ms_per_step": v_ms, "value": pairs_step / (v_ms * 1e-3), "unit": "pairs/s", "steps": vsteps,
                                 "top100_identical_to_exact_fp32": bool(torch.equal(v_i[:nchk], i_ex) and torch.equal(v_s[:nchk], s_ex)),
                                 "what": "precision='shortcut': exact clip scores for every pair via 32 per-clip dots "
                                         "(tcgen05 kind::tf32 x 3) + window scan, fp16 frame gather, exact frame "
                                         "rescoring of the candidates; no dense GEMM, no ambiguity pass"}}

    log("encoder leg (rank 0)")
    # ---- the step right before the path (SURVEY section 8 f1): DLDKD.encode_context over the TVR corpus, PyTorch / cuBLAS
    # mirror against the fused encoder kernels (tcgen05 kind::tf32 x 3 linears + LayerNorm / attention kernels), same
    # synthetic raw features; query independent, run once per corpus, NOT part of the timed step
    encoder = None
    if not stream and rank == 0 and not args.no_encoder:
        g = torch.Generator(device=dev).manual_seed(4242)
        Bv = 200                                                       # eval_context_bsz (method/config.py:48)
        xraw = torch.randn(Bv, shape["L"], shape["Dv"], device=dev, generator=g)
        xraw = xraw / (xraw.norm(dim=-1, keepdim=True) + 1e-5)
        mk = torch.ones(Bv, shape["L"], device=dev)
        nbatch = (Nv + Bv - 1) // Bv

        def enc_time():
            with torch.no_grad():
                model.encode_context(xraw, mk)
                torch.cuda.synchronize()
                t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0.record()
                for _ in range(nbatch):
                    a, b = model.encode_context(xraw, mk)
                t1.record()
                torch.cuda.synchronize()
            return t0.elapsed_time(t1), a, b

        model.enable_fused_encoder(False)
        ms_ref, ra, rb = enc_time()
        model.enable_fused_encoder(True)
        ms_fused, fa, fb = enc_time()
        model.enable_fused_encoder(False)
        enc_flops = nbatch * (2.0 * Bv * shape["L"] * (shape["Dv"] * shape["H"] + 5 * shape["H"] ** 2) * 2
                              + 2.0 * 2 * 2 * Bv * shape["L"] * shape["L"] * shape["H"])
        encoder = {"videos": nbatch * Bv, "ms_pytorch_cublas_fp32": ms_ref, "ms_fused_kernels": ms_fused,
                   "speedup": ms_ref / ms_fused, "fp32_grade_tflops_fused": enc_flops / (ms_fused * 1e-3) / 1e12,
                   "max_abs_diff_vs_pytorch": float(max((fa - ra).abs().max(), (fb - rb).abs().max())),
                   "tolerance": 1e-4, "default": "opt-in (model.enable_fused_encoder()); see DESIGN.md section 6b"}
        del xraw, ra, rb, fa, fb

    log("eval_epoch leg (rank 0)")
    # ---- the reference-named entry end to end: eval_epoch(model, video_dataset, text_dataset, opt) (method/eval.py:237-263)
    # on in-memory datasets of RAW synthetic features (the reference's item layout), wall clock: DataLoader collation,
    # H2D, encode_context / encode_query (PyTorch), corpus preparation, device ranking (opt.precision = "bf16": no
    # dense D2H), R@K on the device.  Once more with opt.precision = "exact" (the reference's dense flow): the R-sums of
    # the two flows must be equal — R@K parity through the drop-in entry at the full TVR shape.
    eval_epoch_leg = None
    if not stream and rank == 0 and not args.no_eval_epoch and head == "two_scale":
        from oracle.datasets import QuerySet, VideoSet
        from dkd_b200 import eval as E
        g = torch.Generator(device=dev).manual_seed(77)
        vids = []
        for lo_ in range(0, Nv, 200):
            x = torch.randn(min(200, Nv - lo_), shape["L"], shape["Dv"], device=dev, generator=g)
            vids.extend((x / (x.norm(dim=-1, keepdim=True) + 1e-5)).cpu().unbind(0))
        qlen = torch.randint(5, shape["Lq"] + 1, (Nq,), generator=torch.Generator().manual_seed(78))
        xq = torch.randn(Nq, shape["Lq"], shape["Dq"], device=dev, generator=g)
        xq = (xq / (xq.norm(dim=-1, keepdim=True) + 1e-5)).cpu()
        qset = QuerySet([xq[i, : int(qlen[i])] for i in range(Nq)], Nv)
        vset = VideoSet(vids)
        del xq
        import types
        opt_e = types.SimpleNamespace(eval_context_bsz=200, eval_query_bsz=50, num_workers=0, pin_memory=False, device=dev,
                                      double_branch=True, scoring="two_scale", precision=args.operand)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rsum_fast = E.eval_epoch(model, vset, qset, opt_e)
        torch.cuda.synchronize()
        t_fast = time.perf_counter() - t0
        opt_e.precision = "exact"
        t0 = time.perf_counter()
        rsum_exact = E.eval_epoch(model, vset, qset, opt_e)
        torch.cuda.synchronize()
        t_exact = time.perf_counter() - t0
        eval_epoch_leg = {"entry": "dkd_b200.eval.eval_epoch(model, video_dataset, text_dataset, opt)  [method/eval.py:237-263]",
                          "seconds_hot_path": t_fast, "pairs_per_s_hot_path": Nq * Nv / t_fast,
                          "seconds_reference_flow_exact": t_exact, "rsum_hot_path": rsum_fast, "rsum_exact_flow": rsum_exact,
                          "rsum_identical": bool(rsum_fast == rsum_exact),
                          "what": "wall clock incl. DataLoader collation of 4.4 GB of raw features (host Python, like the "
                                  "reference), H2D, PyTorch encoders, corpus preparation; the device ranking itself is the "
                                  "timed step above"}
        del vids, vset, qset
        torch.cuda.empty_cache()

    log("strong-scaling leg")
    # ---- strong scaling: ONE fixed corpus of strong_shards x 2,179 videos (the concatenation of the weak-scaling
    # shards 0..7: 17,432 videos, 62 GB of operands on one GPU), split in contiguous blocks over the N ranks; same
    # queries, same step, same merge.  value = Nq x 17,432 / max-over-ranks time: it can fall short of N x the 1-GPU
    # number (merge, tail effects, smaller per-rank GEMMs), unlike the weak-scaling headline.
    strong = None
    if not stream and not args.no_strong and head == "two_scale":
        G = args.strong_shards
        tot = G * Nv
        lo, hi = engine.shard_range(tot, rank, world)
        fr_s, mk_s = [[], []], []
        for g in range(lo // Nv, (hi - 1) // Nv + 1):
            _, f_g, m_g, _ = synth_encoded(shape, dev, g, DLDKD, want_queries=False)
            a, b = max(lo, g * Nv) - g * Nv, min(hi, (g + 1) * Nv) - g * Nv
            fr_s[0].append(f_g[0][a:b])
            fr_s[1].append(f_g[1][a:b])
            mk_s.append(m_g[a:b])
        pc_s = engine.prepare_corpus([torch.cat(x) for x in fr_s], torch.cat(mk_s),
                                     [tuple(t.detach() for t in p) for p in model.attention_params()], T=shape["T"],
                                     heads=(head,), precisions=("exact", args.operand), id_base=lo)
        del fr_s, mk_s
        for _ in range(2):
            step(qs, corpus=pc_s)
        barrier()
        ssteps = max(3, args.steps // 4)
        engine.finish()
        s_fb = engine.STATS["certify_fallback_queries"]
        ev4 = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev4[0].record()
        for _ in range(ssteps):
            st_s, st_i = step(qs, corpus=pc_s)
        ev4[1].record()
        barrier()
        engine.finish()                           # local: patches this rank's lists in place if a certificate failed
        strong_fallbacks = engine.STATS["certify_fallback_queries"] - s_fb
        if any_rank(strong_fallbacks):            # ... after they were merged: redo one step with the in-step read-back
            st_s, st_i = step(qs, corpus=pc_s, cert=True)
        s_ms = ev4[0].elapsed_time(ev4[1]) / ssteps
        if world > 1:
            t = torch.tensor([s_ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            s_ms = float(t.item())
        # cross-check (cheap, integer): the merged lists are sorted, hold valid unique global ids
        ok = bool((st_s[:, :-1] >= st_s[:, 1:]).all()) and int(st_i.min()) >= 0 and int(st_i.max()) < tot
        strong = {"scaling": "strong", "corpus_videos": tot, "videos_per_gpu": hi - lo, "ms_per_step": s_ms,
                  "value": Nq * tot / (s_ms * 1e-3), "unit": "pairs/s", "steps": ssteps, "lists_valid": ok,
                  "checksum_ids": int(st_i.long().sum().item()), "certificate_fallbacks_rank0": strong_fallbacks,
                  "what": "fixed corpus = weak-scaling shards 0..%d concatenated, contiguous blocks per rank; "
                          "checksum_ids must be the same at every N" % (G - 1)}
        del pc_s
        torch.cuda.empty_cache()

    log("c4_stream leg")
    # ---- BASELINE.json configs[3] at a driver-runnable size (the default run has no flags): the streamed engine on
    # c4_sub_videos clip-feature videos PER GPU x c4_sub_queries queries, chunked exactly like the full config
    # (--workload c4_stream runs the 125 k x 100 k per-GPU size), operand building inside the step, N-way merge.
    c4 = None
    if not stream and not args.no_c4 and head == "two_scale":
        c4shape = dict(Nv=args.c4_sub_videos, L=32, Dv=None, Nq=args.c4_sub_queries, Lq=None, Dq=None, H=384, T=32)
        fr4, mk4, q4, at4 = synth_c4(c4shape, dev, rank)

        def c4_step(precision=args.operand):
            pqs = engine.split_queries(q4, args.query_batch)
            chunks = engine.iter_chunks(fr4, mk4, args.chunk_videos, id_base=rank * c4shape["Nv"])
            s4, i4 = engine.rank_streamed(chunks, pqs, at4, K=K_TOP, T=32, precision=precision, Kc=args.candidates)
            if world > 1:
                s4, i4 = engine.merge_shards(s4, i4)
            return s4, i4

        c4_step()
        barrier()
        c4steps = 2
        ev5 = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev5[0].record()
        for _ in range(c4steps):
            c4_s, c4_i = c4_step()
        ev5[1].record()
        barrier()
        c4_ms = ev5[0].elapsed_time(ev5[1]) / c4steps
        if world > 1:
            t = torch.tensor([c4_ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            c4_ms = float(t.item())
        e4_s, e4_i = c4_step(precision="exact") if world == 1 else (c4_s, c4_i)
        c4 = {"workload": "c4_stream (reduced)", "videos_per_gpu": c4shape["Nv"], "queries": c4shape["Nq"],
              "chunk_videos": args.chunk_videos, "query_batch": args.query_batch, "ms_per_step": c4_ms, "steps": c4steps,
              "value": c4shape["Nq"] * c4shape["Nv"] * world / (c4_ms * 1e-3), "unit": "pairs/s",
              "top100_identical_to_exact_fp32": bool(torch.equal(e4_i, c4_i) and torch.equal(e4_s, c4_s)) if world == 1 else None,
              "what": "rank_streamed: operands of every 8,192-video chunk rebuilt inside the step, running top-100 fold"}
        del fr4, mk4, q4
        torch.cuda.empty_cache()

    log("reporting / CPU legs (rank 0)")
    if rank == 0:
        pk = peaks()
        P = ops.num_proposals(shape["T"])
        R = P if head == "two_scale" else shape["L"]
        # algorithmic flops of one branch's contraction over the whole step; the streamed config spreads them
        # over (chunks x query batches) launches, so "per launch" is the average launch
        n_launch_step = max(len(gemm_ms) // max(args.steps, 1), 1)
        flops_launch = 2.0 * Nq * Nv * R * shape["H"] * 2 / n_launch_step
        gemm_avg_ms = float(np.mean(gemm_ms)) if gemm_ms else None
        achieved = flops_launch / (gemm_avg_ms * 1e-3) / 1e12 if gemm_avg_ms else None
        traffic = None
        tp = os.path.join(ROOT, "profiles", "r2_traffic.json")
        if os.path.exists(tp):
            traffic = json.load(open(tp)).get(args.workload)
        roofline = {"bound": "tensor", "kernel": "score_max_bf16_kernel (tcgen05 GEMM + fused max/argmax)" +
                                                   {"fp16": " on IEEE-half operands", "shortcut": " REPLACED by exact_umma_kernel (shortcut variant; "
                                                    "achieved = algorithmic flops of the dense contraction / time)"}.get(args.operand, ""),
                    "achieved": achieved, "peak": pk["bf16_burst"], "unit": "TFLOP/s",
                    "frac": achieved / pk["bf16_burst"] if achieved else None,
                    "frac_of_sustained_peak": achieved / pk["bf16_sustained"] if achieved else None,
                    "peak_source": f"MEASURED_PEAKS.json bf16_tflops (burst), {pk['source']}",
                    "flops_per_launch": flops_launch, "launches_timed": len(gemm_ms), "avg_launch_ms": gemm_avg_ms,
                    "share_of_step": (n_launch_step * gemm_avg_ms / ms_step) if gemm_avg_ms else None,
                    "traffic": traffic}
        # the WHOLE step against the same roofline (north_star's target; SURVEY.md §8d counts the contraction's
        # algorithmic flops only and quotes the target on the sustained peak: the step is a long back-to-back loop)
        step_flops = flops_launch * n_launch_step                      # per GPU: every rank scores its own shard
        step_tf = step_flops / (ms_step * 1e-3) / 1e12
        roofline["step"] = {"algorithmic_flops_per_gpu": step_flops, "achieved": step_tf, "unit": "TFLOP/s per GPU",
                            "frac_of_burst_peak": step_tf / pk["bf16_burst"],
                            "frac_of_sustained_peak": step_tf / pk["bf16_sustained"]}
        line = {"metric": "query-video pairs scored+ranked/sec", "value": value, "unit": "pairs/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": {"bf16": "bf16", "fp16": "f16", "shortcut": "tf32x3"}[args.operand],
                "data": "synthetic", "config": cfg_common,
                "engine": {"parallelism": f"video-shard x{world}", "candidates": args.candidates, "rescoring": "exact fp32"},
                "clocks": clocks, "e2e": e2e, "gpu_launches": launches_per_step * args.steps,
                "gpu_launches_per_step": launches_per_step, "roofline": roofline, "prep_ms": prep_ms,
                "corpus_bytes": pc.nbytes() if pc is not None else int(sum(f.numel() * 4 for f in frames)),
                "kernels_ms": kernels_ms, "parity": parity, "variants": variants, "strong": strong, "c4_stream": c4, "encoder": encoder, "eval_epoch": eval_epoch_leg,
                "certify": {"eps": engine.CERT_EPS, "checked_queries": engine.STATS["certify_checked_queries"],
                            "fallback_queries": engine.STATS["certify_fallback_queries"],
                            "fallback_queries_in_timed_steps": timed_fallbacks,
                            "note": "queries whose exact 100th score is within eps of the last candidate's approximate "
                                    "score are re-ranked by the all-exact path (all calls of this process)"}}
        failed = not (parity["top100_ids_identical_to_exact_fp32"] and parity["top100_scores_identical"])
        if eval_epoch_leg is not None and not eval_epoch_leg["rsum_identical"]:
            failed = True
        if not args.no_cpu_baseline:
            # CPU leg: the oracle port of the reference's eval loop on the SAME encoded tensors (bounded sample of
            # queries x the full corpus, >= ~20 s of CPU work), timed; then, untimed, the parity of the timed GPU
            # result against it (parity.vs_oracle)
            nq = args.cpu_sample_queries or (800 if head == "two_scale" else 3200)
            nq = min(nq, Nq)
            if stream:
                nv_cpu = cpu_shape["Nv"]
                tensors = ([f[:nv_cpu].float().cpu() for f in frames], mask[:nv_cpu].float().cpu(),
                           [q[:nq].float().cpu() for q in qs], [tuple(t.float().cpu() for t in p) for p in attn])
            else:
                tensors = host_tensors[:2] + ([q[:nq].detach().float().cpu() for q in qs], host_tensors[3])
            cpu = CpuBaseline(cpu_shape, args.workload, nq, tensors=tensors)
            cpu.run(50)                                                   # warm the CPU kernels / allocator, untimed
            line["cpu_baseline"] = cpu.run(nq)
            if not stream and not args.no_reference_leg:
                # beside it: the UNMODIFIED reference (baseline/_ref) on the head it ships, same corpus shape — for
                # the tvr_frame workload this IS the cpu_baseline (kind "reference")
                try:
                    nr = min(Nq, 4000)                                  # ~15-20 s of CPU work on 16 threads
                    refb = ReferenceBaseline(shape, nr)
                    refb.run(50)
                    rline = refb.run(nr)
                    if args.workload == "tvr_frame":
                        line["cpu_baseline_port"], line["cpu_baseline"] = line["cpu_baseline"], rline
                    else:
                        line["cpu_reference_frame_head"] = rline
                except Exception as e:                                     # noqa: BLE001 - reported, not fatal
                    line["cpu_reference_frame_head"] = {"unavailable": f"{type(e).__name__}: {e}"}
            nd = min(nq, 150)
            qd = [q[:nd].contiguous() for q in qs]
            if stream:   # the oracle's corpus slice, ranked by the same engine entry as the streamed chunks
                pcs = engine.prepare_corpus([f[:nv_cpu] for f in frames], mask[:nv_cpu], attn, T=shape["T"],
                                            heads=(head,), precisions=("exact", args.operand), id_base=rank * Nv)
                pqd = engine.prepare_queries(qd)
                _, ids_d = engine.rank(pcs, pqd, K=K_TOP, head=head, precision=args.operand, Kc=args.candidates)
                id_base = rank * Nv
            else:
                pcs, pqd, id_base = pc, engine.prepare_queries(qd), rank * Nv
                ids_d = top_i[:nd]                     # the TIMED result itself
                if world > 1:                          # merged lists hold other ranks' videos: rank 0's local lists
                    _, ids_d = engine.rank(pc, pqd, K=K_TOP, head=head, precision=args.operand, Kc=args.candidates)
            if head == "two_scale":
                dense_ex = engine.score_two_scale_head(pcs, pqd, "exact")[0]
                dense_ap = engine.score_two_scale_head(pcs, pqd, args.operand)[0]
            else:
                fr_ex, fr_ap = engine.score_frame_head(pcs, pqd, "exact"), engine.score_frame_head(pcs, pqd, args.operand)
                dense_ex = ops.fuse_scores(fr_ex[0][0], fr_ex[1][0], 0.7, 0.3)
                dense_ap = ops.fuse_scores(fr_ap[0][0], fr_ap[1][0], 0.7, 0.3)
            parity["vs_oracle"] = parity_vs_oracle(cpu, nd, dense_ex, dense_ap, ids_d, id_base)
            failed = failed or not parity["vs_oracle"]["ok"]
        if failed:
            line["parity_failed"] = True
        print(json.dumps(line))
        if failed:   # a fast result that differs from the reference's is not a result
            sys.stdout.flush()
            os._exit(1)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
