#!/usr/bin/env python
"""bench.py — the BASELINE.json configs on B200, one JSON line (contract: DESIGN.md §Measurement).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload all|vitl14|knn|ivf|e2e|plumbing]
                  [--dump-outputs DIR]

Workloads (BASELINE.json `configs`):
  plumbing configs[0] ViT-B/32 clip_inference on 100 synthetic images + captions: the original project's reader /
                      runner / writer job, replayed from its record, around the CUDA ClipMapper -> samples/s
  vitl14  configs[1]  ViT-L/14 image+text inference, synthetic 224^2, batch 1024 per GPU   -> pairs/s
  knn     configs[2]  brute-force cosine kNN, 100M x 768 fp16 rows per GPU, 1000 queries, top-40 -> queries/s
  ivf     configs[3]  IVF-Flat (nlist 65536, nprobe 16/64), rows range-sharded over the ranks, one all-gather -> queries/s
  e2e     configs[4]  clip_back query path: ViT-H/14 text -> embed -> sharded IVF kNN -> ids on the host, p50/p99 + QPS
`--workload all` (the default) prints the vitl14 line (the headline metric's first half) with the other four
nested under "knn", "ivf", "e2e_query", "plumbing" — each a complete sub-line with its own `roofline`, `cpu_baseline`,
`e2e` and `parity_checked`.  `--workload X` prints X's line alone.

Per line: `value` = whole-job throughput with inputs resident in HBM (CUDA events, barrier + sync both sides,
max over ranks); `e2e` = the same metric through the host-buffer API (H2D/D2H inside the timed region);
`roofline` = the dominant kernel's algorithmic work / its event-timed duration against MEASURED_PEAKS.json;
`cpu_baseline` = the oracle port on the host cores on a bounded sample (rank 0, N=1 only);
`parity_checked` = results of the timed configuration verified after the timed region (oracle as the checker).
`--impl reference`: the CPU oracle port of the same workload on the host cores (bounded sample per step).
`--dump-outputs DIR`: after the timed steps, rank 0 writes what each timed path returned in its last step as
DIR/<workload>_<array>.npy (float32, ids as float64; a seeded row sample of an array over 4 MB, its row numbers in
DIR/<workload>_<array>_rows.npy).  Inputs and weights are seeded, so two builds can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}
# The reference's published ViT-L/14 numbers (BASELINE.md section 1): samples/s by GPU count, A100.
PUBLISHED_VITL14 = {1: 312.0, 8: 2500.0}
TOL = 2e-6   # |fp32 sum - exact| of unit vectors, d <= 1024 (tests/test_knn_gpu.py)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        d["_source"] = "measured"
        return d
    d = dict(FALLBACK_PEAKS)
    d["_source"] = "fallback"
    return d


def load_traffic(key):
    """Per-launch DRAM bytes of a kernel from the committed ncu summary of this round (profiles/r02_traffic.json)."""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if not os.path.exists(p):
        return None, None
    t = json.load(open(p)).get(key)
    if not t:
        return None, None
    return t.get("bytes_per_launch"), t.get("source")


def physical_cores():
    try:
        import psutil

        n = psutil.cpu_count(logical=False)
        if n:
            return int(n)
    except Exception:
        pass
    return max(1, (os.cpu_count() or 2) // 2)


# ---- algorithmic work (DESIGN.md §Measurement; SURVEY.md §8d) -----------------------------------------
def tower_gemm_flops(t, tokens):
    w, mlp = t.width, t.mlp
    return t.layers * 2 * tokens * (w * 3 * w + w * w + w * mlp + mlp * w)


def tower_attn_flops(t, T):
    return t.layers * 4 * T * T * t.width


def arch_flops(arch):
    g = arch.image_size // arch.patch
    Ti, Tt = g * g + 1, arch.context_length
    img_gemm = tower_gemm_flops(arch.vision, Ti) + 2 * (g * g) * arch.vision.width * 3 * arch.patch ** 2
    txt_gemm = tower_gemm_flops(arch.text, Tt)
    img = img_gemm + tower_attn_flops(arch.vision, Ti) + 2 * arch.vision.width * arch.embed_dim
    txt = txt_gemm + tower_attn_flops(arch.text, Tt) + 2 * arch.text.width * arch.embed_dim
    return {"image": img, "text": txt, "pair": img + txt, "image_gemm": img_gemm, "text_gemm": txt_gemm}


# ---- clocks sampling ----------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        load = sorted(s for s, p in zip(sm, power) if p > 0.5 * max(power)) or sorted(sm)
        return {"sm_mhz": load[len(load) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power)}


# ---- CPU baselines: the oracle ports on the host cores, bounded samples ---------------------------------
def cpu_embed_sample(arch_name, n_pairs, threads, budget_s=45.0, chunk=16):
    """fp32 oracle (oracle/clip_ref.py) on `n_pairs` image+text pairs in chunks, stopping at the time budget."""
    import torch
    from oracle import clip_ref

    torch.set_num_threads(threads)
    cfg = clip_ref.CONFIGS[arch_name]
    sd = clip_ref.make_state_dict(cfg, seed=0)
    px = clip_ref.synth_images(n_pairs, cfg, seed=3)
    tk = clip_ref.synth_tokens(n_pairs, cfg, seed=3)
    clip_ref.mapper_image(sd, cfg, px[:2]); clip_ref.mapper_text(sd, cfg, tk[:2])  # warm-up (thread pool, allocator)
    done, t0 = 0, time.perf_counter()
    while done < n_pairs:
        m = min(chunk, n_pairs - done)
        clip_ref.mapper_image(sd, cfg, px[done:done + m])
        clip_ref.mapper_text(sd, cfg, tk[done:done + m])
        done += m
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return done / dt, done, dt


def cpu_baseline_embed(arch_name, n_pairs, budget_s=45.0):
    cores = physical_cores()
    v, done, dt = cpu_embed_sample(arch_name, n_pairs, cores, budget_s)
    return {"value": v, "unit": "pairs/s", "cores": cores, "kind": "port",
            "sample": "%d image+text pairs of %s (chunks of 16), fp32 oracle/clip_ref.py, torch with %d threads (physical cores), %.1f s"
                      % (done, arch_name, cores, dt)}


def cpu_knn_sample(X16, Q32, k, threads=0):
    from oracle import knn_c

    t0 = time.perf_counter()
    D, I, used = knn_c.flat_search(X16, Q32, k, nthreads=threads)
    return time.perf_counter() - t0, used, D, I


def cpu_baseline_knn(rows_gpu, d, nq, k, fetch_rows, Q32, budget_s=15.0):
    """The FAISS SQfp16 scan restated in C (oracle/knn_ref.c, all host threads) on a sample of the SAME index rows
    (copied back from the GPU shard) and the same queries; brute force is linear in N, so the whole-index rate is
    the sample rate scaled by N_sample / N (stated in `sample`)."""
    import numpy as np

    n_cal, q_cal = 50_000, min(nq, 64)
    Xc = fetch_rows(0, n_cal)
    dt, used, _, _ = cpu_knn_sample(Xc, Q32[:q_cal], k)
    rate = n_cal * q_cal / max(dt, 1e-6)                       # row x query products per second
    n_s = int(min(rows_gpu, max(100_000, rate * budget_s / nq)))
    n_s = min(n_s, 4_000_000)
    X = fetch_rows(0, n_s)
    dt, used, D, I = cpu_knn_sample(X, Q32, k)
    qps_sample = nq / dt
    return {"value": qps_sample * n_s / rows_gpu, "unit": "queries/s", "cores": used, "kind": "port",
            "sample": "oracle/knn_ref.c (FAISS SQfp16 inner-product scan restated, %d threads): %d queries x the first %d rows of the "
                      "GPU's own index in %.1f s = %.1f queries/s at N=%d; scaled linearly to N=%d"
                      % (used, nq, n_s, dt, qps_sample, n_s, rows_gpu),
            "sample_rows": n_s, "sample_seconds": dt}, (X, D, I)


# ---- shared context ---------------------------------------------------------------------------------------
class Ctx:
    def __init__(self, args):
        import torch
        import torch.distributed as dist

        self.args = args
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.peaks = load_peaks()
        self.dump_bytes = 0
        import clip_retrieval_b200 as m

        self.m = m

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def max_over_ranks(self, x):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def all_true(self, ok):
        if self.world == 1:
            return bool(ok)
        t = self.torch.tensor([1.0 if ok else 0.0], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
        return bool(t.item() > 0.5)

    def timed(self, fn, reps):
        """ms per call of fn(), CUDA events on the current stream, barrier + sync both sides, max over ranks."""
        torch = self.torch
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1)) / reps

    def sampler(self):
        return ClockSampler(self.local).start() if self.rank == 0 else None

    def keep_outputs(self, workload, **arrays):
        """--dump-outputs: rank 0 writes `arrays` (device tensors or numpy) as DIR/<workload>_<name>.npy."""
        if self.args.dump_outputs and self.rank == 0:
            self.dump_bytes += dump_outputs(self.args.dump_outputs, workload, arrays, DUMP_TOTAL_BYTES - self.dump_bytes)


DUMP_ARRAY_BYTES = 4 << 20     # an array larger than this is cut to a seeded sample of its rows
DUMP_TOTAL_BYTES = 64 << 20    # all arrays of one run, row numbers of the samples included


def dump_outputs(folder, workload, arrays, budget):
    """Writes `arrays` as float32 (ids and other integers as float64) .npy files in `folder`, each within
    DUMP_ARRAY_BYTES and all of them within `budget` bytes; returns the bytes written."""
    import numpy as np

    os.makedirs(folder, exist_ok=True)
    used = 0
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)
        a = np.atleast_1d(a.astype(np.float64 if a.dtype.kind in "iub" or a.dtype == np.float64 else np.float32))
        base = os.path.join(folder, "%s_%s" % (workload, name))
        cap = min(DUMP_ARRAY_BYTES, budget - used) - 2 * 256          # two .npy headers (128 bytes each as numpy writes them)
        if a.nbytes > cap:
            row_bytes = a.nbytes // a.shape[0] + 8                      # + its row number in <name>_rows.npy
            keep = min(a.shape[0], cap // row_bytes)
            if keep < 1:
                raise SystemExit("--dump-outputs: %s_%s does not fit the %d bytes left of the dump" % (workload, name, budget - used))
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))
            a = a[rows]
            np.save(base + "_rows.npy", rows.astype(np.float64))
            used += os.path.getsize(base + "_rows.npy")
        np.save(base + ".npy", a)
        used += os.path.getsize(base + ".npy")
    return used


def synth_tokens(torch, n, arch, gen, lo=3, hi=None):
    hi = hi or (arch.context_length - 2)
    tok = torch.zeros(n, arch.context_length, dtype=torch.int64)
    lens = torch.randint(lo, hi, (n,), generator=gen)
    for i in range(n):
        L = int(lens[i])
        tok[i, 0] = arch.vocab_size - 2
        tok[i, 1:1 + L] = torch.randint(1, arch.vocab_size - 2, (L,), generator=gen)
        tok[i, 1 + L] = arch.vocab_size - 1
    return tok


# ---- configs[1]: ViT-L/14 embed ----------------------------------------------------------------------------
def wl_vitl14(ctx):
    torch, m, args = ctx.torch, ctx.m, ctx.args
    arch_name = "ViT-L/14"
    arch = m.ARCHS[arch_name]
    fl = arch_flops(arch)
    B, K, W = args.batch, args.steps, max(args.warmup, 3)
    model = m.B200Clip(arch, device=ctx.local, max_batch=B)
    sd = m.synthetic_state_dict(arch, seed=0)
    model.load_state_dict(sd)
    g = torch.Generator().manual_seed(1000 + ctx.rank)
    px_host = torch.randn(B, 3, arch.image_size, arch.image_size, generator=g).clamp_(-1.80, 2.15).pin_memory()
    tok_host = synth_tokens(torch, B, arch, g).pin_memory()
    px_dev, tok_dev = px_host.to(ctx.dev), tok_host.to(ctx.dev)

    last = [None]

    def step_device():
        last[0] = (model.embed_image_device(px_dev), model.embed_text_device(tok_dev))

    for _ in range(W):
        step_device()
    sampler = ctx.sampler()
    launches0 = m.launch_count()
    ms_per_step = ctx.timed(step_device, K)                  # the timed region: no per-kernel events inside
    launches = m.launch_count() - launches0
    ctx.keep_outputs("vitl14", image_embs=last[0][0], text_embs=last[0][1])
    last[0] = None
    # per-kernel-class device time: a second pass of the same K steps with CUDA events around every kernel
    model.set_profiling(True)
    for _ in range(K):
        step_device()
    torch.cuda.synchronize(ctx.dev)
    tm = model.last_timing()
    model.set_profiling(False)
    gemm_ms, attn_ms, ln_ms, other_ms = tm["gemm"] / K, tm["attention"] / K, tm["layernorm"] / K, tm["other"] / K
    gemm_launches = (arch.vision.layers * 4 + 1) + arch.text.layers * 4

    # e2e through the drop-in mapper contract: pinned host tensors in, numpy fp16 out
    def step_e2e():
        return model.embed_image(px_host), model.embed_text(tok_host)

    for _ in range(2):
        step_e2e()
    ctx.barrier()
    Ke = max(3, min(K, 5))
    t0 = time.perf_counter()
    for _ in range(Ke):
        ei, et = step_e2e()
    torch.cuda.synchronize(ctx.dev)
    e2e_s = ctx.max_over_ranks(time.perf_counter() - t0)
    clocks = sampler.stop() if sampler else None

    # parity of exactly what was timed (batch B, pair GEMMs, pipelined host entry): a handful of samples against the
    # fp32 oracle at the north_star's 1e-3 cosine, and host path == device path
    parity = {"checked": False}
    if not args.no_verify:
        from oracle import clip_ref

        torch.set_num_threads(physical_cores())
        cfg = clip_ref.CONFIGS[arch_name]
        sel = [0, 1, B // 2, B - 1] if B >= 4 else list(range(B))
        ref_i = clip_ref.mapper_image(sd, cfg, px_host[sel])
        ref_t = clip_ref.mapper_text(sd, cfg, tok_host[sel])
        di = model.embed_image_device(px_dev).cpu().numpy()
        dt_ = model.embed_text_device(tok_dev).cpu().numpy()
        import numpy as np

        ci = float((1 - clip_ref.cosine(di[sel], ref_i)).max())
        ct = float((1 - clip_ref.cosine(dt_[sel], ref_t)).max())
        bit_equal = bool(np.array_equal(di, ei) and np.array_equal(dt_, et))
        hd = max(float(np.abs(di.astype(np.float32) - ei.astype(np.float32)).max()), float(np.abs(dt_.astype(np.float32) - et.astype(np.float32)).max()))
        ok = ctx.all_true(ci <= 1e-3 and ct <= 1e-3 and hd <= 2e-3 and bool(np.isfinite(di.astype(np.float32)).all()))
        parity = {"checked": ok, "one_minus_cos_image_max": ci, "one_minus_cos_text_max": ct, "samples": len(sel),
                  "host_entry_vs_device_entry_max_abs_diff": hd, "host_entry_bit_equal_device_entry": bit_equal,
                  "tolerance": 1e-3, "oracle": "oracle/clip_ref.py fp32"}

    value = ctx.world * B / (ms_per_step / 1e3)
    gemm_flops = (fl["image_gemm"] + fl["text_gemm"]) * B
    achieved = gemm_flops / (gemm_ms / 1e3) / 1e12
    peak = ctx.peaks.get("bf16_tflops_sustained", FALLBACK_PEAKS["bf16_tflops_sustained"])
    traffic, traffic_src = load_traffic("gemm_bf16_tcgen05_pair_kernel")
    out = {
        "metric": "ViT-L/14 embeds/s (image+text pairs/s)", "value": value, "unit": "pairs/s", "n_gpus": ctx.world,
        "steps": K, "warmup": W, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": (value / PUBLISHED_VITL14[ctx.world]) if ctx.world in PUBLISHED_VITL14 else None,
        "baseline_note": "BASELINE.md: reference ViT-L/14 embed throughput 312 sample/s on 1 A100, 2500 on 8 "
                         "(docs/distributed_clip_inference.md:205; its own reader/writer included)",
        "dtype": "bf16 (fp32 accumulate, fp32 LN/softmax/norm; fp16 output)", "data": "synthetic",
        "config": {"workload": "ViT-L/14 image+text inference, synthetic 224^2, batch %d per GPU (BASELINE configs[1])" % B,
                   "global_batch": B * ctx.world, "parallelism": "dp%d (independent replicas, no collective)" % ctx.world,
                   "weights": "seeded random init", "l2": "inputs (616.6 MB/step) larger than L2"},
        "e2e": {"value": ctx.world * B * Ke / e2e_s, "unit": "pairs/s",
                "h2d_bytes_per_step": int(px_host.numel() * 4 + tok_host.numel() * 8),
                "d2h_bytes_per_step": int(ei.nbytes + et.nbytes), "steps": Ke,
                "api": "B200Clip.embed_image/embed_text (what ClipMapper.__call__ runs), pinned host tensors"},
        "gpu_launches": int(launches),
        "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_src,
                     "kernel": "gemm_bf16_tcgen05_pair_kernel (cta_group::2; the few small GEMMs use the single-CTA variant)",
                     "launches_per_step": gemm_launches, "peak_source": "%s bf16_tflops_sustained" % ctx.peaks["_source"],
                     "flops_per_step": gemm_flops, "gemm_ms_per_step": gemm_ms,
                     "timing": "CUDA events around every GEMM launch in a second pass of the same %d steps" % K},
        "breakdown_ms_per_step": {"gemm": gemm_ms, "attention": attn_ms, "layernorm": ln_ms, "other": other_ms,
                                  "gemm_by_kind": {k: v / K for k, v in tm["gemm_by_kind"].items()}},
        "model_flops": {"per_pair": fl["pair"], "mfu_of_step": fl["pair"] * B / (ms_per_step / 1e3) / 1e12 / peak},
        "parity_checked": parity["checked"], "parity": parity,
    }
    if clocks is not None:
        out["clocks"] = clocks
    del model, px_dev, tok_dev
    torch.cuda.empty_cache()
    if ctx.rank == 0 and ctx.world == 1 and not args.no_cpu:
        out["cpu_baseline"] = cpu_baseline_embed(arch_name, args.cpu_sample)
    return out


# ---- configs[2]: brute-force kNN ---------------------------------------------------------------------------
def build_flat(ctx, d, rows, seed=1234):
    m = ctx.m
    lo = ctx.rank * rows
    idx = m.B200FlatIndex(d, device=ctx.local)
    idx.reserve(rows)
    spec = m.SynthSpec(seed=seed)
    step_rows = 8_000_000
    for r0 in range(0, rows, step_rows):
        idx.add_synthetic(min(step_rows, rows - r0), spec, row0=lo + r0)
    idx.id_base = lo
    return idx, lo


def fetch_index_rows(ctx, idx, d):
    """rows [a, b) of a flat shard as host fp16 (device reconstruct -> fp16; exact: the store is fp16)."""
    import numpy as np

    torch = ctx.torch

    def fetch(a, b):
        out = np.empty((b - a, d), dtype=np.float16)
        step = 500_000
        for s in range(a, b, step):
            e = min(b, s + step)
            ids = torch.arange(idx.id_base + s, idx.id_base + e, dtype=torch.int64, device=ctx.dev)
            R = torch.empty((e - s, d), dtype=torch.float32, device=ctx.dev)
            from clip_retrieval_b200._lib import lib, check

            check(lib.b200_index_reconstruct_device(idx._h, ids.data_ptr(), e - s, R.data_ptr(),
                                                    torch.cuda.current_stream(ctx.dev).cuda_stream), "reconstruct")
            out[s - a:e - a] = R.to(torch.float16).cpu().numpy()
        return out

    return fetch


def verify_sharded_merge(ctx, sh, D, I, k):
    """Every rank: merged (D, I) == the oracle's merge of the candidates its all-gather delivered (bit-exact)."""
    import numpy as np
    from oracle import knn_ref

    if ctx.world == 1:
        return True
    Dg, Ig = sh.gathered_candidates()
    Do, Io = knn_ref.merge_shards(Dg, Ig, k)
    return bool(np.array_equal(I.cpu().numpy(), Io) and np.array_equal(D.cpu().numpy(), Do))


def wl_knn(ctx):
    import numpy as np

    torch, m, args = ctx.torch, ctx.m, ctx.args
    from clip_retrieval_b200.index import synth_rows

    d, k, nq = 768, 40, args.knn_nq
    free, _ = torch.cuda.mem_get_info(ctx.dev)
    rows = min(args.knn_rows, int((free - (6 << 30)) // (d * 2)))
    idx, lo = build_flat(ctx, d, rows)
    sh = m.ShardedIndex(idx, device=ctx.dev)
    q = synth_rows(nq, d, m.SynthSpec(seed=4321), dtype="float32", device=ctx.local)
    q1 = q[:1].contiguous()
    Wk, Kk = max(1, min(args.warmup, 2)), args.steps
    for _ in range(Wk):
        sh.search_device(q, k)
    sampler = ctx.sampler()
    launches0 = m.launch_count()
    last = [None]

    def step():
        last[0] = sh.search_device(q, k)

    ms = ctx.timed(step, Kk)
    launches = m.launch_count() - launches0
    ctx.keep_outputs("knn", D=last[0][0], I=last[0][1])
    last[0] = None
    s_ms, s_n = idx.last_scan_ms()
    fallbacks = idx.last_hi_only_fallbacks()
    # serving shape: one query at a time (clip_back.py:362 issues nq=1)
    for _ in range(3):
        sh.search_device(q1, k)
    ms1 = ctx.timed(lambda: sh.search_device(q1, k), 20)
    s1_ms, s1_n = idx.last_scan_ms()
    # e2e: host numpy in/out through the FAISS-style call, warmed, median of 3
    qh = q.cpu().numpy()
    sh.search(qh, k)
    e2e_t = []
    for _ in range(3):
        ctx.barrier()
        t0 = time.perf_counter()
        Dh, Ih = sh.search(qh, k)
        e2e_t.append(ctx.max_over_ranks(time.perf_counter() - t0))
    e2e_s = statistics.median(e2e_t)
    clocks = sampler.stop() if sampler else None

    # ---- parity of the timed result at full size (verdict r01: "the 100M-row results are never verified") ----
    parity = {"checked": False}
    if not args.no_verify:
        from oracle import synth_ref

        D, I = sh.search_device(q, k)
        merge_ok = verify_sharded_merge(ctx, sh, D, I, k)
        Dn, In = D.cpu().numpy(), I.cpu().numpy()
        # (a) scores of the top-5 of 8 queries against float64 products with rows regenerated by the CPU twin
        nv = min(8, nq)
        worst = 0.0
        for qi in range(nv):
            for j in range(5):
                gid = int(In[qi, j])
                row = synth_ref.rows_f16(1, d, gid, seed=1234)[0].astype(np.float64)
                worst = max(worst, abs(float(row @ qh[qi].astype(np.float64)) - float(Dn[qi, j])))
        # (b) the FMA scan of the same shard on the same 8 queries agrees with the tensor-core scan (tie-aware)
        Dl, Il = idx.search_device(q[:nv].contiguous(), k)              # local shard, batched (tensor) path
        idx.set_tensor_scan(False)
        Df, If = idx.search_device(q[:nv].contiguous(), k)              # FMA scan
        idx.set_tensor_scan(True)
        same_ids = float((Il == If).float().mean().item())
        dmax = float((Dl - Df).abs().max().item())
        # (c) the nq=1 serving path equals row 0 of the batch
        D1, I1 = sh.search_device(q1, k)
        one_ok = bool(torch.equal(I1[0], I[0])) or float((D1[0] - D[0]).abs().max().item()) <= TOL
        desc = bool((np.diff(Dn, axis=1) <= 0).all()) and bool((In >= 0).all()) and all(len(set(r.tolist())) == k for r in In[:nv])
        ok = ctx.all_true(merge_ok and worst <= TOL and dmax <= TOL and same_ids >= 0.99 and one_ok and desc)
        parity = {"checked": ok, "sharded_merge_equals_host_merge": merge_ok, "top5_score_err_vs_float64": worst,
                  "fma_vs_tensor_scan_id_agreement": same_ids, "fma_vs_tensor_scan_score_diff": dmax,
                  "nq1_equals_batch_row0": one_ok, "queries_checked": nv, "tolerance": TOL,
                  "hi_only_fallbacks": fallbacks}

    peak_hbm = ctx.peaks.get("hbm_gbs", FALLBACK_PEAKS["hbm_gbs"])
    peak_tc = ctx.peaks.get("bf16_tflops_sustained", FALLBACK_PEAKS["bf16_tflops_sustained"])
    bytes_per_launch = rows * d * 2
    ach1 = bytes_per_launch / (s1_ms / max(s1_n, 1) / 1e3) / 1e9
    flops = 2.0 * rows * d * nq
    ach_tc = flops / (s_ms / 1e3) / 1e12 if s_ms > 0 else 0.0
    traffic, traffic_src = load_traffic("flat_scan_staged_kernel")
    out = {
        "metric": "brute-force kNN queries/s (%d x %d fp16 rows per GPU, %d queries, top-%d)" % (rows, d, nq, k),
        "value": nq / (ms / 1e3), "unit": "queries/s", "n_gpus": ctx.world, "steps": Kk, "warmup": Wk, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16 rows, f32 query, f32 accumulate",
        "data": "synthetic",
        "config": {"workload": "brute-force cosine kNN, %d x %d fp16 rows per GPU (%d GPUs, range-sharded, %d rows in total), "
                               "%d queries, top-%d (BASELINE configs[2])" % (rows, d, ctx.world, rows * ctx.world, nq, k),
                   "l2": "index (%.1f GB per GPU) larger than L2" % (bytes_per_launch / 1e9)},
        "rows_per_gpu": rows, "rows_total": rows * ctx.world, "nq": nq, "k": k,
        "single_query_ms": ms1, "single_query_qps": 1e3 / ms1,
        "e2e": {"value": nq / e2e_s, "unit": "queries/s", "h2d_bytes_per_step": int(qh.nbytes),
                "d2h_bytes_per_step": int(Dh.nbytes + Ih.nbytes), "api": "ShardedIndex.search(numpy) -> (D, I) numpy; median of 3 after a warm call"},
        "gpu_launches": int(launches),
        "roofline": {"bound": "tensor", "achieved": ach_tc, "peak": peak_tc, "unit": "TFLOP/s", "frac": ach_tc / peak_tc,
                     "traffic": None,
                     "kernel": "scan_mma_kernel (tcgen05 cta_group::2; hi-only pass incl. its two sampling passes; re-score/verify/select outside)",
                     "flops_per_step": flops, "scan_ms_per_step": s_ms, "scan_launches_per_step": s_n,
                     "peak_source": "%s bf16_tflops_sustained" % ctx.peaks["_source"],
                     "whole_search_tflops": flops / (ms / 1e3) / 1e12},
        "roofline_nq1": {"bound": "hbm", "achieved": ach1, "peak": peak_hbm, "unit": "GB/s", "frac": ach1 / peak_hbm,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": "flat_scan_staged_kernel<1,3> (nq=1 serving shape, cp.async.bulk ring)",
                         "bytes_per_launch": bytes_per_launch, "peak_source": "%s hbm_gbs" % ctx.peaks["_source"]},
        "parity_checked": parity["checked"], "parity": parity,
    }
    if clocks is not None:
        out["clocks"] = clocks
    if ctx.rank == 0 and ctx.world == 1 and not args.no_cpu:
        cb, (Xs, Dc, Ic) = cpu_baseline_knn(rows, d, nq, k, fetch_index_rows(ctx, idx, d), qh)
        out["cpu_baseline"] = cb
        if not args.no_verify:
            # the CPU port and the GPU agree on the sample it scanned (tie-aware ids): parity at the port's own size
            sub = m.B200FlatIndex(d, device=ctx.local)
            sub.add(torch.from_numpy(Xs).to(ctx.dev))
            Dg, Ig = sub.search(qh[:32], k)
            agree = float((Ig == Ic[:32]).mean())
            out["parity"]["gpu_vs_cpu_port_on_sample"] = {"id_agreement": agree, "score_diff": float(np.abs(Dg - Dc[:32]).max())}
            if agree < 0.99 or float(np.abs(Dg - Dc[:32]).max()) > TOL:
                out["parity_checked"] = False
            del sub
    del sh, idx
    torch.cuda.empty_cache()
    return out


# ---- configs[3]: IVF-Flat, range-sharded ---------------------------------------------------------------------
def build_ivf(ctx, d, rows, nlist, seed=5):
    m = ctx.m
    from clip_retrieval_b200.index import synth_rows

    cent = synth_rows(nlist, d, m.SynthSpec(seed=7), dtype="float32", device=ctx.local).cpu().numpy()  # generating centroids
    idx = m.B200IVFFlatIndex(d, nlist, cent, device=ctx.local)
    lo = ctx.rank * rows
    idx.add_synthetic(rows, m.SynthSpec(seed=seed, clustered=True, centroid_seed=7, nlist=nlist, cw=3, nw=1), row0=lo)
    idx.id_base = lo
    return idx, lo, cent


def ivf_exact_check(ctx, idx, lo, rows, d, nlist, nprobe, qvec, D_row, I_row, k, seed=5):
    """Exactness of ONE query on this rank's shard at full size: recompute the shard's probed lists on the CPU
    (list(row) is a hash of the row id; rows regenerated by the CPU twin) and rank them in float64."""
    import numpy as np
    from oracle import knn_ref, synth_ref

    C16 = synth_ref.centroids_f32(nlist, d, 7).astype(np.float16)
    cs = knn_ref.scores_f64(C16, qvec[None, :])[0]
    order = np.lexsort((np.arange(nlist), -cs))
    probes = order[:nprobe]
    if nprobe < nlist and cs[order[nprobe - 1]] - cs[order[nprobe]] < 1e-5:
        return None, "probe boundary within 1e-5: fp32 and float64 coarse rankings may differ, query skipped", 0
    lists = np.empty(rows, dtype=np.int64)
    step = 10_000_000
    for s in range(0, rows, step):
        e = min(rows, s + step)
        lists[s:e] = synth_ref.list_of_rows(7, np.arange(lo + s, lo + e, dtype=np.uint64), nlist)
    cand = np.nonzero(np.isin(lists, probes))[0]
    del lists
    kw = dict(seed=seed, clustered=True, centroid_seed=7, nlist=nlist, cw=3, nw=1)
    X = np.concatenate([synth_ref.rows_f16(1, d, int(lo + r), **kw) for r in cand]) if len(cand) < 64 else \
        _rows_by_ids(synth_ref, cand + lo, d, kw)
    S = knn_ref.scores_f64(X, qvec[None, :])
    ok, msg, _ = knn_ref.check_topk(D_row[None, :], I_row[None, :], S, k, ids=(cand + lo).astype(np.int64), tol=TOL)
    return ok, msg, int(len(cand))


def _rows_by_ids(synth_ref, ids, d, kw):
    """Synthetic rows for arbitrary (sorted) row ids: generated in runs of consecutive ids."""
    import numpy as np

    out = np.empty((len(ids), d), dtype=np.float16)
    i = 0
    while i < len(ids):
        j = i
        while j + 1 < len(ids) and ids[j + 1] == ids[j] + 1:
            j += 1
        out[i:j + 1] = synth_ref.rows_f16(j + 1 - i, d, int(ids[i]), **kw)
        i = j + 1
    return out


def cpu_baseline_ivf(ctx, d, nq, k, nprobe, rows_gpu, nlist_gpu, budget_rows=3_000_000):
    """oracle/knn_ref.c IVF search (FAISS IndexIVFFlat restated, threads over queries) on a clustered sample with the
    SAME rows per list as the GPU run (so the per-query list-scan work equals the full-size run's); the coarse
    quantiser is proportionally smaller (stated)."""
    import numpy as np
    from oracle import knn_c, synth_ref
    from clip_retrieval_b200.index import synth_rows

    m = ctx.m
    per_list = rows_gpu / nlist_gpu
    n_s = int(min(rows_gpu, budget_rows))
    nlist_s = max(nprobe, int(round(n_s / per_list)))
    kw = dict(seed=5, clustered=True, centroid_seed=7, nlist=nlist_s, cw=3, nw=1)
    X = synth_rows(n_s, d, m.SynthSpec(**kw), dtype="float16", device=ctx.local).cpu().numpy()
    assign = synth_ref.list_of_rows(7, np.arange(n_s, dtype=np.uint64), nlist_s)
    Xl, off, ids = knn_c.ivf_layout(X, assign, nlist_s)
    C16 = synth_rows(nlist_s, d, m.SynthSpec(seed=7), dtype="float32", device=ctx.local).cpu().numpy().astype(np.float16)
    Q = synth_rows(nq, d, m.SynthSpec(seed=77, clustered=True, centroid_seed=7, nlist=nlist_s), dtype="float32", device=ctx.local).cpu().numpy()
    knn_c.ivf_search(Xl, off, ids, C16, Q[:8], k, nprobe)
    t0 = time.perf_counter()
    D, I, used = knn_c.ivf_search(Xl, off, ids, C16, Q, k, nprobe)
    dt = time.perf_counter() - t0
    return {"value": nq / dt, "unit": "queries/s", "cores": used, "kind": "port",
            "sample": "oracle/knn_ref.c IVF-Flat (FAISS IndexIVFFlat inner product restated, %d threads over queries): %d queries, nprobe %d, "
                      "%d clustered rows in %d lists (%.0f rows per list as in the GPU run of %d rows / %d lists; coarse step over %d "
                      "instead of %d centroids), %.2f s" % (used, nq, nprobe, n_s, nlist_s, per_list, rows_gpu, nlist_gpu, nlist_s, nlist_gpu, dt)}


def wl_ivf(ctx, d=768):
    import numpy as np

    torch, m, args = ctx.torch, ctx.m, ctx.args
    from clip_retrieval_b200.index import synth_rows

    k, nq, nlist = 40, args.knn_nq, args.ivf_nlist
    free, _ = torch.cuda.mem_get_info(ctx.dev)
    # the list-ordered store + ids, and transient sort buffers of the build (12 B per row)
    rows = min(args.ivf_rows, int((free - (8 << 30)) // (d * 2 + 16)))
    t_build = time.perf_counter()
    idx, lo, _ = build_ivf(ctx, d, rows, nlist)
    torch.cuda.synchronize(ctx.dev)
    t_build = time.perf_counter() - t_build
    sh = m.ShardedIndex(idx, device=ctx.dev)
    q = synth_rows(nq, d, m.SynthSpec(seed=77, clustered=True, centroid_seed=7, nlist=nlist), dtype="float32", device=ctx.local)
    q1 = q[:1].contiguous()
    qh = q.cpu().numpy()
    peak_hbm = ctx.peaks.get("hbm_gbs", FALLBACK_PEAKS["hbm_gbs"])
    sampler = ctx.sampler()
    per = {}
    launches = 0
    Kk = args.steps
    for nprobe in (16, 64):
        idx.nprobe = nprobe
        for _ in range(2):
            sh.search_device(q, k)
        l0 = m.launch_count()
        last = [None]

        def step():
            last[0] = sh.search_device(q, k)

        ms = ctx.timed(step, Kk)
        launches += m.launch_count() - l0
        ctx.keep_outputs("ivf", **{"nprobe%d_D" % nprobe: last[0][0], "nprobe%d_I" % nprobe: last[0][1]})
        del last
        s_ms, s_n = idx.last_scan_ms()
        for _ in range(3):
            sh.search_device(q1, k)
        ms1 = ctx.timed(lambda: sh.search_device(q1, k), 50)
        s1_ms, s1_n = idx.last_scan_ms()
        bytes_q = nprobe * (rows / nlist) * d * 2
        per[nprobe] = {"qps": nq / (ms / 1e3), "ms_per_step": ms, "single_query_ms": ms1,
                       "list_scan_ms": s_ms, "list_scan_launches": s_n,
                       "list_scan_gbps": bytes_q * nq / (s_ms / 1e3) / 1e9 if s_ms > 0 else 0.0,
                       "single_query_list_scan_gbps": bytes_q / (s1_ms / 1e3) / 1e9 if s1_ms > 0 else 0.0,
                       "bytes_per_query": bytes_q}
    idx.nprobe = 16
    sh.search(qh, k)
    e2e_t = []
    for _ in range(3):
        ctx.barrier()
        t0 = time.perf_counter()
        Dh, Ih = sh.search(qh, k)
        e2e_t.append(ctx.max_over_ranks(time.perf_counter() - t0))
    e2e_s = statistics.median(e2e_t)
    clocks = sampler.stop() if sampler else None

    parity = {"checked": False}
    if not args.no_verify:
        D, I = sh.search_device(q, k)
        merge_ok = verify_sharded_merge(ctx, sh, D, I, k)
        Dl, Il = idx.search_device(q[:4].contiguous(), k)                 # this rank's shard alone
        for qi in range(4):
            ok_q, msg, ncand = ivf_exact_check(ctx, idx, lo, rows, d, nlist, 16, qh[qi], Dl[qi].cpu().numpy(), Il[qi].cpu().numpy(), k)
            if ok_q is not None:
                break
        ok_q = bool(ok_q)
        D1, I1 = sh.search_device(q1, k)
        one_ok = bool(torch.equal(I1[0], I[0]))
        ok = ctx.all_true(merge_ok and ok_q and one_ok)
        parity = {"checked": ok, "sharded_merge_equals_host_merge": merge_ok, "local_shard_exact_vs_float64": ok_q,
                  "float64_check": msg, "probed_rows_rescanned_on_cpu": ncand, "nq1_equals_batch_row0": one_ok, "tolerance": TOL}

    p16 = per[16]
    out = {
        "metric": "IVF-Flat kNN queries/s (nlist %d, nprobe 16, %d x %d fp16 rows per GPU, %d queries, top-%d)" % (nlist, rows, d, nq, k),
        "value": p16["qps"], "unit": "queries/s", "n_gpus": ctx.world, "steps": Kk, "warmup": 2, "ms_per_step": p16["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16 rows, f32 query, f32 accumulate",
        "data": "synthetic (clustered: 65536 generating centroids, rows = normalise(3 c + noise))",
        "config": {"workload": "IVF-Flat cosine kNN, nlist %d, nprobe 16 (and 64), %d x %d fp16 rows per GPU, %d GPUs range-sharded "
                               "(%d rows in total; 1B x 768 fp16 = 1.5 TB does not fit 8 x 180 GB), one all-gather of per-shard top-%d, "
                               "%d queries (BASELINE configs[3])" % (nlist, rows, d, ctx.world, rows * ctx.world, k, nq),
                   "l2": "each query scans its own lists (%.2f MB at nprobe 16); %d queries touch %.1f GB > L2"
                         % (p16["bytes_per_query"] / 1e6, nq, p16["bytes_per_query"] * nq / 1e9),
                   "build_seconds": t_build},
        "rows_per_gpu": rows, "rows_total": rows * ctx.world, "nq": nq, "k": k, "nlist": nlist,
        "nprobe16": p16, "nprobe64": per[64],
        "single_query_ms": p16["single_query_ms"],
        "e2e": {"value": nq / e2e_s, "unit": "queries/s", "h2d_bytes_per_step": int(qh.nbytes),
                "d2h_bytes_per_step": int(Dh.nbytes + Ih.nbytes), "api": "ShardedIndex.search(numpy) -> (D, I) numpy, nprobe 16; median of 3 after a warm call"},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": p16["list_scan_gbps"], "peak": peak_hbm, "unit": "GB/s",
                     "frac": p16["list_scan_gbps"] / peak_hbm, "traffic": None,
                     "kernel": "ivf_scan_kernel (list scan; bytes = nq * nprobe * N/nlist * d * 2)",
                     "bytes_per_step": p16["bytes_per_query"] * nq, "peak_source": "%s hbm_gbs" % ctx.peaks["_source"],
                     "nprobe64_frac": per[64]["list_scan_gbps"] / peak_hbm},
        "parity_checked": parity["checked"], "parity": parity,
    }
    if clocks is not None:
        out["clocks"] = clocks
    if ctx.rank == 0 and ctx.world == 1 and not args.no_cpu:
        out["cpu_baseline"] = cpu_baseline_ivf(ctx, d, nq, k, 16, rows, nlist)
    del sh, idx
    torch.cuda.empty_cache()
    return out


# ---- configs[4]: the clip_back query path ---------------------------------------------------------------------
def wl_e2e(ctx):
    import numpy as np

    torch, m, args = ctx.torch, ctx.m, ctx.args
    arch_name = "open_clip:ViT-H-14"
    arch = m.ARCHS[arch_name]
    d, k, nlist, nprobe = arch.embed_dim, 40, args.ivf_nlist, 16
    model = m.B200Clip(arch, device=ctx.local, max_batch=64)
    sd = m.synthetic_state_dict(arch, seed=0)
    model.load_state_dict(sd)
    free, _ = torch.cuda.mem_get_info(ctx.dev)
    rows = min(args.e2e_rows, int((free - (8 << 30)) // (d * 2 + 16)))
    idx, lo, _ = build_ivf(ctx, d, rows, nlist)
    idx.nprobe = nprobe
    sh = m.ShardedIndex(idx, device=ctx.dev)
    res = m.ClipResource(model, image_index=sh, text_index=sh)
    svc = m.B200KnnService({"bench": res})
    nreq = args.e2e_queries
    g = torch.Generator().manual_seed(99)                        # identical on every rank: queries are replicated
    toks = synth_tokens(torch, nreq, arch, g, lo=3, hi=30)
    toks_dev = toks.to(ctx.dev)

    def one(i):
        return svc.query(text_tokens=toks_dev[i:i + 1], modality="image", num_images=k, num_result_ids=k, deduplicate=False)

    for i in range(10):
        one(i % nreq)
    sampler = ctx.sampler()
    ctx.barrier()
    lat, l0 = [], m.launch_count()
    t_all = time.perf_counter()
    for i in range(nreq):
        t0 = time.perf_counter()
        r = one(i)                                                 # ends with the ids on the host
        lat.append(time.perf_counter() - t0)
    serial_s = ctx.max_over_ranks(time.perf_counter() - t_all)
    launches = m.launch_count() - l0
    lat_ms = np.array(lat) * 1e3
    # device-resident throughput: batches of 64 queries, embed + search, results stay on the device
    last = []

    def step_dev():
        last.clear()
        for s in range(0, nreq - 63, 64):
            qv = model.embed_text_device(toks_dev[s:s + 64], dtype=torch.float32)
            last.append((qv,) + tuple(sh.search_device(qv, k)))
    step_dev()
    nb = len(range(0, nreq - 63, 64)) * 64
    ms_dev = ctx.timed(step_dev, args.steps)
    if last:
        ctx.keep_outputs("e2e", query_embs=torch.cat([x[0] for x in last]), D=torch.cat([x[1] for x in last]),
                         I=torch.cat([x[2] for x in last]))
    last.clear()
    # closed loop through the micro-batching front: `conc` client threads, each waits for its answer before the next
    conc = 64
    mb = m.MicroBatcher(model, sh if ctx.world == 1 else idx, max_batch=64, max_wait_ms=0.3, k=k)
    done = [0]
    lock = threading.Lock()
    per_thread = max(4, nreq // conc * 2)

    def client(c):
        for j in range(per_thread):
            mb.submit(toks[(c * per_thread + j) % nreq]).result(timeout=120)
            with lock:
                done[0] += 1

    if ctx.world == 1:
        ths = [threading.Thread(target=client, args=(c,)) for c in range(conc)]
        t0 = time.perf_counter()
        [t.start() for t in ths]
        [t.join() for t in ths]
        closed_s = time.perf_counter() - t0
        closed_qps, closed_batches = done[0] / closed_s, mb.batches
    else:
        # under torchrun every rank must issue identical collectives, so the threaded front (whose batch boundaries
        # depend on thread timing) is replaced by its body in lock step: 64 host token rows in -> ids on the host
        t0 = time.perf_counter()
        n_closed = 0
        for rep in range(3):
            for s in range(0, nreq - 63, 64):
                qv = model.embed_text_device(toks[s:s + 64].to(ctx.dev, non_blocking=True), dtype=torch.float32)
                Dd, Id = sh.search_device(qv, k)
                Dd.cpu(), Id.cpu()
                n_closed += 64
        closed_s = ctx.max_over_ranks(time.perf_counter() - t0)
        closed_qps, closed_batches = n_closed / closed_s, n_closed // 64
    mb.close()
    clocks = sampler.stop() if sampler else None

    parity = {"checked": False}
    if not args.no_verify:
        from oracle import clip_ref

        torch.set_num_threads(physical_cores())
        cfg = clip_ref.CONFIGS["ViT-H/14"]
        nv = 2
        qd = svc.compute_query_device(res, text_tokens=toks_dev[:nv]).cpu().numpy()
        qo = np.concatenate([clip_ref.query_embedding(sd, cfg, tokens=toks[i:i + 1]) for i in range(nv)])
        cos = float((1 - clip_ref.cosine(qd, qo)).max())
        D, I = sh.search_device(torch.from_numpy(qd).to(ctx.dev), k)
        merge_ok = verify_sharded_merge(ctx, sh, D, I, k)
        Dl, Il = idx.search_device(torch.from_numpy(qd).to(ctx.dev), k)
        for qi in range(nv):
            ok_q, msg, ncand = ivf_exact_check(ctx, idx, lo, rows, d, nlist, nprobe, qd[qi], Dl[qi].cpu().numpy(), Il[qi].cpu().numpy(), k)
            if ok_q is not None:
                break
        ok_q = bool(ok_q)
        ids_api = [x["id"] for x in one(0)]
        api_ok = ids_api == [int(v) for v in I[0].cpu().numpy() if v >= 0]
        ok = ctx.all_true(cos <= 1e-3 and merge_ok and ok_q and api_ok)
        parity = {"checked": ok, "query_embedding_one_minus_cos_vs_fp32_oracle": cos, "sharded_merge_equals_host_merge": merge_ok,
                  "local_shard_exact_vs_float64": ok_q, "float64_check": msg, "probed_rows_rescanned_on_cpu": ncand,
                  "query_api_ids_equal_search_ids": api_ok}

    fl = arch_flops(arch)
    weight_bytes = 2 * (arch.text.layers * (4 * arch.text.width ** 2 + 2 * arch.text.width * arch.text.mlp))
    bytes_q = nprobe * (rows / nlist) * d * 2 + nlist * d * 2
    peak_hbm = ctx.peaks.get("hbm_gbs", FALLBACK_PEAKS["hbm_gbs"])
    floor_ms = (weight_bytes + bytes_q) / (peak_hbm * 1e9) * 1e3
    p50 = float(np.percentile(lat_ms, 50))
    out = {
        "metric": "clip_back query path queries/s (ViT-H/14 text -> embed -> IVF-Flat kNN over %d x %d rows per GPU -> ids)" % (rows, d),
        "value": nb / (ms_dev / 1e3), "unit": "queries/s", "n_gpus": ctx.world, "steps": args.steps, "warmup": 1,
        "ms_per_step": ms_dev, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "baseline_note": "README.md:433-435: reference averages 18.6 ms text embed + 26.7 ms knn on its CPU/A100 setup",
        "dtype": "bf16 text tower (fp32 accumulate), f16 rows / f32 query search", "data": "synthetic",
        "config": {"workload": "end2end clip_back: ViT-H/14 text tower (D=%d) -> normalised fp32 query -> IVF-Flat (nlist %d, nprobe %d) over "
                               "%d x %d fp16 rows per GPU, %d GPUs range-sharded (%d rows in total) -> top-%d ids on the host "
                               "(BASELINE configs[4]); the index dimension follows the model (SURVEY §8a)" %
                               (d, nlist, nprobe, rows, d, ctx.world, rows * ctx.world, k),
                   "value_is": "device-resident batches of 64 queries (embed + sharded search), %d queries per step" % nb},
        "p50_ms": p50, "p99_ms": float(np.percentile(lat_ms, 99)), "mean_ms": float(lat_ms.mean()),
        "serial_qps": nreq / serial_s, "closed_loop": {"concurrency": conc, "qps": closed_qps, "batches": closed_batches,
                                                       "front": "MicroBatcher(max_batch=64, max_wait_ms=0.3)"},
        "e2e": {"value": closed_qps, "unit": "queries/s", "h2d_bytes_per_step": int(64 * arch.context_length * 8),
                "d2h_bytes_per_step": int(64 * k * 12), "p50_ms_single": p50,
                "api": "B200KnnService.query(text_tokens) one at a time (p50/p99) and MicroBatcher.submit() closed loop (value): host tokens in, ids out"},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": (weight_bytes + bytes_q) / (p50 / 1e3) / 1e9, "peak": peak_hbm, "unit": "GB/s",
                     "frac": floor_ms / p50, "traffic": None,
                     "kernel": "one query = text tower at batch 1 (weights read once: %.0f MB) + coarse scan + %d probed lists (%.1f MB)" %
                               (weight_bytes / 1e6, nprobe, bytes_q / 1e6),
                     "floor_ms": floor_ms, "peak_source": "%s hbm_gbs" % ctx.peaks["_source"],
                     "note": "latency-bound path: frac = (bytes that must be read / HBM peak) / measured p50"},
        "parity_checked": parity["checked"], "parity": parity,
    }
    if clocks is not None:
        out["clocks"] = clocks
    if ctx.rank == 0 and ctx.world == 1 and not args.no_cpu:
        out["cpu_baseline"] = cpu_baseline_e2e(ctx, arch, d, k, nprobe, rows, nlist)
    del svc, res, sh, idx, model
    torch.cuda.empty_cache()
    return out


def cpu_baseline_e2e(ctx, arch, d, k, nprobe, rows_gpu, nlist_gpu, nquery=8):
    """One query at a time on the host cores: fp32 oracle text tower (batch 1) + the C IVF port on a sample index with
    the GPU run's rows per list."""
    import numpy as np
    import torch
    from oracle import clip_ref, knn_c, synth_ref
    from clip_retrieval_b200.index import synth_rows

    m = ctx.m
    cores = physical_cores()
    torch.set_num_threads(cores)
    cfg = clip_ref.CONFIGS["ViT-H/14"]
    sd = clip_ref.make_state_dict(cfg, seed=0)
    per_list = rows_gpu / nlist_gpu
    n_s = int(min(rows_gpu, 2_000_000))
    nlist_s = max(nprobe, int(round(n_s / per_list)))
    kw = dict(seed=5, clustered=True, centroid_seed=7, nlist=nlist_s, cw=3, nw=1)
    X = synth_rows(n_s, d, m.SynthSpec(**kw), dtype="float16", device=ctx.local).cpu().numpy()
    assign = synth_ref.list_of_rows(7, np.arange(n_s, dtype=np.uint64), nlist_s)
    Xl, off, ids = knn_c.ivf_layout(X, assign, nlist_s)
    C16 = synth_rows(nlist_s, d, m.SynthSpec(seed=7), dtype="float32", device=ctx.local).cpu().numpy().astype(np.float16)
    toks = clip_ref.synth_tokens(nquery + 1, cfg, seed=5)
    clip_ref.query_embedding(sd, cfg, tokens=toks[:1])
    lat = []
    for i in range(1, nquery + 1):
        t0 = time.perf_counter()
        q = clip_ref.query_embedding(sd, cfg, tokens=toks[i:i + 1])
        knn_c.ivf_search(Xl, off, ids, C16, q, k, nprobe, nthreads=1)
        lat.append(time.perf_counter() - t0)
    p50 = statistics.median(lat)
    return {"value": 1.0 / p50, "unit": "queries/s", "cores": cores, "kind": "port", "p50_ms": p50 * 1e3,
            "sample": "%d single queries: fp32 oracle ViT-H/14 text tower at batch 1 (torch, %d threads) + oracle/knn_ref.c IVF search "
                      "(1 thread, as FAISS runs one query) over %d rows in %d lists (%.0f rows per list as in the GPU run); value = 1 / p50"
                      % (nquery, cores, n_s, nlist_s, per_list)}


# ---- the B200 arm ---------------------------------------------------------------------------------------------
# ---- configs[0]: the clip_inference plumbing (reference reader -> runner -> mapper -> writer) -------------------
# What the original project's FilesReader -> Runner -> NumpyWriter did over make_plumbing_dataset()'s files, recorded by
# tests/golden/make_reference_golden.py: its code cannot be installed offline, so its job is replayed from this record.
RUNNER_TRACE = os.path.join(ROOT, "tests", "golden", "reference_runner_trace.json")


def hashed_tokenizer(texts, context_length=77, vocab=49408):
    """Stands in for the CLIP BPE tokenizer (its vocabulary file cannot be downloaded here): SOT, one hashed id per
    word, EOT (the largest id, which is what the text tower's argmax pooling looks for)."""
    import torch

    out = torch.zeros(len(texts), context_length, dtype=torch.int64)
    for i, t in enumerate(texts):
        ids = [1 + ((sum(w.encode()) * 31 + j) % (vocab - 408)) for j, w in enumerate(t.split())][:context_length - 2]
        out[i, 0] = vocab - 2
        if ids:
            out[i, 1:1 + len(ids)] = torch.tensor(ids, dtype=torch.int64)
        out[i, 1 + len(ids)] = vocab - 1
    return out


def make_plumbing_dataset(folder, n, seed=0):
    """`n` synthetic images (every third exactly 224x224, the rest ragged so Resize/CenterCrop do work) + captions."""
    import numpy as np
    from PIL import Image

    os.makedirs(folder, exist_ok=True)
    rng = np.random.default_rng(seed)
    for i in range(n):
        h, w = (224, 224) if i % 3 == 0 else (200 + i % 150, 260 + (i * 7) % 90)
        Image.fromarray(rng.integers(0, 256, (h, w, 3), dtype=np.uint8)).save(os.path.join(folder, "%04d.png" % i))
        with open(os.path.join(folder, "%04d.txt" % i), "w") as f:
            f.write("a photo of object %d" % i)


def load_runner_trace(n, parts, batch_size):
    with open(RUNNER_TRACE) as f:
        for t in json.load(f):
            if (t["samples"], t["partitions"], t["batch_size"]) == (n, parts, batch_size):
                return t
    raise ValueError("no recorded clip_inference job with %d samples, %d partitions, batch %d in %s"
                     % (n, parts, batch_size, RUNNER_TRACE))


def _batch_fields(batch):
    import torch

    return {k: [str(v.dtype), list(v.shape)] if torch.is_tensor(v) else type(v).__name__ for k, v in sorted(batch.items())}


def run_reference_runner(src, out_root, mapper, preprocess, tokenizer, parts=2, batch_size=32):
    """One clip_inference job as the original project's own FilesReader, Runner and NumpyWriter run it
    (runner.py:17-62), replayed from RUNNER_TRACE over make_plumbing_dataset()'s `NNNN.png` / `NNNN.txt` in `src`:
    the batches its reader yielded (checked field by field: keys, tensor dtypes and shapes, sample files), in the
    order its Runner handed them to the mapper, and the .npy shards its writer left (checked against the recorded
    path, dtype, rows and sample order; the metadata parquet files it also writes are not reproduced).  The original
    keys files by path INCLUDING the extension (reader.py:17-32), so image and caption keys never intersect and a
    folder job is one pass over the images and one over the captions (as its own tests do, test_reader.py:39).
    `mapper(batch, img, txt)` is the ClipMapper-contract callable under test.  Returns seconds inside mapper()."""
    import numpy as np
    import torch
    from PIL import Image

    n = sum(1 for f in os.listdir(src) if f.endswith(".png"))
    trace = load_runner_trace(n, parts, batch_size)
    spent = 0.0
    rows = {}
    for run in trace["runs"]:
        img = run["modality"] == "image"
        embs, samples = [], []
        for b in run["batches"]:
            if img:
                files = [os.path.join(src, f) for f in b["image_filename"]]
                batch = {"image_filename": files, "image_tensor": torch.stack([preprocess(Image.open(f)) for f in files])}
            else:
                texts = []
                for i in b["samples"]:
                    with open(os.path.join(src, "%04d.txt" % i)) as f:
                        texts.append(f.read())
                if texts != b["text"]:
                    raise ValueError("captions in %s differ from the recorded job" % src)
                batch = {"text": texts, "text_tokens": tokenizer(texts)}
            if _batch_fields(batch) != b["fields"]:
                raise ValueError("batch %r differs from the recorded reader batch %r" % (_batch_fields(batch), b["fields"]))
            t0 = time.perf_counter()
            r = mapper(batch, img, not img)
            spent += time.perf_counter() - t0
            embs.append(r["image_embs"] if img else r["text_embs"])
            samples += b["samples"]
        rows[(run["modality"], tuple(samples))] = np.concatenate(embs)
    for f in trace["files"]:
        if not f["path"].endswith(".npy"):
            continue
        a = rows.pop((f["path"].split("/")[0][len("out_"):], tuple(f["samples"])))
        if str(a.dtype) != f["dtype"] or a.shape[0] != f["shape"][0]:
            raise ValueError("shard %s: %s %r, the recorded writer left %s %r" % (f["path"], a.dtype, a.shape, f["dtype"], f["shape"]))
        path = os.path.join(out_root, f["path"])
        os.makedirs(os.path.dirname(path), exist_ok=True)
        np.save(path, a)
    assert not rows, "mapper output not written by the recorded writer: %r" % list(rows)
    return spent


def read_plumbing_output(out_root):
    import numpy as np
    from clip_retrieval_b200.index import list_embedding_shards

    img = [np.load(f) for f in list_embedding_shards(os.path.join(out_root, "out_image", "img_emb"))]
    txt = [np.load(f) for f in list_embedding_shards(os.path.join(out_root, "out_text", "text_emb"))]
    return img, txt


def wl_plumbing(ctx):
    """BASELINE configs[0]: ViT-B/32 clip_inference on 100 synthetic images + captions — the original project's
    reader / runner / writer job (replayed from its record) around the CUDA `ClipMapper`; the CPU arm is the same job
    around the fp32 oracle."""
    import shutil
    import tempfile

    import numpy as np
    import torch

    m = ctx.m
    n, parts, bs = 100, 2, 32
    base = {"metric": "ViT-B/32 clip_inference samples/s (image + caption files -> fp16 .npy shards)", "unit": "samples/s",
            "n_gpus": ctx.world, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "ViT-B/32 clip_inference on %d synthetic images + captions per GPU: the batches and .npy shards of the "
                                   "original project's FilesReader / Runner / NumpyWriter job (tests/golden/reference_runner_trace.json), "
                                   "batch %d, %d output partitions (BASELINE configs[0])" % (n, bs, parts)}}
    tmp = tempfile.mkdtemp(prefix="b200clip_plumbing_%d_" % ctx.rank)
    try:
        src = os.path.join(tmp, "images")
        make_plumbing_dataset(src, n)
        mapper = m.ClipMapper(enable_image=True, enable_text=True, enable_metadata=False, use_mclip=False,
                              clip_model="synthetic:ViT-B/32", use_jit=True, mclip_model="", warmup_batch_size=bs)
        arch = mapper.model.arch
        from clip_retrieval_b200.model import make_preprocess

        preprocess = make_preprocess(arch.image_size)

        def cuda_mapper(batch, img, txt):
            mapper.enable_image, mapper.enable_text = img, txt
            return mapper(batch)

        steps, times, inside = ctx.args.steps, [], []
        launches0 = None
        for it in range(1 + steps):                                      # one warm-up job, then `steps` timed jobs
            out = os.path.join(tmp, "gpu_%d" % it)
            ctx.barrier()
            if it == 1:
                launches0 = m.launch_count()
            t0 = time.perf_counter()
            sec = run_reference_runner(src, out, cuda_mapper, preprocess, hashed_tokenizer, parts, bs)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if it:
                times.append(ctx.max_over_ranks(dt))
                inside.append(sec)
        launches = (m.launch_count() - launches0) // steps
        t_job = statistics.median(times)
        if ctx.args.dump_outputs:
            img_l, txt_l = read_plumbing_output(os.path.join(tmp, "gpu_%d" % steps))
            ctx.keep_outputs("plumbing", image_embs=np.concatenate(img_l), text_embs=np.concatenate(txt_l))
        img_g, txt_g = read_plumbing_output(os.path.join(tmp, "gpu_1"))
        ok_layout = (len(img_g) == parts and len(txt_g) == parts
                     and all(a.dtype == np.float16 and a.shape == (n // parts, arch.embed_dim) for a in img_g + txt_g))
        res = dict(base)
        res.update({"value": ctx.world * n / t_job, "steps": steps, "warmup": 1, "ms_per_step": 1e3 * t_job,
                    "gpu_launches": int(launches),
                    "e2e": {"value": ctx.world * n / t_job, "unit": "samples/s",
                            "h2d_bytes_per_step": n * (3 * arch.image_size ** 2 * 4 + arch.context_length * 8),
                            "d2h_bytes_per_step": 2 * n * arch.embed_dim * 2},
                    "mapper_ms_per_step": 1e3 * statistics.median(inside),
                    "note": "host-bound by design: PNG decode + torchvision Resize/CenterCrop run on one host thread, as in the "
                            "original's DataLoader (num_workers 0); `mapper_ms_per_step` is the part this engine replaces "
                            "(H2D, both towers, normalise, fp16, D2H for %d images and %d captions)" % (n, n)})
        res["roofline"] = None
        if ctx.rank == 0 and not ctx.args.no_cpu:
            from oracle import clip_ref

            cfg = clip_ref.CONFIGS["ViT-B/32"]
            sd = m.synthetic_state_dict(arch, seed=0)
            cores = physical_cores()
            torch.set_num_threads(cores)

            def cpu_mapper(batch, img, txt):
                return {"image_embs": clip_ref.mapper_image(sd, cfg, batch["image_tensor"]) if img else None,
                        "text_embs": clip_ref.mapper_text(sd, cfg, batch["text_tokens"]) if txt else None,
                        "image_filename": batch["image_filename"] if img else None, "text": batch["text"] if txt else None,
                        "metadata": None}

            clip_ref.mapper_image(sd, cfg, clip_ref.synth_images(2, cfg)); clip_ref.mapper_text(sd, cfg, clip_ref.synth_tokens(2, cfg))  # warm-up
            t0 = time.perf_counter()
            sec_cpu = run_reference_runner(src, os.path.join(tmp, "cpu"), cpu_mapper, preprocess, hashed_tokenizer, parts, bs)
            dt_cpu = time.perf_counter() - t0
            res["cpu_baseline"] = {"value": n / dt_cpu, "unit": "samples/s", "cores": cores, "kind": "port",
                                   "mapper_ms_per_step": 1e3 * sec_cpu,
                                   "sample": "the same %d-sample job once, same recorded reader/runner/writer job, mapper = fp32 oracle/clip_ref.py "
                                             "with %d torch threads (the reference's own mapper needs all_clip/open_clip, not installable)"
                                             % (n, cores)}
            img_c, txt_c = read_plumbing_output(os.path.join(tmp, "cpu"))
            worst = 0.0
            for a, b in zip(img_g + txt_g, img_c + txt_c):
                worst = max(worst, float((1 - clip_ref.cosine(a, b)).max()))
            res["parity"] = {"shard_layout_as_reference_writer": bool(ok_layout), "max_1_minus_cos_vs_oracle_job": worst,
                             "embeddings_within_1e-3_cosine": bool(worst <= 1e-3)}
            ok = ok_layout and worst <= 1e-3
        else:
            res["parity"] = {"shard_layout_as_reference_writer": bool(ok_layout)}
            ok = ok_layout
        res["parity_checked"] = ctx.all_true(ok)
        return res
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


WORKLOADS = {"vitl14": wl_vitl14, "knn": wl_knn, "ivf": wl_ivf, "e2e": wl_e2e, "plumbing": wl_plumbing}
NEST_KEY = {"knn": "knn", "ivf": "ivf", "e2e": "e2e_query", "plumbing": "plumbing"}


def run_b200(args):
    ctx = Ctx(args)
    names = ["vitl14", "knn", "ivf", "e2e", "plumbing"] if args.workload == "all" else [args.workload]
    for skip, flag in (("knn", args.no_knn), ("ivf", args.no_ivf), ("e2e", args.no_e2e), ("plumbing", args.no_plumbing)):
        if flag and skip in names and len(names) > 1:
            names.remove(skip)
    results = {}
    for n in names:
        t0 = time.perf_counter()
        results[n] = WORKLOADS[n](ctx)
        results[n]["wall_s"] = time.perf_counter() - t0
    top = results[names[0]]
    for n in names[1:]:
        top[NEST_KEY[n]] = results[n]
    if len(names) > 1:
        top["parity_checked_all"] = all(bool(results[n].get("parity_checked")) for n in names if results[n].get("parity_checked") is not None)
    if ctx.rank == 0:
        emit(top)
    if ctx.world > 1:
        ctx.dist.destroy_process_group()


# ---- the reference arm: the CPU oracle port of the same workload ---------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    K, W = args.steps, 1
    cores = physical_cores()
    n = max(2, min(args.cpu_sample, 64))
    vals = []
    cpu_embed_sample("ViT-L/14", min(4, n), cores, budget_s=20.0)            # warm-up step
    for _ in range(K):
        v, done, dt = cpu_embed_sample("ViT-L/14", n, cores, budget_s=60.0)
        vals.append(v)
    value = statistics.median(vals)
    cb = {"value": value, "unit": "pairs/s", "cores": cores, "kind": "port",
          "sample": "median of %d steps of %d image+text pairs (chunks of 16), fp32 oracle/clip_ref.py, torch %d threads (physical cores); "
                    "per-step pairs/s %s" % (len(vals), n, cores, ["%.2f" % v for v in vals])}
    emit({
        "impl": "reference", "metric": "ViT-L/14 embeds/s (image+text pairs/s)", "value": value, "unit": "pairs/s",
        "n_gpus": world, "steps": len(vals), "warmup": W, "ms_per_step": 1e3 * n / value,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "ViT-L/14 image+text inference, synthetic 224^2, batch %d per GPU (BASELINE configs[1]); each step a bounded "
                               "sample of %d pairs of that workload" % (args.batch, n)},
        "cpu_baseline": cb,
        "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "the reference's own path (all_clip/open_clip) cannot be installed offline; this is the CPU oracle port (oracle/clip_ref.py)",
    })


_REAL_STDOUT = None


def capture_stdout():
    """Library chatter (e.g. the NCCL version banner) must not share stdout with the one JSON line:
    route fd 1 to stderr for the run and keep the real stdout for emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_REAL_STDOUT, line)


def main():
    capture_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="all", choices=["all", "vitl14", "knn", "ivf", "e2e", "plumbing"])
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--cpu-sample", type=int, default=64)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--no-knn", action="store_true")
    ap.add_argument("--no-ivf", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-plumbing", action="store_true")
    ap.add_argument("--knn-rows", type=int, default=100_000_000)
    ap.add_argument("--knn-nq", type=int, default=1000)
    ap.add_argument("--ivf-rows", type=int, default=100_000_000)
    ap.add_argument("--ivf-nlist", type=int, default=65536)
    ap.add_argument("--e2e-rows", type=int, default=75_000_000)
    ap.add_argument("--e2e-queries", type=int, default=256)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs of every workload run as DIR/<workload>_<array>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1 (every workload times exactly --steps steps)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
