#!/usr/bin/env python
"""bench.py -- G->R reversal + cosine top-k search throughput (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # our arm (libganrev_cuda.so)
  python bench.py --impl reference --gpus N ...             # CPU arm: the oracle port on host cores
  python bench.py --config 5 ...                            # BASELINE configs[4]: 3x64x64 G/R, d=256 database, k=1024 kmeans
  python bench.py ... --dump-outputs DIR                    # also write the last timed step's outputs as DIR/*.npy

Workload (default, BASELINE.json configs[3] = north_star's target run): `--images` (default 1,000,000) generated 32x32
grayscale faces from 100-dim N(0,1) noise IN TOTAL, sharded by image over the N ranks (STRONG scaling: 125k per GPU at
N = 8), batched G -> R, the recovered vectors stay on the GPU that made them as its database row shard, then a
4096-query cosine top-20 search over the whole recovered set (needles = recovered rows i*244; local top-k per shard, one
NCCL allgather + merge).  One step = one such pass.  `--scaling weak` gives every rank `--images` faces instead.

`value`  : images/s with the noise already resident in HBM (device-timed, CUDA events on the library's stream, max over
           ranks), per-kernel profiling OFF; the per-kernel profile comes from a separate pass of the same step.
`e2e`    : the same through the C ABI with HOST buffers (pinned noise in, recovered vectors and top-k ids/scores out),
           copies inside the timed region.
`verified`: after the timed loops, sampled rows of the LAST step's images / recovered vectors and 4 needles' top-k are
           checked against the CPU oracle (outside the timed region); false -> exit code 1.
Synthetic data, random-init ("heuristic", weight-init.lua) weights.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

C, H, W, ND = 1, 32, 32, 100
Q, TOPK = 4096, 20
PIX_TOL, COS_TOL = 2e-2, 0.999          # north_star's tolerances


def flops_for(Cc, Hh, Ww, nd):
    """Direct-form (algorithmic) FLOPs per image, SURVEY.md 8a/8d: G, R, and the two dominant layers."""
    px = Hh * Ww
    g = 2.0 * (nd * 512 * px / 16 + (px / 4) * 256 * 4608 + px * 128 * 2304 + px * Cc * 1152)
    r = 2.0 * (px * 64 * 9 * Cc + 2 * px * 64 * 576 + (px / 4) * (128 * 576 + 2 * 128 * 1152) + (128 * px / 16) * 512 + 512 * nd)
    direct = {"g_conv1_up": 2.0 * (px / 4) * 256 * 4608, "g_conv2_up": 2.0 * px * 128 * 2304}
    return g, r, direct


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1353.9), d.get("hbm_gbs", 6552.0), "measured (MEASURED_PEAKS.json, sustained bf16)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region."""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines, self.t_mark = gpu_index, None, [], None

    def mark(self):
        """The timed region starts now: only samples that arrive from here on are reported (nvidia-smi takes ~1 s to
        deliver its first line, so it is started before the warm-up; a timed region shorter than the sampling period
        -- 1M faces over 8 GPUs is 0.3 s -- falls back to the warm-up + timed window and says so)."""
        self.t_mark = time.time()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        timed_only = [ln for t, ln in self.lines if self.t_mark is not None and t >= self.t_mark]
        window = "timed region" if len(timed_only) >= 2 else "warm-up + timed region (timed region shorter than two sampling periods)"
        for ln in (timed_only if len(timed_only) >= 2 else [ln for _, ln in self.lines]):
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window}


# ------------------------------------------------------------------------------------------------ CPU legs
def cpu_port(n_img, n_db, n_q, threads=None, geom=None, topk=TOPK):
    """Time the CPU oracle (kind 'port') on a bounded sample: G->R over n_img faces, then n_q
    queries top-k over n_db recovered rows.  Returns (images/s, queries/s, cores, description, t_gr, t_s)."""
    from oracle import oracle as orc
    from __graft_entry__ import load_package
    pkg = load_package()
    Cc, Hh, Ww, nd = geom or (C, H, W, ND)
    orc.set_num_threads(threads or host_threads())     # explicit: torchrun exports OMP_NUM_THREADS=1
    cores = orc.num_threads()
    gb = pkg.weights.init_G(Cc, Hh, Ww, nd, seed=1)
    rb = pkg.weights.init_R(Cc, Hh, Ww, nd, seed=2)
    noise = np.random.default_rng(7).normal(size=(n_img, nd)).astype(np.float32)
    orc.forward_G(gb, Cc, Hh, Ww, nd, noise[:cores])           # warm the threads / caches
    t0 = time.perf_counter()
    img = orc.forward_G(gb, Cc, Hh, Ww, nd, noise)
    att = orc.forward_R(rb, Cc, Hh, Ww, nd, img)
    t_gr = time.perf_counter() - t0
    db = np.random.default_rng(8).normal(size=(n_db, nd)).astype(np.float32)
    db[: min(n_img, n_db)] = att[: min(n_img, n_db)]
    qs = db[np.arange(n_q) * max(1, n_db // n_q)]
    t0 = time.perf_counter()
    orc.search_cosine(db, qs, topk)
    t_s = time.perf_counter() - t0
    sample = (f"G->R over {n_img} {Cc}x{Hh}x{Ww} faces ({t_gr:.1f} s) + {n_q}-query top-{topk} over {n_db} x {nd} rows ({t_s:.1f} s), "
              f"oracle C port, OpenMP {cores} threads")
    return n_img / t_gr, n_q / t_s, cores, sample, t_gr, t_s


def cpu_torch(n_img, geom=None, batch=32, threads=8):
    """B-torchcpu (BASELINE.md section 3): the same G3 / R graphs in PyTorch-CPU -- the living descendant of Torch7's
    TH/THNN -- at apply_r.lua's own batch size 32 and 8 threads (apply_r.lua:14, 17).  A labelled stand-in: Torch7 cannot run."""
    import torch
    from oracle import torch_cpu
    from __graft_entry__ import load_package
    pkg = load_package()
    Cc, Hh, Ww, nd = geom or (C, H, W, ND)
    old = torch.get_num_threads()
    torch.set_num_threads(threads)
    try:
        gp = pkg.weights.unpack(pkg.weights.init_G(Cc, Hh, Ww, nd, seed=1), pkg.weights.g_layout(Cc, Hh, Ww, nd))
        rp = pkg.weights.unpack(pkg.weights.init_R(Cc, Hh, Ww, nd, seed=2), pkg.weights.r_layout(Cc, Hh, Ww, nd))
        G, R = torch_cpu.TorchG(gp, Cc, Hh, Ww, nd), torch_cpu.TorchR(rp, Cc, Hh, Ww, nd)
        noise = torch.from_numpy(np.random.default_rng(7).normal(size=(n_img, nd)).astype(np.float32))
        R(G(noise[:batch]))                                     # warm-up
        t0 = time.perf_counter()
        for lo in range(0, n_img, batch):                       # NN_UTILS.forwardBatched, nn_utils.lua:5-33
            R(G(noise[lo:lo + batch]))
        dt = time.perf_counter() - t0
    finally:
        torch.set_num_threads(old)
    return {"value": n_img / dt, "unit": "images/s", "cores": threads, "kind": "port",
            "sample": f"PyTorch-CPU {torch.__version__} stand-in for Torch7 nn: G->R over {n_img} faces in batches of {batch}, {threads} threads ({dt:.1f} s)"}


def run_reference(args, world, rank, geom, workload_name):
    """--impl reference: the reference's CPU implementation of the path on host cores.  Torch7
    cannot run here (no lua/luajit/th, un-vendored rocks), so this is the oracle port, on every host thread."""
    if rank != 0:
        return
    n_img, n_db, n_q = args.ref_images, 20000, 64
    vals, qps = [], []
    cores, sample = 0, ""
    for i in range(args.warmup + args.steps):
        if i < args.warmup and i > 0:
            continue                                   # one untimed pass warms caches and threads; the port has no other state
        ips, q, cores, sample, t_gr, t_s = cpu_port(n_img, n_db, n_q, geom=geom)
        if i >= args.warmup:
            vals.append(ips); qps.append(q)
    v = float(np.mean(vals))
    line = {
        "impl": "reference", "metric": "g2r_images_per_sec", "value": v, "unit": "images/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * n_img / v, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name, "images_per_step_sample": n_img,
                   "note": "CPU arm: bounded sample of the same per-image work on all host threads; Torch7 itself cannot run here"},
        "search_queries_per_sec": float(np.mean(qps)),
        "cpu_baseline": {"value": v, "unit": "images/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ side measurements
def hbm_kernels(ctx, pkg, peak_gbs):
    """Bandwidth rooflines of the HBM-bound kernels of the path (north_star: L2, kmeans, small-Q search), each on
    inputs larger than L2, timed with CUDA events on the library stream (ganrev_profile_*)."""
    out = {}
    rng = np.random.default_rng(11)

    def timed(name, fn, alg_bytes, reps):
        fn()                                                       # warm-up
        ctx.profile_reset(); ctx.profile_enable(True)
        for _ in range(reps):
            fn()
        ctx.profile_enable(False)
        e = ctx.profile()[name]
        ms = e["ms"] / max(e["launches"], 1)
        gbs = alg_bytes / (ms * 1e-3) * 1e-9
        return {"bound": "hbm", "achieved": gbs, "peak": peak_gbs, "unit": "GB/s", "frac": gbs / peak_gbs, "ms_per_launch": ms}

    # torch.dist over 200k pairs of 32x32 faces (apply_r.lua:366): 8*C*H*W algorithmic bytes per pair
    n = 200_000
    a = rng.random((n, 1024), dtype=np.float32)
    b = a[::-1].copy()
    out["l2_pairs"] = timed("l2_pairs", lambda: ctx.l2(a, b), 8.0 * n * 1024, 2)
    out["l2_pairs"]["workload"] = f"{n} pairs of 32x32 fp32 faces, 8*C*H*W algorithmic bytes per pair"
    # nearest training image by torch.dist for 8 query faces (sample.lua:128-148, SURVEY 8f rank 3): the set is read once
    out["nearest_l2_q8"] = timed("nearest_l2", lambda: ctx.nearest_l2(b[:8], a), 4.0 * n * 1024, 3)   # explicit set: independent of the geometry
    out["nearest_l2_q8"]["workload"] = f"8 query faces against {n} 32x32 fp32 faces, 4*C*H*W algorithmic bytes per set row"
    del a, b
    # kmeans k=20 over 4M x 100 rows (recovered-vector shape): 4*N*d algorithmic bytes per iteration
    N, d, k = 4_000_000, 100, 20
    ctx.db_synthetic(N, d, seed=11)
    init = rng.standard_normal(size=(k, d), dtype=np.float32)
    init /= np.linalg.norm(init, axis=1, keepdims=True)
    out["kmeans_assign_k20"] = timed("kmeans_assign", lambda: ctx.kmeans(k, 2, init, want_labels=False), 4.0 * N * d, 2)
    out["kmeans_assign_k20"]["workload"] = f"k=20 over {N} x {d} fp32 rows, 4*N*d algorithmic bytes per iteration"
    out["assign_cosine_min_k20"] = timed("assign_cosine_min", lambda: ctx.assign_cosine_min(init), 4.0 * N * d, 2)
    out["assign_cosine_min_k20"]["workload"] = f"cosine-min over k=20 centroids, {N} x {d} fp32 rows, 4*N*d algorithmic bytes"
    # cosine top-20 for 4 needles (BASELINE config 1 shape) over the same rows: 4*N*d algorithmic bytes
    rows = np.array([99, 199, 299, 399], np.int64)
    out["search_q4"] = timed("search_scan", lambda: ctx.search_rows(rows, TOPK), 4.0 * N * d, 3)
    out["search_q4"]["workload"] = f"4 needles, top-{TOPK}, over {N} x {d} fp32 rows, 4*N*d algorithmic bytes"
    return out


def train_leg(ctx, pkg, geom, fp32_tf, cpu=True, B=32, steps=20):
    """SURVEY 8f rank 4: one optimisation step of R (train_r.lua:138-170: G forward of the batch, R forward in training mode,
    MSE, backward, L2 penalty, clamp, Adam) at the reference's batch size, timed on the device with the library's CUDA events;
    beside it the same step (without the optimiser) in PyTorch-CPU autograd, the stand-in for Torch7 nn on the host cores."""
    Cc, Hh, Ww, nd = geom
    rng = np.random.default_rng(5)
    rb = pkg.weights.init_R(Cc, Hh, Ww, nd, seed=2)
    ctx.train_R_init(Cc, Hh, Ww, nd, rb)
    noise = rng.standard_normal(size=(B, nd)).astype(np.float32)
    from oracle.torch_cpu import train_masks, train_R_step
    masks = train_masks(rng, B, Cc, Hh, Ww, False)
    for _ in range(3):
        ctx.train_R_step(noise, masks)
    ctx.profile_reset(); ctx.profile_enable(True)
    for _ in range(steps):
        ctx.train_R_step(noise, masks)
    ctx.profile_enable(False)
    pr = ctx.profile()
    ms = pr["train_R_step"]["ms"] / steps
    g_ms = sum(v["ms"] for k, v in pr.items() if k.startswith("g_")) / steps
    r_flops = 3.0 * flops_for(Cc, Hh, Ww, nd)[1] * B                                  # forward + backward-data + backward-weights of every contraction
    tf = r_flops / (ms * 1e-3) * 1e-12
    out = {"batch": B, "ms_per_step": ms, "g_forward_ms": g_ms, "faces_per_sec": B / ((ms + g_ms) * 1e-3), "dtype": "f32",
           "fp32_tflops": tf, "frac_of_fp32_fma_peak": (tf / fp32_tf) if fp32_tf else None,
           "kernels": "fp32 CUDA-core kernels (csrc/train.cuh): conv fwd / dgrad / wgrad, batch-norm statistics, ELU, dropout, Adam"}
    if cpu:
        import torch
        torch.set_num_threads(host_threads())
        images = ctx.forward_G(noise)
        t0 = time.perf_counter()
        for _ in range(3):
            train_R_step(pkg, rb, Cc, Hh, Ww, nd, images, noise, masks, False, False, 0.0, 1e-4, 1.0)
        out["cpu_torch_ms_per_step"] = (time.perf_counter() - t0) / 3 * 1e3
        out["cpu_torch_threads"] = torch.get_num_threads()
    return out


def fp32_peak(ctx):
    """Measured fp32 FMA roof at the clocks this run sees (MEASURED_PEAKS.json has no fp32 figure)."""
    try:
        return ctx.fma_peak()
    except Exception:
        return None


# ------------------------------------------------------------------------------------------------ verification
def merge_topk(lists, k):
    """lists: [(scores [k], ids [k]), ...] -> the k best by (score desc, NaN last, id asc)."""
    sc = np.concatenate([l[0] for l in lists]); ids = np.concatenate([l[1] for l in lists])
    keep = ids >= 0
    sc, ids = sc[keep], ids[keep]
    key = np.where(np.isnan(sc), -np.inf, sc + 0.0)
    order = np.lexsort((ids, -key))[:k]
    return sc[order], ids[order]


def verify(pkg, ctx, td, world, rank, geom, gb, rb, noise, attrs_host, n_local, row0, qrows, ids, scores, topk, n_check=256):
    """Oracle spot-check of the LAST step's outputs, outside any timed region."""
    from oracle import oracle as orc
    orc.set_num_threads(host_threads())
    Cc, Hh, Ww, nd = geom
    res = {}
    blocks = 8
    per = max(1, min(n_check // blocks, n_local // blocks if n_local >= blocks else n_local))
    starts = sorted(set([0, max(0, n_local - per)] + [int(x) for x in np.linspace(0, max(0, n_local - per), blocks)]))
    pix_err, cos_min, rel = 0.0, 1.0, 0.0
    for s in starts:
        img = ctx.buffer_get(pkg._lib.BUF_IMAGES, s, per)
        att = ctx.buffer_get(pkg._lib.BUF_ATTRS0, s, per)
        want_img = orc.forward_G(gb, Cc, Hh, Ww, nd, noise[s:s + per])
        want_att = orc.forward_R(rb, Cc, Hh, Ww, nd, img)
        pix_err = max(pix_err, float(np.abs(img - want_img).max()))
        a, b = att.astype(np.float64), want_att.astype(np.float64)
        cos_min = min(cos_min, float(((a * b).sum(1) / np.sqrt((a * a).sum(1) * (b * b).sum(1) + 1e-300)).min()))
        rel = max(rel, float(np.sqrt(((a - b) ** 2).sum() / max((b ** 2).sum(), 1e-300))))
        if attrs_host is not None:
            res["e2e_attrs_equal_resident"] = bool(res.get("e2e_attrs_equal_resident", True) and np.array_equal(attrs_host[s:s + per], att))
    res.update({"rows_checked": per * len(starts), "pixel_max_abs": pix_err, "attrs_min_cosine": cos_min, "attrs_rel_l2": rel})
    ok = pix_err <= PIX_TOL and cos_min >= COS_TOL and res.get("e2e_attrs_equal_resident", True)
    # top-k of a few needles: oracle over every rank's shard (exact fmaf-chain scores), merged on the host like the NCCL path
    nq = 4
    sel = np.linspace(0, len(qrows) - 1, nq).astype(int)
    local = ctx.buffer_get(pkg._lib.BUF_ATTRS0, 0, n_local) if attrs_host is None else attrs_host
    qv = np.zeros((nq, nd), np.float32)
    for i, qi in enumerate(sel):
        r = int(qrows[qi]) - row0
        if 0 <= r < n_local:
            qv[i] = local[r]
    if world > 1:
        import torch
        t = torch.from_numpy(qv.view(np.uint32).astype(np.int64)).cuda()
        td.all_reduce(t, op=td.ReduceOp.MAX)
        qv = t.cpu().numpy().astype(np.uint32).view(np.float32).reshape(nq, nd)
    l_ids, l_sc = orc.search_cosine(local, qv, topk)
    mine = [(l_sc[i], np.where(l_ids[i] >= 0, l_ids[i] + row0, -1)) for i in range(nq)]
    if world > 1:
        gathered = [None] * world
        td.all_gather_object(gathered, mine)
    else:
        gathered = [mine]
    topk_ok = True
    if rank == 0:
        for i, qi in enumerate(sel):
            w_sc, w_ids = merge_topk([g[i] for g in gathered], topk)
            topk_ok &= bool(np.array_equal(ids[qi][: len(w_ids)], w_ids) and
                            np.array_equal(scores[qi][: len(w_sc)].view(np.uint32), w_sc.astype(np.float32).view(np.uint32)))
    res["topk_needles_checked"] = nq
    res["topk_exact"] = topk_ok
    ok = ok and topk_ok
    if world > 1:
        import torch
        t = torch.tensor([1 if ok else 0], device="cuda")
        td.all_reduce(t, op=td.ReduceOp.MIN)
        ok = bool(t.item())
    return ok, res


DUMP_SEED, DUMP_IMAGE_BYTES = 20240, 32 << 20


def dump_outputs(out_dir, pkg, ctx, n_local, search):
    """--dump-outputs: what the last timed step left for its caller, as .npy files that two builds can be compared by (the
    inputs are seeded, so the same arguments give the same inputs).  The images and recovered vectors stay on the device and
    are 4 GB / 400 MB at the default size, so the same fixed, seeded sample of rows is written from both (at most 32 MB of
    images); the top-k ids and scores of the in-step search (config 4) are written whole, the ids as float64 (exact below
    2^53).  Under torchrun rank 0 writes, and its samples come from its own shard."""
    Cc, Hh, Ww, nd = ctx.geom
    n = min(n_local, DUMP_IMAGE_BYTES // (4 * Cc * Hh * Ww))
    rows = np.sort(np.random.default_rng(DUMP_SEED).choice(n_local, size=n, replace=False))

    def gather(which):
        return np.concatenate([ctx.buffer_get(which, int(r), 1) for r in rows])

    out = {"images_sample": gather(pkg._lib.BUF_IMAGES), "recovered_vectors_sample": gather(pkg._lib.BUF_ATTRS0)}
    if search is not None:
        ids, scores = search
        out["topk_ids"] = ids.astype(np.float64)
        out["topk_scores"] = scores
    assert sum(a.nbytes for a in out.values()) <= 64 << 20
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=4, choices=[4, 5], help="4 = BASELINE configs[3] (default, north_star's target); 5 = configs[4]")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong (default): --images faces IN TOTAL, sharded over the ranks; weak: --images faces per rank")
    ap.add_argument("--images", type=int, default=0, help="faces (default 1,000,000 for config 4, 100,000 for config 5)")
    ap.add_argument("--db-rows", type=int, default=0, help="config 5: synthetic database rows in total (default 1,250,000 x world: the 8-GPU shard of 10M per GPU)")
    ap.add_argument("--chunk", type=int, default=0, help="pipeline chunk (0 = library default)")
    ap.add_argument("--ref-images", type=int, default=0, help="CPU-arm sample size per step (default ~8 s of 16-thread CPU work)")
    ap.add_argument("--cpu-images", type=int, default=0, help="cpu_baseline sample size (default ~10 s of 16-thread CPU work)")
    ap.add_argument("--geom", default="", help="C,H,W,nd override")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-hbm-kernels", action="store_true", help="skip the L2 / kmeans / small-Q search bandwidth rooflines")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write what the last timed step computed to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU arm only")

    global C, H, W, ND, TOPK
    if args.config == 5:
        C, H, W, ND, TOPK = 3, 64, 64, 256, 100
    if args.geom:
        C, H, W, ND = (int(v) for v in args.geom.split(","))
    geom = (C, H, W, ND)
    FLOP_G, FLOP_R, FLOP_DIRECT = flops_for(*geom)
    n_images = args.images or (1_000_000 if args.config == 4 else 100_000)
    args.ref_images = args.ref_images or (1536 if H * W <= 1024 else 384)
    args.cpu_images = args.cpu_images or (2048 if H * W <= 1024 else 512)
    if args.config == 4:
        workload_name = (f"configs[3]: G->R reversal of {C}x{H}x{W} faces (nd={ND}), {n_images} faces "
                         f"{'in total' if args.scaling == 'strong' else 'per GPU'}, + {Q}-query cosine top-{TOPK} over the recovered set")
    else:
        workload_name = (f"configs[4]: G->R reversal of {C}x{H}x{W} faces (nd={ND}), {n_images} faces "
                         f"{'in total' if args.scaling == 'strong' else 'per GPU'}; {Q}-query cosine top-{TOPK} and one kmeans(k=1024) iteration over a synthetic N(0,1) x {ND} database")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, world, rank, geom, workload_name)
        return

    import torch
    import torch.distributed as td
    from __graft_entry__ import load_package
    pkg = load_package()

    torch.cuda.set_device(local_rank)
    if world > 1:
        td.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = pkg.Context(local_rank)
    sharded_parity = None
    if world > 1:
        pkg.dist.init_comm(ctx)
        # warm-up duty: every row-sharded operation against the single-shard oracle, on hardware, before anything is timed
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import multi_gpu_check
        chk = multi_gpu_check.run_checks(pkg, ctx, world, rank)
        t = torch.tensor([1 if all(chk.values()) else 0], device="cuda")
        td.all_reduce(t, op=td.ReduceOp.MIN)
        sharded_parity = {"ok": bool(t.item()), "checks": chk}
    if args.chunk:
        ctx.set_option("chunk", args.chunk)
    if args.scaling == "strong":
        lo, hi = pkg.dist.shard_range(n_images, world, rank)
        N, row0, n_total = hi - lo, lo, n_images
    else:
        N, row0, n_total = n_images, rank * n_images, n_images * world
    gb = pkg.weights.init_G(C, H, W, ND, seed=1)
    rb = pkg.weights.init_R(C, H, W, ND, seed=2)
    ctx.load_G(C, H, W, ND, gb)
    ctx.load_R(0, C, H, W, ND, rb)

    # synthetic inputs: N(0,1) noise (seed 7 + rank), pinned on the host
    noise_t = torch.empty((N, ND), dtype=torch.float32).pin_memory()
    noise = noise_t.numpy()
    rng = np.random.default_rng(7 + rank)
    for lo_ in range(0, N, 1 << 18):
        hi_ = min(N, lo_ + (1 << 18))
        noise[lo_:hi_] = rng.standard_normal(size=(hi_ - lo_, ND), dtype=np.float32)
    attrs_t = torch.empty((N, ND), dtype=torch.float32).pin_memory()
    attrs = attrs_t.numpy()
    # needles = recovered rows i*244 at 1M rows (SURVEY 8d cfg 4), GLOBAL row ids spread over every rank's shard
    qrows64 = (np.arange(1, Q + 1, dtype=np.int64) * max(1, n_total // (Q + 1))).clip(0, n_total - 1)
    search_in_step = args.config == 4

    stream = torch.cuda.ExternalStream(ctx.stream(), device=torch.device("cuda", local_rank))

    def step_resident():
        ctx.forward_G(None, N=N, want_images=False)
        ctx.forward_R(0, None, N=N, want_attrs=False)
        if not search_in_step:
            return None
        ctx.db_set(None, N=N, d=ND)                          # the database IS the recovered vectors where R left them
        return ctx.search_rows(qrows64, TOPK)                 # queries gathered on the device from the database rows

    def step_e2e():
        ctx.forward_G(noise, want_images=False)              # H2D noise
        ctx.forward_R(0, None, N=N, out=attrs)               # D2H recovered vectors
        if not search_in_step:
            return None
        ctx.db_set(None, N=N, d=ND)
        return ctx.search_rows(qrows64, TOPK)                # H2D needle rows, D2H ids + scores

    def barrier():
        if world > 1:
            td.barrier()
        torch.cuda.synchronize()
        ctx.sync()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = ctx.launch_count()
        e0.record(stream)
        out = None
        for _ in range(steps):
            out = fn()
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device="cuda", dtype=torch.float64)
            td.all_reduce(t, op=td.ReduceOp.MAX)
            ms = float(t.item())
        return ms, ctx.launch_count() - l0, out

    ctx.buffer_put(pkg._lib.BUF_NOISE, noise)
    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(args.warmup):
        step_resident()
    barrier()
    sampler.mark()
    ms_res, launches, last_res = timed(step_resident, args.steps)   # headline: per-kernel profiling OFF
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, pkg, ctx, N, last_res)
    # per-kernel profile: the same step, CUDA events around every launch of the library (separate pass)
    prof_steps = max(1, min(args.steps, 3))
    ctx.profile_reset()
    ctx.profile_enable(True)
    ms_prof, _, _ = timed(step_resident, prof_steps)
    ctx.profile_enable(False)
    prof = ctx.profile()
    for _ in range(max(1, args.warmup // 3)):
        step_e2e()
    ms_e2e, _, last = timed(step_e2e, args.steps)

    # kmeans leg (apply_r.lua:198 at this scale): k = 20, 3 iterations over the recovered set, one int64 allreduce per iteration
    kmeans_leg = None
    if args.config == 4:
        ctx.db_set(None, N=N, d=ND)
        init = np.random.default_rng(6).standard_normal(size=(20, ND)).astype(np.float32)
        init /= np.linalg.norm(init, axis=1, keepdims=True)
        ctx.kmeans(20, 1, init, want_labels=False)
        ctx.profile_reset(); ctx.profile_enable(True)
        ms_km, _, _ = timed(lambda: ctx.kmeans(20, 3, init, want_labels=False), 1)
        ctx.profile_enable(False)
        kp = ctx.profile()
        kmeans_leg = {"k": 20, "iters": 3, "rows_total": n_total, "ms_per_iter": ms_km / 3,
                      "assign_ms_per_iter": kp.get("kmeans_assign", {}).get("ms", 0.0) / 3,
                      "allreduce_ms_per_iter": kp.get("nccl_allreduce_centroids", {}).get("ms", 0.0) / 3 if world > 1 else 0.0,
                      "assign_gbs_per_gpu": 4.0 * N * ND / max(kp.get("kmeans_assign", {}).get("ms", 1e9) / 3 * 1e-3, 1e-12) * 1e-9}

    # the same search shape over a WELL-SPREAD database (synthetic N(0,1) rows -- what a trained R recovers, since it regresses
    # N(0,1) noise; also BASELINE configs[4]'s database).  The recovered vectors of the random-init R this benchmark must use are
    # all within 1e-5 cosine of each other, below any approximate filter's resolution, so the in-step search above is answered
    # by the fmaf-chain kernels; this leg shows the tensor-core filter + exact re-score path on the identical shape.
    search_tc_leg = None
    if args.config == 4:
        tc0 = ctx.tc_counters()
        ctx.db_synthetic(N, ND, seed=8, global_row0=row0)
        ctx.search_rows(qrows64, TOPK)
        ctx.profile_reset(); ctx.profile_enable(True)
        ms_tc, _, out_tc = timed(lambda: ctx.search_rows(qrows64, TOPK), 3)
        ctx.profile_enable(False)
        tp = ctx.profile()
        tc1 = ctx.tc_counters()
        search_tc_leg = {"rows_total": n_total, "d": ND, "queries": Q, "top_k": TOPK, "ms_per_search": ms_tc / 3,
                         "queries_per_sec": Q / (ms_tc / 3 * 1e-3), "fp32_tflops_equiv": 2.0 * n_total * Q * ND / (ms_tc / 3 * 1e-3) * 1e-12,
                         "served_by_tensor_core_path": tc1[0] - tc0[0], "fell_back": tc1[1] - tc0[1],
                         "self_first": bool((out_tc[0][:, 0] == qrows64).all()),
                         "kernels_ms_per_search": {n_: round(v["ms"] / 3, 4) for n_, v in tp.items()},
                         "data": "synthetic N(0,1) rows generated on the device (counter-based), needles = database rows"}

    verified, vres = None, None
    if not args.no_verify:
        if search_in_step:
            ids, scores = last
        else:
            ctx.db_set(None, N=N, d=ND)
            ids, scores = ctx.search_rows(qrows64[:64], TOPK)
        verified, vres = verify(pkg, ctx, td, world, rank, geom, gb, rb, noise, attrs, N, row0,
                                qrows64 if search_in_step else qrows64[:64], ids, scores, TOPK)

    cfg5 = None
    if args.config == 5:
        cfg5 = run_config5_db(args, ctx, pkg, td, world, rank, timed)

    if rank != 0:
        ctx.close()
        if world > 1:
            td.destroy_process_group()
        sys.exit(0 if verified in (None, True) else 1)

    total_images = n_total * args.steps
    value = total_images / (ms_res * 1e-3)
    e2e = total_images / (ms_e2e * 1e-3)
    peak_tf, peak_gbs, peak_src = load_peaks()
    # dominant kernel = the conv GEMM with the largest share of device time
    conv_names = [k for k in prof if k.startswith(("g_conv1", "g_conv2", "r_conv", "g_linear", "r_linear"))]
    dom = max(conv_names, key=lambda k: prof[k]["ms"]) if conv_names else None
    roofline = None
    if dom:
        e = prof[dom]
        ms_launch = e["ms"] / max(e["launches"], 1)
        imgs_launch = N * prof_steps / max(e["launches"], 1)
        exec_tf = e["flops"] / max(e["ms"], 1e-9) * 1e-9
        alg = FLOP_DIRECT.get(dom)
        alg_tf = (alg * imgs_launch) / (ms_launch * 1e-3) * 1e-12 if alg else exec_tf
        traffic, traffic_src = None, None
        for rnd in ("r02", "r01"):
            try:
                tj = json.load(open(os.path.join(ROOT, "profiles", rnd, "ncu_traffic.json")))
                if dom in tj and (C, H, W) == (1, 32, 32):
                    traffic = tj[dom]["dram_bytes_per_image"] * imgs_launch
                    traffic_src = f"profiles/{rnd}/ncu_traffic.json (committed ncu --set full capture, dram bytes per image x images per launch)"
                    break
            except Exception:
                pass
        roofline = {"bound": "tensor", "kernel": dom, "achieved": exec_tf, "peak": peak_tf, "unit": "TFLOP/s",
                    "frac": exec_tf / peak_tf, "traffic": traffic, "traffic_source": traffic_src,
                    "achieved_algorithmic": alg_tf, "frac_algorithmic": alg_tf / peak_tf,
                    "note": "achieved / frac = FLOPs the kernel EXECUTES (upsample folded into 4 phase convs = 2.25x fewer MACs than the "
                            "direct form) / CUDA-event time per launch, from the profiled pass; *_algorithmic = the layer's direct-form FLOPs "
                            "(SURVEY 8d) over the same time, not a hardware fraction; peak = " + peak_src,
                    "avg_launch_ms": ms_launch, "images_per_launch": imgs_launch}
    tot_ms = sum(v["ms"] for v in prof.values()) or 1.0
    kernels = {k: {"launches": v["launches"], "ms": round(v["ms"], 3), "share": round(v["ms"] / tot_ms, 4),
                   "tflops_executed": round(v["flops"] / max(v["ms"], 1e-9) * 1e-9, 2),
                   "gbs": round(v["bytes"] / max(v["ms"], 1e-9) * 1e-6, 1)} for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])}
    srch_ms = sum(prof[k]["ms"] for k in prof if k.startswith(("search", "gather_rows", "nccl_allgather_topk", "nccl_allreduce_queries", "vec_prep"))) / prof_steps
    collectives = {k: round(v["ms"] / prof_steps, 4) for k, v in prof.items() if k.startswith("nccl_") or k == "search_merge_global"}
    fp32_tf = fp32_peak(ctx)
    line = {
        "metric": "g2r_images_per_sec", "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_res / args.steps, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": workload_name, "images_total": n_total, "images_per_gpu": N, "queries": Q, "top_k": TOPK, "noise_dim": ND,
                   "weights": "random-init (weight-init.lua heuristic)",
                   "l2_flush": "inputs larger than L2 (activation stream per chunk >> 126 MB)",
                   "arith": "bf16 operands, fp32 accumulate (conv GEMMs); fp32 fmaf chains for every returned score (search)"},
        "algorithmic_tflops": value * (FLOP_G + FLOP_R) * 1e-12,
        "e2e": {"value": e2e, "unit": "images/s", "h2d_bytes_per_step": int(n_total * ND * 4 + (Q * 8 if search_in_step else 0)),
                "d2h_bytes_per_step": int(n_total * ND * 4 + (Q * TOPK * 12 if search_in_step else 0)), "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roofline,
        "verified": verified, "verification": vres,
        "profiled_pass": {"steps": prof_steps, "ms_per_step": ms_prof / prof_steps,
                          "note": "per-kernel CUDA events on; the headline loop ran with them off"},
        "kernels": kernels,
    }
    if search_in_step:
        # the SAME Q queries are answered once per step over the whole (sharded) database: not multiplied by the world size
        line["search_queries_per_sec"] = Q / (srch_ms * 1e-3) if srch_ms > 0 else None
        line["search_ms_per_step"] = srch_ms
        served, fell = ctx.tc_counters()
        line["search_path_in_step"] = ("tensor-core filter + exact re-score" if not any(k.startswith("search_scan") for k in prof) else
                                       "fmaf-chain kernels (the tensor-core filter declined: recovered vectors of a random-init R are packed within its resolution)")
        line["search_fp32_tflops_equiv"] = 2.0 * n_total * Q * ND / (srch_ms * 1e-3) * 1e-12 if srch_ms > 0 else None
    if fp32_tf:
        line["fp32_fma_peak_tflops"] = {"value": fp32_tf, "how": "ganrev_debug_fma_peak: 16 independent fmaf chains per thread on every SM, this run's clocks (builder-side measurement; MEASURED_PEAKS.json has no fp32 figure)"}
    if world > 1:
        line["collectives_ms_per_step"] = collectives
        line["sharded_parity"] = sharded_parity
    if kmeans_leg:
        line["kmeans_leg"] = kmeans_leg
    if search_tc_leg:
        line["search_wellspread_leg"] = search_tc_leg
    if cfg5:
        line["config5"] = cfg5
    if world == 1 and not args.no_hbm_kernels:
        line["hbm_kernels"] = hbm_kernels(ctx, pkg, peak_gbs)
    if world == 1 and not args.no_hbm_kernels:
        try:
            line["train_leg"] = train_leg(ctx, pkg, geom, fp32_tf, cpu=not args.no_cpu_baseline)
        except Exception as ex:
            line["train_leg"] = {"unavailable": repr(ex)[:200]}
    if world == 1 and not args.no_cpu_baseline:
        ips, qps, cores, sample, _, _ = cpu_port(args.cpu_images, 20000, 64, geom=geom)
        line["cpu_baseline"] = {"value": ips, "unit": "images/s", "cores": cores, "kind": "port", "sample": sample,
                                "search_queries_per_sec": qps}
        try:
            line["cpu_baseline_torchcpu"] = cpu_torch(max(64, args.cpu_images // 8), geom=geom)
        except Exception as ex:                                  # the stand-in is optional colour, never a reason to lose the line
            line["cpu_baseline_torchcpu"] = {"unavailable": repr(ex)[:200]}
    print(json.dumps(line))
    ctx.close()
    if world > 1:
        td.destroy_process_group()
    if verified is False or (sharded_parity and not sharded_parity["ok"]):
        sys.exit(1)


def run_config5_db(args, ctx, pkg, td, world, rank, timed):
    """BASELINE configs[4]'s database legs: 4096-query top-100 and one kmeans(k=1024) iteration over a synthetic N(0,1)
    x 256 database generated on the device (SURVEY 8d cfg 5), row-sharded over the ranks."""
    d, k = 256, 1024
    rows_total = args.db_rows or 1_250_000 * world
    lo, hi = pkg.dist.shard_range(rows_total, world, rank)
    ctx.db_synthetic(hi - lo, d, seed=8, global_row0=lo)
    rows = (np.arange(1, Q + 1, dtype=np.int64) * max(1, rows_total // (Q + 1))).clip(0, rows_total - 1)
    ctx.search_rows(rows, 100)                                   # warm-up at the full shape (buffers are sized by Q and k)
    ctx.profile_reset(); ctx.profile_enable(True)
    ms_s, _, out = timed(lambda: ctx.search_rows(rows, 100), 1)
    ctx.profile_enable(False)
    sp = ctx.profile()
    ids, sc = out
    init = np.random.default_rng(10).standard_normal(size=(k, d)).astype(np.float32)
    init /= np.linalg.norm(init, axis=1, keepdims=True)
    ctx.kmeans(k, 1, init, want_labels=False)                    # warm-up at the full shape (work buffers are sized by k and d)
    ctx.profile_reset(); ctx.profile_enable(True)
    ms_k, _, _ = timed(lambda: ctx.kmeans(k, 1, init, want_labels=False), 1)
    ctx.profile_enable(False)
    kp = ctx.profile()
    return {"db_rows_total": rows_total, "db_rows_per_gpu": hi - lo, "d": d,
            "search": {"queries": Q, "top_k": 100, "ms": ms_s, "queries_per_sec": Q / (ms_s * 1e-3),
                       "fp32_tflops_equiv": 2.0 * rows_total * Q * d / (ms_s * 1e-3) * 1e-12,
                       "self_first": bool((ids[:, 0] == rows).all()), "sorted": bool((np.diff(sc, axis=1) <= 0).all()),
                       "kernels": {n: round(v["ms"], 3) for n, v in sp.items()}},
            "kmeans": {"k": k, "ms_per_iter": ms_k, "fp32_tflops_equiv": 2.0 * rows_total * k * d / (ms_k * 1e-3) * 1e-12,
                       "kernels": {n: round(v["ms"], 3) for n, v in kp.items()}},
            "note": "database legs graded against the compute roof (AI ~ Q/2 and k/2 FLOP/B, SURVEY 8d): fp32-equivalent TFLOP/s = 2*N*Q*d / time"}


if __name__ == "__main__":
    main()
