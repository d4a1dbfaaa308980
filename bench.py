#!/usr/bin/env python
"""
bench.py -- map_cells_to_space iterations/sec on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3|c2|c4|c5] [--precision bf16|fp32] [--dump-outputs DIR]
    python bench.py --impl reference ...      # the reference's own CPU path (unmodified Mapper from oracle/_ref), full size

A "step" is one optimizer iteration (loss, backward, Adam) of the hot path on synthetic
expression-like inputs (SURVEY.md 8(d)).  N>1: launched by torchrun, one rank per GPU, the
cells axis sharded (strong scaling: the total problem is fixed), one NCCL all-reduce per step issued by the library itself
(tgb200_comm_init_rank + tgb200_run).
Prints ONE JSON line on rank 0.
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

WORKLOADS = {
    # name: (cells, voxels, genes, types, clusters-mode, description)
    "c1": (26_431, 9_852, 249, 0, False,
           "reference fixtures data/test_ad_sc.h5ad x data/test_ad_sp.h5ad (tests/golden/c1_reference.npz), mode=cells"),
    "c2": (10_000, 1_000, 1_000, 0, False, "synthetic 10k cells x 1k voxels x 1k genes, mode=cells"),
    "c3": (100_000, 10_000, 2_000, 0, False, "synthetic 100k cells x 10k voxels x 2k genes, mode=cells"),
    "c4": (256, 50_000, 5_000, 0, True, "synthetic 256 clusters x 50k voxels x 5k genes, mode=clusters"),
    "c5": (50_000, 5_000, 2_000, 32, False,
           "synthetic 50k cells x 5k voxels x 2k genes, neighbourhood + ct-islands + Getis-Ord on"),
    "tiny": (300, 80, 50, 0, False, "synthetic 300 cells x 80 voxels x 50 genes (smoke test of the bench arms themselves)"),
}
C5_LAMBDAS = dict(lambda_neighborhood_g1=0.96, lambda_ct_islands=0.17, lambda_getis_ord=0.71,
                  lambda_r=2.95e-9, lambda_l2=1e-18)
L2_BYTES = 126e6


def shard_rows_for(n_cells, rank, world):
    from tangram_b200.sharded import shard_rows
    return shard_rows(n_cells, rank, world)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return dict(hbm=j["hbm_gbs"], tf_burst=j["bf16_tflops"], tf_sust=j.get("bf16_tflops_sustained", j["bf16_tflops"]),
                    src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback (B200_PROFILING.md)")


def gen_inputs(name, r0, r1, seed=0):
    """Rows [r0, r1) of the synthetic workload (S rows are generated per block so that ranks agree)."""
    N, V, K, T, clusters, _ = WORKLOADS[name]
    if name == "c1":      # real data: the reference's own test fixtures, exported by tests/golden/make_c1_golden.py
        import scipy.sparse as sp
        z = np.load(os.path.join(ROOT, "tests", "golden", "c1_reference.npz"))
        S = sp.csr_matrix((z["S_data"], z["S_indices"], z["S_indptr"]), shape=tuple(z["S_shape"]))[r0:r1].toarray()
        return dict(S=np.ascontiguousarray(S, dtype=np.float32), G=z["G"], d=z["d"])
    rng = np.random.default_rng(seed)
    G = np.log1p(rng.poisson(2.0, (V, K))).astype(np.float32)
    G[:, ~G.any(axis=0)] = 1.0
    out = dict(G=G)
    if clusters:
        w = np.random.default_rng(seed + 1).random(N) + 0.1
        out["d_source"] = (w / w.sum()).astype(np.float32)[r0:r1]
        out["d"] = (np.ones(V) / V).astype(np.float32)
    else:
        out["d"] = (G.sum(axis=1) / G.sum()).astype(np.float32)
    S = np.empty((r1 - r0, K), dtype=np.float32)
    blk = 4096
    for b0 in range((r0 // blk) * blk, r1, blk):
        rb = np.random.default_rng([seed, 7, b0])
        rows = np.log1p(rb.poisson(0.6, (blk, K))).astype(np.float32)
        lo, hi = max(b0, r0), min(b0 + blk, r1)
        S[lo - r0:hi - r0] = rows[lo - b0:hi - b0]
    S[0, ~S.any(axis=0)] = 1.0
    out["S"] = S
    if T:
        lab = np.random.default_rng(seed + 2).integers(0, T, N)[r0:r1]
        E = np.zeros((r1 - r0, T), dtype=np.float32)
        E[np.arange(r1 - r0), lab] = 1.0
        out["ct_encode"] = E
    return out


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        self.gpu, self.rows, self.proc = gpu, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) < 9:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def host_threads():
    """Threads for the reference's CPU path: the physical cores (os.cpu_count() counts hyper-threads).  Set explicitly so
    that torchrun's OMP_NUM_THREADS=1 cannot change it."""
    return max(1, (os.cpu_count() or 2) // 2)


def mem_available_gb():
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable"):
                return int(line.split()[1]) / 1e6
    except OSError:
        pass
    return 0.0


def reference_present():
    """The reference legs need the unmodified reference Mapper that build() copies into oracle/_ref where the reference
    tree exists; without it they are reported as not measured."""
    from oracle import build_ref
    return os.path.exists(build_ref.REF_DST) or os.path.exists(build_ref.REF_SRC)


def dump_outputs(out_dir, eng, n_rows, n_voxels, hist, budget=64_000_000):
    """What the timed path computed, as .npy files for comparing two builds output for output: one float32 file per loss
    term a Mapper.train caller receives (total_loss.npy, main_loss.npy, ...), one value per timed step, and softmax(M) after
    the last timed step (mapping.npy, float32).  A term whose lambda is 0 is NaN by the reference's convention (x / lambda)
    and is not written.  When the whole mapping does not fit the budget it is a fixed seeded sample of rows, sorted,
    listed in mapping_rows.npy (float64)."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    c = eng.cfg
    terms = {"total_loss": 1.0, "main_loss": c.lambda_g1, "vg_reg": c.lambda_g2, "kl_reg": c.lambda_d, "entropy_reg": c.lambda_r}
    losses = {name: np.ascontiguousarray(hist[:, col]) for col, (name, lam) in enumerate(terms.items()) if lam != 0}
    k = int(min(n_rows, (budget - sum(x.nbytes for x in losses.values())) // (4 * n_voxels + 8)))
    rows = np.arange(n_rows) if k == n_rows else np.sort(np.random.default_rng(0).choice(n_rows, k, replace=False))
    P = torch.empty((n_rows, n_voxels), dtype=torch.float32, device="cuda")
    eng.get_mapping(P)
    torch.cuda.synchronize()
    np.save(os.path.join(out_dir, "mapping.npy"), P[torch.from_numpy(rows).cuda()].cpu().numpy())
    del P
    torch.cuda.empty_cache()
    np.save(os.path.join(out_dir, "mapping_rows.npy"), rows.astype(np.float64))
    for name, x in losses.items():
        np.save(os.path.join(out_dir, name + ".npy"), x)


def reference_kwargs(name, inp, device, random_state=42):
    """Constructor keywords of the UNMODIFIED reference Mapper (oracle/_ref/mapping_optimizer.py) for a workload."""
    N, V, K, T, clusters, _ = WORKLOADS[name]
    kw = dict(S=inp["S"], G=inp["G"], d=inp["d"], lambda_d=1.0, device=device, random_state=random_state)
    if clusters:
        kw["d_source"] = inp["d_source"]
    return kw


def reference_cpu_full(name, steps_requested, budget_s=150.0):
    """The reference's own CPU implementation of the path (tangram/mapping_optimizer.py:358-408, autograd + torch.optim.Adam),
    unmodified, on the host cores, at the FULL workload: one warm-up epoch, then as many epochs as fit the time budget
    (at least 2, at most the requested count) in ONE train() call."""
    import torch
    from oracle import build_ref
    threads = host_threads()
    torch.set_num_threads(threads)
    ref = build_ref.load()
    N, V, K, T, clusters, desc = WORKLOADS[name]
    need_gb = 16.0 * N * V * 4 / 1e9 + 8.0 * N * V / 1e9      # ~16 N x V f32 temporaries at the autograd peak + the f64 M0 draw
    note = None
    if mem_available_gb() and mem_available_gb() < need_gb:
        note = f"{name} needs ~{need_gb:.0f} GB of host memory, {mem_available_gb():.0f} GB available: ran c2 at full size instead"
        name = "c2"
        N, V, K, T, clusters, desc = WORKLOADS[name]
    inp = gen_inputs(name, 0, N)
    t0 = time.perf_counter()
    mp = ref.Mapper(**reference_kwargs(name, inp, "cpu"))
    init_s = time.perf_counter() - t0
    t0 = time.perf_counter()
    mp.train(num_epochs=1, learning_rate=0.1, print_each=None)                 # warm-up (allocator, thread pool)
    t1 = time.perf_counter() - t0
    n = int(max(2, min(steps_requested, budget_s // max(t1, 1e-3))))
    t0 = time.perf_counter()
    mp.train(num_epochs=n, learning_rate=0.1, print_each=None)
    dt = time.perf_counter() - t0
    return dict(name=name, steps=n, warmup=1, seconds=dt, init_s=init_s, threads=threads, note=note, desc=desc,
                shape=(N, V, K))


def reference_cpu_sample(name, target_seconds=15.0):
    """cpu_baseline of our own arm: the unmodified reference on a BOUNDED sample of the workload (a row slice of the cells
    axis; the work is linear in cells), timed for a few epochs.  The full-size run is `--impl reference`."""
    import torch
    from oracle import build_ref
    threads = host_threads()
    torch.set_num_threads(threads)
    ref = build_ref.load()
    N, V, K, T, clusters, _ = WORKLOADS[name]
    n_s = int(min(N, max(256, 2.0e7 // V)))            # ~2e7 mapping elements: a few hundred ms per epoch
    inp = gen_inputs(name, 0, n_s)
    kw = reference_kwargs(name, inp, "cpu")
    if clusters:
        kw["d_source"] = inp["d_source"] / inp["d_source"].sum()
    mp = ref.Mapper(**kw)
    mp.train(num_epochs=2, learning_rate=0.1, print_each=None)
    t0 = time.perf_counter()
    mp.train(num_epochs=3, learning_rate=0.1, print_each=None)
    t3 = (time.perf_counter() - t0) / 3
    n = int(max(3, min(200, target_seconds // max(t3, 1e-4))))
    t0 = time.perf_counter()
    mp.train(num_epochs=n, learning_rate=0.1, print_each=None)
    dt = (time.perf_counter() - t0) / n
    return dict(value=1.0 / (dt * N / n_s), unit="iterations/s", cores=threads, kind="reference",
                sample=f"{n} epochs of the unmodified reference Mapper (oracle/_ref, device='cpu', {threads} threads) on "
                       f"cells[0:{n_s}] x {V} voxels x {K} genes: {dt * 1e3:.1f} ms/epoch on the sample; value = that rate "
                       f"scaled by {n_s}/{N} (work is linear in cells).  The full-size measurement is `bench.py --impl reference`.")


def load_traffic():
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of the kernels, from the committed
    `ncu --set full` capture of this round: profiles/traffic.json is written by tools/ncu_traffic.py from the raw csv."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(p))
    except (OSError, ValueError):
        return {}


def expected_losses(key):
    """Loss trajectory of the default run recorded by an earlier single-GPU run (tests/golden/bench_expected.json);
    the seeded inputs and the sharding-independent device RNG make it the same computation at every N."""
    try:
        return json.load(open(os.path.join(ROOT, "tests", "golden", "bench_expected.json"))).get(key)
    except (OSError, ValueError):
        return None


def timed_steps(one_step, barrier, steps, flush_buf):
    """K steps between barrier + synchronize, CUDA events on the launching stream -> seconds."""
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if flush_buf is None:
        barrier()
        e0.record()
        one_step(steps)                   # one tgb200_run(K): what Mapper.train(K) issues
        e1.record()
        barrier()
        return e0.elapsed_time(e1) / 1e3
    elapsed = 0.0       # small state: L2 flush between timed iterations, per-iteration events
    for _ in range(steps):
        flush_buf.zero_()
        barrier()
        e0.record()
        one_step(1)
        e1.record()
        barrier()
        elapsed += e0.elapsed_time(e1) / 1e3
    return elapsed


def rel_fro_gpu(a, b, rows=8192):
    """||a - b|| / ||b|| over row blocks, on the device (a, b: N x V f32 tensors, device or host)."""
    import torch
    num = den = 0.0
    for r in range(0, a.shape[0], rows):
        x = a[r:r + rows].cuda().double()
        y = b[r:r + rows].cuda().double()
        num += float(((x - y) ** 2).sum())
        den += float((y ** 2).sum())
    return (num / max(den, 1e-300)) ** 0.5


def reference_gpu_legs(a, inp, local, engine_factory, n_total):
    """The PyTorch-GPU comparator (SURVEY 8(d)(ii)): the UNMODIFIED reference Mapper with device='cuda' on this B200, and
    -- from the very same initial mapping (the reference's own seed-42 draw, taken from its device tensor) -- our bf16 and
    bf16x3 paths for the same number of epochs: loss-trajectory and final-mapping parity at the benchmark size."""
    import torch
    from oracle import build_ref
    ref = build_ref.load()
    dev = f"cuda:{local}"
    t0 = time.perf_counter()
    rm = ref.Mapper(**reference_kwargs(a.workload, inp, dev))
    torch.cuda.synchronize()
    init_s = time.perf_counter() - t0
    M0 = rm.M.detach().clone()                       # f32 cast of the reference's legacy draw (:150, :155-157)
    ours = {}
    for prec in ("bf16", "bf16x3"):
        eng = engine_factory(prec)
        eng.set_mapping(M0)
        stream = torch.cuda.current_stream().cuda_stream
        n_timed = a.steps if prec == "bf16" else min(a.steps, 10)
        eng.run(n_total - n_timed, 0.1, stream)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        eng.run(n_timed, 0.1, stream)
        e1.record()
        torch.cuda.synchronize()
        out = torch.empty_like(M0)
        eng.get_mapping(out)
        ours[prec] = dict(loss=eng.history()[:n_total, 0].astype(np.float64), out=out.cpu(),
                          ms=e0.elapsed_time(e1) / n_timed, timed=n_timed)
        eng.close()
        del eng, out
    del M0
    torch.cuda.empty_cache()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ref_out, ref_hist = rm.train(num_epochs=n_total, learning_rate=0.1, print_each=None)      # also the warm-up
    torch.cuda.synchronize()
    first_s = time.perf_counter() - t0
    t0 = time.perf_counter()
    rm.train(num_epochs=a.steps, learning_rate=0.1, print_each=None)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    ref_loss = np.array([float(x) for x in ref_hist["total_loss"]], dtype=np.float64)
    ref_out = torch.from_numpy(ref_out)
    parity = {"what": f"{n_total} epochs from the reference's own M0 (random_state=42), identical inputs: ours vs the "
                      f"unmodified reference Mapper(device='cuda') on the same GPU; loss = max_t |ours - ref| / |ref|, "
                      f"mapping = ||softmax(M)_ours - softmax(M)_ref||_F / ||.||_F over all {ref_out.shape[0]} x {ref_out.shape[1]} entries",
              "north_star_bound": 1e-4}
    for prec, o in ours.items():
        parity[prec] = {"loss_traj_max_rel": float(np.max(np.abs(o["loss"] - ref_loss) / np.abs(ref_loss))),
                        "loss_first": float(o["loss"][0]), "loss_last": float(o["loss"][-1]),
                        "mapping_rel_fro": rel_fro_gpu(o["out"], ref_out)}
    parity["reference_loss_first"], parity["reference_loss_last"] = float(ref_loss[0]), float(ref_loss[-1])
    refgpu = {"value": a.steps / dt, "unit": "iterations/s", "ms_per_step": dt / a.steps * 1e3, "steps": a.steps,
              "warmup": n_total, "init_s": init_s, "first_call_s": first_s,
              "what": "unmodified reference Mapper (oracle/_ref/mapping_optimizer.py) with device='cuda': fp32 cuBLAS SGEMM "
                      "(TF32 off), autograd, torch.optim.Adam, per-epoch .tolist() syncs; init_s includes its host-side "
                      "float64 M0 draw", "torch_allow_tf32": bool(torch.backends.cuda.matmul.allow_tf32)}
    x3 = {"value": 1e3 / ours["bf16x3"]["ms"], "unit": "iterations/s", "ms_per_step": ours["bf16x3"]["ms"],
          "steps": ours["bf16x3"]["timed"], "warmup": n_total - ours["bf16x3"]["timed"],
          "what": "the parity-grade mode (3 x bf16 split operands, six partial products) on the same workload, device-timed"}
    del rm
    torch.cuda.empty_cache()
    return refgpu, parity, x3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)     # long enough to sit at the sustained (power-capped) clocks
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("TGB200_WORKLOAD", "c3"), choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default=os.environ.get("TGB200_PRECISION", "bf16"), choices=["bf16", "bf16x3", "fp32"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-refgpu", action="store_true", help="skip the PyTorch-GPU comparator and the parity legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed steps computed to DIR/*.npy (rank 0: its own cells; at most 64 MB)")
    a = ap.parse_args()
    a.warmup = max(a.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    N, V, K, T, clusters, desc = WORKLOADS[a.workload]
    metric = "map_cells_to_space iterations/sec"
    config = {"workload": f"{desc}, lambda_g1=1, lambda_d=1, lr=0.1", "cells": N, "voxels": V, "genes": K,
              "parallelism": f"cells-sharded x{world}" if world > 1 else "single GPU"}

    # ------------------------------------------------------------------ reference arm (the reference's CPU path, unmodified)
    if a.impl == "reference":
        if rank != 0:
            return
        r = reference_cpu_full(a.workload, a.steps)
        Nr, Vr, Kr = r["shape"]
        value = r["steps"] / r["seconds"]
        config = {"workload": f"{r['desc']}, lambda_g1=1, lambda_d=1, lr=0.1", "cells": Nr, "voxels": Vr, "genes": Kr,
                  "parallelism": f"host cores ({r['threads']} threads)"}
        sample = (f"{r['steps']} epochs in one train() call after {r['warmup']} warm-up epoch, full workload "
                  f"({Nr} x {Vr} x {Kr}), unmodified reference Mapper (oracle/_ref/mapping_optimizer.py, device='cpu', "
                  f"torch.set_num_threads({r['threads']}), os.cpu_count()={os.cpu_count()}); {r['seconds']:.1f} s timed, "
                  f"init {r['init_s']:.1f} s; --steps {a.steps} --warmup {a.warmup} were requested and bounded to keep the run within minutes")
        if r["note"]:
            sample += "; " + r["note"]
        cb = dict(value=value, unit="iterations/s", cores=r["threads"], kind="reference", sample=sample)
        line = {"impl": "reference", "metric": metric, "value": value, "unit": "iterations/s", "n_gpus": a.gpus,
                "steps": r["steps"], "warmup": r["warmup"], "steps_requested": a.steps, "warmup_requested": a.warmup,
                "ms_per_step": r["seconds"] / r["steps"] * 1e3, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": cb,
                "e2e": {"value": value, "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------ our arm (B200)
    import torch
    import torch.distributed as dist
    from tangram_b200 import _lib
    from tangram_b200.engine import Engine
    from tangram_b200.mapping_optimizer import Mapper, shard_rows
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    if clusters and world > 1:
        raise SystemExit("clusters mode (c4) does not shard over cells: replicas only (DESIGN.md)")
    r0, r1 = shard_rows(N, rank, world)
    inp = gen_inputs(a.workload, r0, r1)
    lambdas = dict(C5_LAMBDAS) if a.workload == "c5" else {}
    graphs = None
    if a.workload == "c5":
        from oracle.tangram_oracle import grid_graph, spatial_weights_from_graph  # input generator only
        conn, dmat = grid_graph(V)
        graphs = {_lib.GRAPH_VOXEL_WEIGHTS: spatial_weights_from_graph(conn, dmat, True, True),
                  _lib.GRAPH_NEIGHBORHOOD_FILTER: spatial_weights_from_graph(conn, dmat, False, False),
                  _lib.GRAPH_SPATIAL_WEIGHTS: spatial_weights_from_graph(conn, dmat, False, True)}

    def make_engine(precision, rows=(r0, r1), data=inp):
        e = Engine(rows[1] - rows[0], V, K, n_types=T, n_cells_global=N, device=local, precision=precision,
                   density_mode=_lib.DENSITY_SOURCE if clusters else _lib.DENSITY_CELLS, **lambdas)
        e.set_expression(data["S"], data["G"])
        e.set_density(data["d"], data.get("d_source"))
        if graphs:
            for which, g in graphs.items():
                e.set_graph(which, g)
            e.set_ct_encode(data["ct_encode"])
        return e

    eng = make_engine(a.precision)
    SEED = 1234
    eng.init_mapping_normal(SEED, first_row=r0)      # device Philox keyed by the global cell index: same M0 at every N
    stream = torch.cuda.current_stream().cuda_stream
    if world > 1:
        # the library's own NCCL communicator (one per process and group, tgb200_comm_create; torch.distributed only carries
        # the 128-byte id): the per-iteration exchange runs inside tgb200_run.  Created here, before any timed region, like
        # dist.init_process_group -- Mapper(process_group=) in the e2e leg reuses it.
        from tangram_b200.sharded import nccl_comm_for_group
        comm, _, _ = nccl_comm_for_group(dist.group.WORLD, local)
        eng.set_comm(comm, rank, world)

    def one_step(n=1):
        eng.run(n, 0.1, stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    one_step(a.warmup)
    barrier()
    state_bytes = 3.0 * 4 * N * V / world
    flush = state_bytes < 2 * L2_BYTES
    flush_buf = torch.empty(int(3 * L2_BYTES) // 4, dtype=torch.float32, device="cuda") if flush else None
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = eng.kernel_launches()
    elapsed = timed_steps(one_step, barrier, a.steps, flush_buf)
    launches = eng.kernel_launches() - launches0
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([elapsed], device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed = float(t.item())
    value = a.steps / elapsed

    # ---------------- parity of this very run: the loss before the first and the last update against the recorded trajectory
    n_total = a.warmup + a.steps
    hist = eng.history()[:n_total]
    key = f"{a.workload}/{a.precision}/philox{SEED}"
    exp = expected_losses(key)
    parity = {"loss_first": float(hist[0, 0]), "loss_last": float(hist[-1, 0]), "epochs": n_total, "expected_key": key,
              "what": "total loss before update 0 and before the last timed update of THIS run (device history, rank 0); "
                      "expected_* = the same entries of the single-GPU trajectory recorded in tests/golden/bench_expected.json "
                      "(seeded inputs + sharding-independent device RNG: the same computation at every N)"}
    if exp and len(exp["total_loss"]) >= n_total:
        parity["expected_first"], parity["expected_last"] = exp["total_loss"][0], exp["total_loss"][n_total - 1]
        parity["max_abs_diff_vs_expected"] = float(np.max(np.abs(hist[:, 0].astype(np.float64) - np.array(exp["total_loss"][:n_total]))))
    if os.environ.get("TGB200_RECORD_EXPECTED") and rank == 0 and world == 1:
        parity["recorded_trajectory"] = [float(x) for x in hist[:, 0]]
    if a.dump_outputs and rank == 0:      # before the profiled steps below move the mapping on
        dump_outputs(a.dump_outputs, eng, r1 - r0, V, hist[a.warmup:])

    # ---------------- roofline of the dominant kernel, timed live with CUDA events on this stream
    prof = {}
    for _ in range(3):
        if world == 1:
            per_step = {}                        # a kernel launched once per cell chunk: its launches of one step add up
            for name, ms in eng.profile_step(0.1, stream):
                per_step[name] = per_step.get(name, 0.0) + ms
            for name, ms in per_step.items():
                prof.setdefault(name, []).append(ms)
        else:
            break
    roof = None
    pk = peaks()
    if prof:
        avg = {k: float(np.mean(v)) for k, v in prof.items()}
        step_ms = sum(avg.values())
        top = max(avg, key=avg.get)
        Nl = r1 - r0
        sS = 2.0 if a.precision == "bf16" else (6.0 if a.precision == "bf16x3" else 4.0)
        # algorithmic work of each kernel (DESIGN.md section 4): flops, HBM bytes per launch
        pb = {"bf16": 2.0, "bf16x3": 6.0}.get(a.precision, 4.0)          # bytes per element of the stored P
        work = {
            "gemm_fwd": (2.0 * Nl * V * K, pb * Nl * V + sS * Nl * K + 4.0 * V * K),
            "gemm_rowdot": (2.0 * Nl * V * K, pb * Nl * V + sS * Nl * K + sS * V * K),
            "gemm_bwd_adam": (2.0 * Nl * V * K, 24.0 * Nl * V + sS * Nl * K + sS * V * K),
            "gemm_bwd_dp": (2.0 * Nl * V * K, 4.0 * Nl * V + sS * Nl * K + sS * V * K),      # Pt in (2), dq out (2)
            "adam_rows": (0.0, 24.0 * Nl * V),                                               # M, v (f32) + m (bf16) in+out, dq in, Pt out
            "softmax_rows": (0.0, (4.0 + pb) * Nl * V),
            "loss_reduce": (0.0, 4.0 * V * K * (1 + 1)),
            "scale_rows": (0.0, 6.0 * Nl * K),
        }
        known = {k: v for k, v in avg.items() if any(w in k for w in work)}
        if known:
            top = max(known, key=known.get)
        key_k = next((k for k in work if k in top), None)
        traffic = load_traffic().get(f"{a.workload}/{a.precision}", {})
        if key_k:
            fl, by = work[key_k]
            t_s = avg[top] / 1e3
            # bf16x3 issues 6 bf16 MMAs per useful product; fp32 FFMA peak: 148 SM x 128 lanes x 2 x 1.965 GHz
            tf_peak = pk["tf_sust"] if a.precision == "bf16" else (pk["tf_sust"] / 6.0 if a.precision == "bf16x3" else 74.0)
            t_fl = fl / (tf_peak * 1e12) if fl else 0.0
            t_by = by / (pk["hbm"] * 1e9)
            if t_fl >= t_by:
                roof = {"bound": "tensor" if a.precision != "fp32" else "fp32-ffma", "achieved": fl / t_s / 1e12,
                        "peak": tf_peak, "unit": "TFLOP/s"}
            else:
                roof = {"bound": "hbm", "achieved": by / t_s / 1e9, "peak": pk["hbm"], "unit": "GB/s"}
            roof["frac"] = roof["achieved"] / roof["peak"]
            roof.update({"kernel": top, "kernel_ms": avg[top], "share_of_step": avg[top] / step_ms,
                         "traffic": traffic.get(key_k), "traffic_source": "profiles/traffic.json" if traffic.get(key_k) else None,
                         "peak_source": pk["src"], "per_kernel_ms": avg})
            # the contraction kernels against the tensor roofline (explains the step)
            others = {}
            for kname, ms in avg.items():
                kk = next((k for k in ("gemm_fwd", "gemm_rowdot", "gemm_bwd_adam", "gemm_bwd_dp") if k in kname), None)
                if kk and a.precision != "fp32":
                    others[kname] = {"tflops": work[kk][0] / (ms / 1e3) / 1e12,
                                     "frac_of_sustained_bf16_peak": work[kk][0] / (ms / 1e3) / 1e12 / pk["tf_sust"],
                                     "hbm_GBs": work[kk][1] / (ms / 1e3) / 1e9}
            roof["contractions"] = others
        hb, fl_it = eng.algorithmic_cost()
        roof_step = max(hb / (pk["hbm"] * 1e9), fl_it / ({"bf16": pk["tf_sust"], "bf16x3": pk["tf_sust"] / 6.0}.get(a.precision, 74.0) * 1e12))
        if roof is not None:
            roof["step_roofline_frac"] = roof_step / (elapsed / a.steps)
            roof["sum_kernel_ms"] = step_ms
            roof["mts_tflops"] = 2.0 * Nl * V * K / (avg.get(next((k for k in avg if "gemm_fwd" in k), top), 1e9) / 1e3) / 1e12
    eng.close()
    del eng
    torch.cuda.empty_cache()

    # ---------------- e2e: the public Mapper API with HOST buffers (H2D + steps + D2H inside the timed region)
    e2e = None
    if not a.no_e2e:
        Nl = r1 - r0
        M0 = torch.empty((Nl, V), dtype=torch.float32).pin_memory()
        M0.normal_(generator=torch.Generator().manual_seed(99 + rank))
        Sp = torch.from_numpy(inp["S"]).pin_memory()
        kw = dict(S=Sp.numpy(), G=inp["G"], d=inp["d"], lambda_d=1.0, M0=M0.numpy(), precision=a.precision,
                  device=f"cuda:{local}", n_cells_global=N, process_group=(dist.group.WORLD if world > 1 else None))
        if clusters:
            kw["d_source"] = inp["d_source"]
        if graphs:
            kw.update(lambdas, voxel_weights=graphs[0], neighborhood_filter=graphs[1], spatial_weights=graphs[2],
                      ct_encode=inp["ct_encode"])
        # two calls, the faster one is reported (both listed): the first Mapper of a process sometimes pays 0.5-0.7 s of one-off
        # allocation cost in its constructor (seen on some boxes, not others) that a user's second call never sees
        runs = []
        for _ in range(2):
            barrier()
            t0 = time.perf_counter()
            mp = Mapper(**kw)
            torch.cuda.synchronize()
            t_ctor = time.perf_counter() - t0
            out, hist_e = mp.train(a.steps, learning_rate=0.1, print_each=None)
            barrier()
            dt = time.perf_counter() - t0
            tt = torch.tensor([dt, t_ctor], device="cuda")
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            runs.append((float(tt[0].item()), float(tt[1].item())))
            d2h = out.size * 4.0 + a.steps * 16 * 4.0
            mp.release()
            del mp, out
        dt, t_ctor = min(runs)
        h2d = (Sp.numel() + inp["G"].size + inp["d"].size + M0.numel()) * 4.0
        e2e = {"value": a.steps / dt, "unit": "iterations/s", "h2d_bytes_per_step": h2d / a.steps,
               "d2h_bytes_per_step": d2h / a.steps, "runs_s": [round(r[0], 4) for r in runs],
               "what": f"Mapper(S,G,d,M0 in pinned host memory).train({a.steps}): upload + {a.steps} iterations + softmax(M) download; "
                       f"total {dt:.2f} s per rank ({t_ctor:.2f} s create + upload, {dt - t_ctor:.2f} s iterations + download; copies are per "
                       f"call, not per iteration); the faster of two identical calls (runs_s lists both).  The initial mapping is passed in: the "
                       f"reference API's default host-side float64 draw of M0 (mapping_optimizer.py:150) is outside this region "
                       f"(reference_gpu.init_s shows what it costs)"}
        del M0, Sp

    # ---------------- reference legs (rank 0, single GPU): PyTorch-GPU comparator + parity at the benchmark size, CPU sample
    refgpu = x3 = None
    have_ref = reference_present()
    if rank == 0 and world == 1 and not a.no_refgpu and have_ref:
        torch.cuda.empty_cache()
        refgpu, par_ref, x3 = reference_gpu_legs(a, inp, local, make_engine, n_total)
        parity["vs_reference_gpu"] = par_ref
    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu and have_ref:
        cpu = reference_cpu_sample(a.workload)

    if rank == 0:
        line = {"metric": metric, "value": value, "unit": "iterations/s", "n_gpus": world, "steps": a.steps,
                "warmup": a.warmup, "ms_per_step": elapsed / a.steps * 1e3, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None,
                "dtype": {"bf16": "bf16 operands / f32 accumulate+state", "bf16x3": "f32 via 3xbf16 split operands on tensor cores / f32 accumulate+state"}.get(a.precision, "f32"),
                "data": "synthetic", "config": dict(config, precision=a.precision,
                                                    l2="L2 flushed between timed iterations" if flush else "state exceeds L2 (no flush)"),
                "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roof, "cpu_baseline": cpu,
                "collective": ({"name": "ncclAllReduce(sum, f32) of the exchange buffer [Y_ext (voxels x Ke) | 8 row-scalar partials], in place",
                                "bytes_per_step_per_rank": (V * (-(-(K + 2 + T) // 64) * 64) + 8) * 4, "per_step": 1,
                                "issued_by": "tgb200_run on the handle's own stream (communicator from tgb200_comm_create, lent with tgb200_set_comm); the buffer "
                                             "lives in ncclMemAlloc memory registered with the communicator (NVLS in-switch reduction on user buffers)"}
                               if world > 1 else None),
                "parity": parity, "reference_gpu": refgpu,
                "reference_note": None if have_ref else "oracle/_ref/mapping_optimizer.py absent: reference legs not measured",
                "vs_reference_gpu": (value / refgpu["value"]) if refgpu else None, "bf16x3": x3}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
