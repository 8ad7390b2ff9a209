#!/usr/bin/env python
"""bench.py — BASELINE.json metric on the BASELINE.json configuration.

Default workload (configs[1]): 1M x 1M symmetric 2048-bit Tanimoto + Butina clustering (similarity >= 0.7, i.e.
distance cutoff 0.3), synthetic clustered fingerprints (20,000 centres x 50 members, seed 20260924), one GPU.
A step = one pass of the hot path over the whole batch: thresholded similarity graph (counts + edge list, every
unordered pair evaluated once) -> CSR -> greedy Butina loop -> cluster ids. `value` = unique pairs / s with the
fingerprints resident in HBM; `e2e` = the same through the public API with HOST buffers (pinned H2D of the fingerprints
and D2H of the ids inside the timed region).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload butina|etkdg_mmff]
                    [--dump-outputs DIR]
    torchrun --nproc-per-node N bench.py --gpus N ...     (one rank per GPU; rank 0 prints the JSON line)

--dump-outputs DIR writes what the last timed step of each leg returned as DIR/<name>.npy (see write_dumps); the inputs
are seeded, so two builds run with the same arguments can be compared output for output.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CUTOFF = 0.3  # similarity threshold 0.7
METRIC_NAME = "tanimoto_pairs_per_s"
UNIT = "pairs/s"


def fp4_possible(words: int) -> bool:
    return (words * 32) % 256 == 0  # the library's eligibility rule for the fp4 count tile (tanimoto_tc.cu)


def unique_pairs(n: int) -> float:
    return n * (n - 1) / 2.0


# ----------------------------------------------------------------------------------------------- helpers
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.gpu)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.splitlines()[0].split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self) -> dict:
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for name, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


DUMP_LIMIT_BYTES = 64 << 20
DUMP_SAMPLE = 1 << 20  # entries of the materialised cross-similarity sampled into the dump
DUMP_CONFORMERS = 4096  # conformer slots whose coordinates are sampled into the dump


def write_dumps(out_dir: str, arrays: dict) -> None:
    """--dump-outputs: one DIR/<name>.npy per array, integer and float32 outputs as float32 (exact below 2^24), float64
    outputs as float64. Large outputs enter as fixed, seeded samples so that the whole dump stays under 64 MB."""
    arrays = {k: np.ascontiguousarray(v, dtype=np.float64 if v.dtype == np.float64 else np.float32) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total / 2**20:.1f} MB of outputs at this size, more than {DUMP_LIMIT_BYTES >> 20} MB")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def measured_peaks() -> tuple[float, str]:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
        except Exception:
            pass
    return 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


# ----------------------------------------------------------------------------------------------- reference arm
def cpu_sample_size(words: int = 64, target_s: float = 10.0) -> tuple[int, float]:
    """Calibrate the oracle on a small set, then size a sample worth ~target_s of CPU work (multiple of 50 rows)."""
    import oracle
    from nvmolkit_b200 import synthetic

    fp = synthetic.clustered_fingerprints(160, 50, seed=synthetic.SEED + 1)
    t0 = time.perf_counter()
    oracle.butina_fp(fp, CUTOFF)
    rate = unique_pairs(len(fp)) / (time.perf_counter() - t0)
    n = int((2.0 * rate * target_s) ** 0.5)
    n = max(2000, min(100_000, n // 50 * 50))
    return n, rate


def run_reference(args) -> None:
    """The reference's CPU implementation of the path, timed on this box's host cores.

    The reference's path is RDKit (BulkTanimotoSimilarity + ML.Cluster.Butina.ClusterData(reordering=True)); RDKit
    cannot be built or imported here, so the arm times the C restatement in oracle/ ("port") with OpenMP on all cores,
    on a bounded sample of the same workload.
    """
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    from nvmolkit_b200 import synthetic

    cores = oracle.set_threads(os.cpu_count() or 1)  # (torchrun exports OMP_NUM_THREADS=1 to its workers)
    n, _ = cpu_sample_size()
    if args.n_centres:
        n = min(n, args.n_centres * 50)
    fp = synthetic.clustered_fingerprints(n // 50, 50, seed=synthetic.SEED)
    for _ in range(args.warmup):
        oracle.butina_fp(fp, CUTOFF)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ids, cen = oracle.butina_fp(fp, CUTOFF)
    dt = (time.perf_counter() - t0) / args.steps
    value = unique_pairs(len(fp)) / dt
    sample = f"{len(fp)} x {len(fp)} clustered 2048-bit fingerprints ({len(fp) // 50} centres x 50), cutoff {CUTOFF}"
    print(json.dumps({
        "impl": "reference", "metric": METRIC_NAME, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "u32 popcount + f64 divide", "data": "synthetic",
        "config": {"workload": "1Mx1M symmetric 2048-bit Tanimoto + Butina (sim>=0.7), CPU on a bounded sample",
                   "sample_rows": len(fp), "cutoff": CUTOFF},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "n_clusters": int(len(cen)),
    }))


# ----------------------------------------------------------------------------------------------- B200 arm
def run_b200(args) -> None:
    import torch
    import torch.distributed as dist

    from nvmolkit_b200 import _lib, synthetic
    from nvmolkit_b200.clustering import fused_butina_device, fused_butina_sharded
    from nvmolkit_b200.distributed import sharded_upload

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: nvmolkit_b200 has no CPU fallback")
    # the conformer pool is generated first: its worker processes are forked before this process touches CUDA / NCCL
    pool = None
    if args.workload in ("all", "conformers") and args.etkdg_mols > 0:
        t_pool = time.perf_counter()
        procs = args.pool_procs or max(1, min(48, (os.cpu_count() or 8) // max(1, world)))
        pool = conformer_pool(min(args.pool, max(args.etkdg_mols, 1)), synthetic.SEED, procs)
        t_pool = time.perf_counter() - t_pool
    torch.cuda.set_device(local)
    _lib.check(_lib.load().b200mol_check_device(local))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    _lib.profile_enable(True)
    if args.tensor_cluster >= 0:
        _lib.set_option("similarity_tensor_cluster", args.tensor_cluster)
    if args.superpose >= 0:
        _lib.set_option("similarity_superpose", args.superpose)
    if args.bfgs_l2_persist:
        _lib.set_option("bfgs_l2_persist", 1)
    if args.superpose_cols >= 0:
        _lib.set_option("similarity_superpose_cols", args.superpose_cols)
    if args.pipeline_chunks >= 0:
        _lib.set_option("similarity_pipeline_chunks", args.pipeline_chunks)
    if args.superpose_auto >= 0:
        _lib.set_option("similarity_superpose_auto", args.superpose_auto)
    dumps = {}
    if args.workload == "conformers":
        legs = run_conformer_legs(args, pool, dev, world, rank, dumps)
        if rank == 0:
            line = dict(legs["etkdg_mmff"])
            line.update({"warmup": 1, "higher_is_better": True, "vs_baseline": None, "data": "synthetic",
                         "config4_mmff": legs.get("config4_mmff"), "config5_etkdg_mmff": legs.get("config5_etkdg_mmff"),
                         "pool_generation_s": t_pool})
            _attach_conformer_cpu_baseline(line, pool, args)
            if args.dump_outputs:
                write_dumps(args.dump_outputs, dumps)
            print(json.dumps(line))
        if world > 1:
            dist.destroy_process_group()
        return

    n_centres = args.n_centres or 20000
    fp_host = synthetic.clustered_fingerprints(n_centres, 50, seed=synthetic.SEED)
    n, words = fp_host.shape
    h_fp = torch.from_numpy(fp_host.view(np.int32)).pin_memory()
    d_fp = h_fp.to(dev)
    h_ids = torch.empty(n, dtype=torch.int32).pin_memory()
    stream = torch.cuda.current_stream()

    def step_device(x):
        if world == 1:
            return fused_butina_device(x, CUTOFF)
        return fused_butina_sharded(x, CUTOFF)

    def step_e2e():
        # one GPU: the whole array over PCIe; several: each rank uploads 1/world of the rows and the ranks all-gather the
        # slices over NVLink (nvmolkit_b200.distributed.sharded_upload) - the public multi-GPU entry for host fingerprints
        x = sharded_upload(h_fp, dev) if world > 1 else h_fp.to(dev, non_blocking=True)
        ids, cen = step_device(x)
        h_ids.copy_(ids, non_blocking=True)
        stream.synchronize()
        return ids, cen

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = None
        for _ in range(steps):
            out = fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) / steps, out

    for _ in range(args.warmup):
        step_device(d_fp)
    launches0 = _lib.launch_count()
    with ClockSampler(local) as clocks:
        ms_dev, (ids, cen) = timed(lambda: step_device(d_fp), args.steps)
        launches = _lib.launch_count() - launches0
        # dominant kernel alone (CUDA events on its own stream, recorded inside the library around the tile kernel)
        pass_ms = []
        tensor_path = True
        for _ in range(max(1, min(3, args.steps))):
            step_device(d_fp)
            try:
                pass_ms.append(_lib.profile_read("neighbor_pass_tc"))
            except ValueError:
                tensor_path = False
                pass_ms.append(_lib.profile_read("neighbor_pass"))
        phases = {k: _lib.profile_read(k) for k in ("neighbor_pass", "csr_build", "cluster_loop")}
        try:
            phases["verify_candidates"] = _lib.profile_read("verify_candidates")
        except ValueError:
            pass
        if tensor_path:
            phases["neighbor_pass_tc"] = _lib.profile_read("neighbor_pass_tc")
    # end to end after the clock sampler has stopped (nvidia-smi queries take the driver for a while; this loop is host-driven:
    # a pinned 256 MB copy, the call, a 4 MB copy back). Its time depends on the box's host link: 59-70 ms per step on most
    # boxes of the pool, 115 ms on some (profiles/r02_path_a_summary.md)
    step_e2e()
    ms_e2e, _ = timed(step_e2e, args.steps)

    # materialised cross-similarity (the reference's crossTanimotoSimilarity output format): HBM-write bound, 8 B / pair
    cross = None
    if args.cross_n > 0 and rank == 0:
        from nvmolkit_b200.similarity import crossTanimotoSimilarity

        xa = d_fp[: args.cross_n]
        xb = d_fp[args.cross_n: 2 * args.cross_n] if n >= 2 * args.cross_n else d_fp[: args.cross_n]
        for _ in range(2):
            res = crossTanimotoSimilarity(xa, xb)
        torch.cuda.synchronize()
        times = []
        for _ in range(3):
            res = crossTanimotoSimilarity(xa, xb)
            try:
                times.append(_lib.profile_read("cross_tc"))
            except ValueError:
                times = []
                break
        if times:
            nb = xb.shape[0]
            ms_c = float(np.mean(times))
            bytes_c = 8.0 * args.cross_n * nb + 256.0 * (args.cross_n + nb)
            peak_c, src_c = measured_peaks()
            cross = {"pairs_per_s": args.cross_n * nb / (ms_c * 1e-3), "kernel_ms": ms_c, "shape": [args.cross_n, nb],
                     "roofline": {"bound": "hbm", "achieved": bytes_c / (ms_c * 1e-3) / 1e9, "peak": peak_c, "unit": "GB/s",
                                  "frac": bytes_c / (ms_c * 1e-3) / 1e9 / peak_c, "algorithmic_bytes": bytes_c,
                                  "kernel": "simTensorKernel<materialise> (cross_tc)", "peak_source": src_c}}
        rng = np.random.default_rng(synthetic.SEED)
        ri = torch.from_numpy(rng.integers(0, res.torch().shape[0], DUMP_SAMPLE)).to(dev)
        ci = torch.from_numpy(rng.integers(0, res.torch().shape[1], DUMP_SAMPLE)).to(dev)
        dumps["cross_tanimoto_sample"] = res.torch()[ri, ci].cpu().numpy()
        del res
        # BASELINE config 1: 1k x 1k (whole call through the public function, CUDA events on the current stream)
        ya, yb = d_fp[:1000], d_fp[1000:2000]
        for _ in range(5):
            crossTanimotoSimilarity(ya, yb)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(50):
            res1 = crossTanimotoSimilarity(ya, yb)
        e1.record()
        torch.cuda.synchronize()
        ms1 = e0.elapsed_time(e1) / 50
        dumps["cross_tanimoto_1k_x_1k"] = res1.numpy()
        if cross is not None:
            cross["config1_1k_x_1k"] = {"ms_per_call": ms1, "pairs_per_s": 1e6 / (ms1 * 1e-3),
                                        "algorithmic_GBps": (8.0e6 + 256.0 * 2000) / (ms1 * 1e-3) / 1e9}

    # second half of the BASELINE metric: ETKDG + MMFF mols/s on config 3 (and configs 4 / 5 on eight GPUs)
    legs = run_conformer_legs(args, pool, dev, world, rank, dumps) if pool is not None else {}

    ids_h = ids.cpu().numpy()
    dumps["butina_cluster_ids"], dumps["butina_centroids"] = ids_h, cen.cpu().numpy()
    n_clusters = int(cen.numel())
    assert ids_h.min() == 0 and ids_h.max() == n_clusters - 1
    sizes = np.bincount(ids_h, minlength=n_clusters)
    assert (np.diff(sizes) <= 0).all(), "cluster sizes must be non-increasing"

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    value = unique_pairs(n) / (ms_dev * 1e-3)
    e2e = unique_pairs(n) / (ms_e2e * 1e-3)
    peak, peak_src = measured_peaks()
    kernel_ms = float(np.mean(pass_ms))
    n_edges = None
    algo_bytes = 256.0 * n + 4.0 * n  # fingerprints read once + counts written (SURVEY.md §8d "fused count" pass)
    achieved = algo_bytes / (kernel_ms * 1e-3) / 1e9
    # integer-issue roof of the same kernel: 64 POPC per pair at 16 lanes/clk/SM (148 SMs, measured max clock)
    pairs_per_rank = unique_pairs(n) / world
    popc_rate = pairs_per_rank * words / (kernel_ms * 1e-3)

    if tensor_path:
        # dominant kernel = tcgen05 block-scaled fp4 MMA tile (kind::mxf4 over the 0/1 E2M1 expansion, unit scale
        # factors): 2 * bits ops per pair over the tiles actually visited (upper triangle). Dense fp4 issues at 4x the
        # bf16 rate on B200 (9 vs 2.25 PFLOP/s nominal), so the roof is 4 x the MEASURED bf16 throughput.
        bf16 = 1700.1
        try:
            bf16 = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops"])
        except Exception:
            pass
        fp4 = (words * 32) % 256 == 0  # the library's own eligibility rule (tanimoto_tc.cu); else the int8 tile runs
        mult = 4.0 if fp4 else 2.0
        tiles_pairs = unique_pairs(n) / world  # + diagonal-tile overhead (< 0.1 % at 1M)
        # superposition: one tensor-core row (column) carries the sum of S (C) fingerprints, so the pass ISSUES 1/(S C) of
        # the pair-by-pair contraction (the survivors' exact re-count is the separate verify kernel, in phases_ms);
        # superS below = S * C = pairs bounded by one accumulator
        superS = max(1, _lib.get_option("similarity_superpose_last")) if fp4_possible(words) else 1
        tops = tiles_pairs / superS * 2.0 * words * 32 / (kernel_ms * 1e-3) / 1e12
        operand_bytes = ((128 + 112) * (words * 32 // 2) / (128.0 * superS * 224.0) if fp4
                         else (128 + 256) * (words * 32) / (128.0 * 256.0))
        roofline = {"bound": "tensor", "achieved": tops, "peak": mult * bf16, "unit": "TFLOP/s", "frac": tops / (mult * bf16),
                    "traffic": measured_traffic().get("simTensorKernel<count>") if n == 1_000_000 and world == 1 else None,
                    "kernel": ("simTensorKernel<count, fp4, cluster2> (tcgen05.mma kind::mxf4.block_scale, neighbor_pass_tc)" if fp4
                               else "simTensorKernel<count> (tcgen05.mma kind::i8, neighbor_pass_tc)"),
                    "kernel_ms": kernel_ms, "ops_per_pair": 2 * words * 32 / superS, "pairs_per_accumulator": superS,
                    "candidates_verified": _lib.get_option("similarity_candidates_last") if superS > 1 else 0,
                    "unsuperposed_equivalent_TOPs": tops * superS,
                    "peak_source": f"{mult:.0f} x MEASURED_PEAKS.json bf16_tflops (dense {'fp4' if fp4 else 'u8'} = {mult:.0f} x bf16 rate; of measured)",
                    "hbm_algorithmic_GBps": (n * words * 32 / (2 if fp4 else 1) + 260.0 * n) / (kernel_ms * 1e-3) / 1e9,
                    "l2_operand_bytes_per_pair": operand_bytes,
                    "l2_operand_TBps": tiles_pairs * operand_bytes / (kernel_ms * 1e-3) / 1e12,
                    "note": "exact: 0/1 products, fp32 accumulation of sums <= 4096; HBM share negligible, the operand "
                            "stream comes from L2 (TMA, column operand multicast to the CTA pair)"}
    else:
        roofline = None
    out = {
        "metric": METRIC_NAME, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_dev, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "e2m1 0/1 x e2m1 0/1 -> f32 (exact integer counts), integer threshold test = the f64 predicate", "data": "synthetic",
        "config": {"workload": "1Mx1M symmetric 2048-bit Tanimoto + Butina (sim>=0.7)" if n == 1_000_000 else
                   f"{n}x{n} symmetric 2048-bit Tanimoto + Butina (sim>=0.7) [reduced size override]",
                   "n_fingerprints": n, "fp_bits": words * 32, "cutoff": CUTOFF, "pairs_counted": "unique n(n-1)/2",
                   "l2": "inputs (256 MB) larger than L2", "parallelism": f"row-group x{world}" if world > 1 else "1gpu"},
        "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": int(n * words * 4), "d2h_bytes_per_step": int(n * 4),
                "ms_per_step": ms_e2e,
                "h2d": ("whole job: every rank copies 1/world of the rows from pinned host memory, the slices are all-gathered "
                        "over NVLink (distributed.sharded_upload)") if world > 1 else "pinned host -> device, whole array"},
        "gpu_launches": int(launches),
        "clocks": clocks.summary(),
        "roofline": roofline if roofline is not None else {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": None, "kernel": "simTileKernel<count> (neighbor_pass)", "kernel_ms": kernel_ms,
                     "algorithmic_bytes": algo_bytes, "peak_source": peak_src,
                     "note": "pass is integer-issue bound by construction (5e-4 B/pair); see popc_roof"},
        "popc_roof": {"achieved_popc_per_s": popc_rate, "peak_popc_per_s": 148 * 16 * 1.965e9,
                      "frac": popc_rate / (148 * 16 * 1.965e9), "unit": "32-bit POPC/s"},
        "phases_ms": phases, "n_clusters": n_clusters,
    }

    # CPU baseline (oracle port, OpenMP on the host cores) on a bounded sample + exact parity on that sample
    import oracle

    cpu_threads = oracle.set_threads(os.cpu_count() or 1)  # torchrun exports OMP_NUM_THREADS=1 to its workers
    ns, _ = cpu_sample_size(target_s=12.0)
    if args.n_centres:
        ns = min(ns, n)
    fps = synthetic.clustered_fingerprints(ns // 50, 50, seed=synthetic.SEED)
    t0 = time.perf_counter()
    ids_cpu, cen_cpu = oracle.butina_fp(fps, CUTOFF)
    dt = time.perf_counter() - t0
    g_ids, g_cen = fused_butina_device(torch.from_numpy(fps.view(np.int32)).to(dev), CUTOFF)
    parity = bool((g_ids.cpu().numpy() == ids_cpu).all() and (g_cen.cpu().numpy() == cen_cpu).all())
    out["cpu_baseline"] = {"value": unique_pairs(len(fps)) / dt, "unit": UNIT, "cores": cpu_threads,
                           "kind": "port",
                           "sample": f"{len(fps)}x{len(fps)} clustered 2048-bit fingerprints, cutoff {CUTOFF}, {dt:.1f} s"}
    out["parity_on_sample"] = "bit-exact" if parity else "MISMATCH"
    out["etkdg_mmff"] = legs.get("etkdg_mmff")
    out["config4_mmff"] = legs.get("config4_mmff")
    out["config5_etkdg_mmff"] = legs.get("config5_etkdg_mmff")
    out["cross_similarity"] = cross
    if out["etkdg_mmff"] is not None:
        out["etkdg_mmff"]["pool_generation_s"] = t_pool
        _attach_conformer_cpu_baseline(out["etkdg_mmff"], pool, args)
    if args.dump_outputs:
        write_dumps(args.dump_outputs, dumps)
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


# ----------------------------------------------------------------------------------------------- path B (conformers)
ETKDG_PARAMS = dict(seed=20260924, boxSize=10.0, optimizerForceTol=1e-3, enforceChirality=1, useExpTorsions=1,
                    useBasicKnowledge=1, maxAttempts=0, dgIters=400, fourthIters=200, etkIters=300, maxRestarts=20)
POOL_CHUNK = 50  # molecules per generator task; task c draws from seed + c, so the pool does not depend on the process count


def _pool_chunk(task):
    """One generator task (runs in a forked worker: NumPy + the host-side wave scheduler only, no CUDA)."""
    from nvmolkit_b200 import synthetic
    from nvmolkit_b200.forcefield import FlatSystem

    chunk_id, n, seed = task
    flat, mols = synthetic.random_embed_molecules(n, 20, 50, seed=seed + 7919 * chunk_id, strict_checks=False)
    mmff = FlatSystem.from_molecules("mmff", [len(m["z"]) for m in mols], [m["terms"] for m in mols])
    return chunk_id, flat, mmff, np.concatenate([m["xyz"] for m in mols])


def conformer_pool(n_mols: int, seed: int, procs: int):
    """`n_mols` DISTINCT pseudo drug-like molecules (20-50 heavy atoms + hydrogens: 43-110 atoms) with DG / ETK / check
    and MMFF term tables - SURVEY.md 8d's synthetic stand-in for the ChEMBL subset of configs 3-5 (no RDKit on the box).
    Returns (FlatEmbedMolecules, MMFF FlatSystem, generator coordinates [atoms, 3])."""
    import multiprocessing as mp

    from nvmolkit_b200.embedMolecules import FlatEmbedMolecules
    from nvmolkit_b200.forcefield import FlatSystem

    tasks = [(c, min(POOL_CHUNK, n_mols - c * POOL_CHUNK), seed) for c in range((n_mols + POOL_CHUNK - 1) // POOL_CHUNK)]
    procs = max(1, min(procs, len(tasks)))
    if procs == 1:
        parts = [_pool_chunk(t) for t in tasks]
    else:
        with mp.get_context("fork").Pool(procs) as pool:
            parts = pool.map(_pool_chunk, tasks, chunksize=1)
    parts.sort(key=lambda r: r[0])
    return (FlatEmbedMolecules.concat([r[1] for r in parts]), FlatSystem.concat([r[2] for r in parts]),
            np.concatenate([r[3] for r in parts]))


class ConformerLeg:
    """ETKDG embed of `confs` conformers per molecule, then MMFF94 200-iteration BFGS of every embedded conformer, on
    this rank's molecule range of `mol_ids` (indices into the pool); N > 1 ends with the all-gather of the results."""

    def __init__(self, flat, mmff, dev, world, rank, max_attempts=-1):
        self.flat, self.mmff, self.dev, self.world, self.rank, self.max_attempts = flat, mmff, dev, world, rank, max_attempts

    def step(self, mol_ids, confs, embed=True, start_xyz=None, gather=True):
        import torch

        from nvmolkit_b200.distributed import all_gather_v, molecule_range
        from nvmolkit_b200.embedMolecules import EmbedParameters, embed_slots
        from nvmolkit_b200.forcefield import ConformerBatch
        from nvmolkit_b200.minimizer import minimize

        lo, hi = molecule_range(len(mol_ids), self.rank, self.world)
        mine = np.ascontiguousarray(mol_ids[lo:hi], dtype=np.int32)
        if embed:
            raw = embed_slots(self.flat, EmbedParameters(randomSeed=ETKDG_PARAMS["seed"]), confs, self.max_attempts, mol_indices=mine)
            batch = ConformerBatch(raw.slot_mol, raw.slot_atom_start, np.zeros((0, 3)))
            res = minimize(self.mmff, batch, 200, 1e-4, positions=raw.coords, active=raw.ok.to(torch.uint8))
        else:  # config 4: MMFF from pre-embedded coordinates (start_xyz = (atom offsets of the pool, coordinates))
            raw = None
            offs, xyz = start_xyz
            counts = self.mmff.atom_counts[mine]
            order = np.argsort(-counts, kind="stable")  # largest first: evens out the persistent CTAs' tail
            mine = mine[order]
            from nvmolkit_b200._hostutil import rows_of

            rows = rows_of(offs, mine)
            starts = np.concatenate([[0], np.cumsum(self.mmff.atom_counts[mine])]).astype(np.int32)
            batch = ConformerBatch(mine, starts, np.zeros((0, 3)))
            pos = torch.from_numpy(xyz[rows]).to(self.dev)
            res = minimize(self.mmff, batch, 200, 1e-4, positions=pos)
        if self.world > 1 and gather:  # the one collective of the path: all-gather-v of the results
            all_gather_v(res.energies)
            all_gather_v(res.positions)
        return raw, res


def _event_timed(fn, dev, world):
    """One call of fn bracketed by barrier + synchronize, CUDA events, max over ranks (ms)."""
    import torch
    import torch.distributed as dist

    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item()), out


def _conformer_roofline(stats, phases, peak, peak_src, traffic):
    """HBM roofline of the two kernels of the path from the device-side work counters: ALGORITHMIC bytes by SURVEY.md
    8d's (the reference's) scheme - per BFGS iteration 3 n^2 x 8 B of inverse Hessian + (1 + k_ls) x term bytes, summed
    over the iterations the kernel actually ran - divided by the kernel's CUDA-event duration."""
    out = {}
    for bank, phase, kernel in (("embed", "etkdg", "etkdgKernel"), ("minimize", "bfgs", "bfgsKernel<Mmff>")):
        st, ms = stats[bank], phases.get(phase)
        if not ms or not st["bfgs_iterations"]:
            continue
        ach = st["algorithmic_bytes"] / (ms * 1e-3) / 1e9
        # what THIS design has to move for the same iterations: one read + one write of the upper triangle of the inverse
        # Hessian (f32 in the embedder, f64 in MMFF) instead of three passes over the full f64 matrix, same term bytes
        own = st["algorithmic_bytes"] - 24 * st["n2_iterations"] + (4 if bank == "embed" else 8) * st["n2_iterations"]
        out[bank] = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                     "own_scheme_bytes": own, "own_scheme_GBps": own / (ms * 1e-3) / 1e9,
                     "own_scheme_frac": own / (ms * 1e-3) / 1e9 / peak,
                     "note": "achieved = the reference scheme's bytes (SURVEY.md 8d: 3 n^2 x 8 B + term records per iteration) / "
                             "time, so frac > 1 means: faster than that scheme could run at the HBM roof; own_scheme_* = the bytes "
                             "this kernel's one-sweep triangular update needs",
                     "traffic": traffic.get(kernel), "kernel": kernel, "kernel_ms": ms,
                     "algorithmic_bytes": st["algorithmic_bytes"], "bfgs_iterations": st["bfgs_iterations"],
                     "energy_evals": st["energy_evals"], "gradient_evals": st["gradient_evals"],
                     "minimisations": st["minimisations"], "peak_source": peak_src}
    return out


def measured_traffic() -> dict:
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernels, from the committed ncu --set full
    captures of this same command (profiles/traffic.json: {kernel: {"bytes": ..., "source": ...}})."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return {k: v["bytes"] for k, v in json.load(open(p)).items()}
    except Exception:
        return {}


def run_conformer_legs(args, pool, dev, world, rank, dumps):
    """Configs 3 (always), 4 and 5 (8 GPUs, or --all-configs) of BASELINE.json. Returns the dict for the JSON line and
    puts this rank's config-3 results into `dumps`."""
    import torch

    from nvmolkit_b200 import _lib

    flat, mmff, gen_xyz = pool
    n_pool = len(flat)
    leg = ConformerLeg(flat, mmff, dev, world, rank)
    peak, peak_src = measured_peaks()
    traffic = measured_traffic()
    atom_offs = np.concatenate([[0], np.cumsum(flat.atom_counts)]).astype(np.int64)
    out = {}

    # ---- config 3: n_pool distinct molecules x `confs` conformers, ETKDG + MMFF
    n3 = args.etkdg_mols
    ids3 = (np.arange(n3) % n_pool).astype(np.int32)
    warm = ids3[:: max(1, n3 // max(1, 512 * world))]  # a short warm-up on a strided subset (allocator, clocks, caches)
    leg.step(warm, args.confs)
    # --steps counts the steps of the line's headline; beside the Butina headline this leg (tens of seconds a step) runs
    # one. Every step is timed on its own; launches, work counters and phases are those of the last step.
    steps = args.steps if args.workload == "conformers" else 1
    step_ms = []
    for _ in range(steps):
        _lib.stats_read(reset=True)
        l0 = _lib.launch_count()
        ms, (raw, res) = _event_timed(lambda: leg.step(ids3, args.confs), dev, world)
        step_ms.append(ms)
    ms = float(np.mean(step_ms))
    launches = _lib.launch_count() - l0
    stats = _lib.stats_read(reset=True)
    phases = {"etkdg": _lib.profile_read("etkdg"), "bfgs": _lib.profile_read("bfgs")}
    ok = raw.ok.cpu().numpy().astype(bool)
    st = res.status.cpu().numpy()
    it = res.iters.cpu().numpy()
    # a slot that failed to embed holds no conformer (its energy and coordinates are undefined): the dump keeps the
    # per-slot embedded flag, and energies and sampled coordinates of the embedded slots only
    embedded = np.nonzero(ok)[0]
    dumps["etkdg_mmff_slot_mol"] = raw.slot_mol
    dumps["etkdg_mmff_embedded"] = ok
    dumps["etkdg_mmff_energies"] = res.energies.cpu().numpy()[embedded]
    from nvmolkit_b200._hostutil import rows_of
    from nvmolkit_b200.synthetic import SEED

    pick = np.sort(np.random.default_rng(SEED).choice(embedded, min(len(embedded), DUMP_CONFORMERS), replace=False))
    rows = rows_of(raw.slot_atom_start, pick)
    dumps["etkdg_mmff_coords_sample"] = res.positions.reshape(-1, 3)[torch.from_numpy(rows).to(dev)].cpu().numpy()
    dumps["etkdg_mmff_coords_sample_slots"] = pick

    # end to end through the public API: host term tables in (uploaded inside the timed region), coordinates and energies
    # out to pinned host memory
    n_atoms_mine = int(raw.slot_atom_start[-1])
    h_pos = torch.empty((n_atoms_mine, 3), dtype=torch.float64).pin_memory()
    h_en = torch.empty(len(raw.slot_mol), dtype=torch.float64).pin_memory()

    def e2e_step():
        flat.drop_device()
        mmff._device.clear()
        _r, rs = leg.step(ids3, args.confs)
        h_pos.copy_(rs.positions.reshape(-1, 3), non_blocking=True)
        h_en.copy_(rs.energies, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return rs

    ms_e2e = float(np.mean([_event_timed(e2e_step, dev, world)[0] for _ in range(steps)]))
    h2d = flat.nbytes() + mmff.nbytes()
    # (the ncu traffic capture is of THIS workload at its default size on one GPU: not quoted for anything else)
    roof = _conformer_roofline(stats, phases, peak, peak_src, traffic if (n3 == 10000 and args.confs == 10 and world == 1) else {})
    out["etkdg_mmff"] = {
        "metric": "etkdg_mmff_mols_per_s", "value": n3 / (ms * 1e-3), "unit": "mols/s", "ms_per_step": ms, "steps": steps,
        "n_gpus": world, "scaling": "strong",
        "dtype": "f64 energies / gradients / line search; inverse Hessian f32 in the embedder (option etkdg_hessian_fp64: f64, "
                 "measured beside it under embedder_hessian_f32_vs_f64), f64 in MMFF",
        "config": {"workload": f"config 3: {n3} drug-like pseudo-mols ({min(n3, n_pool)} distinct, 20-50 heavy atoms + H, mean "
                               f"{float(flat.atom_counts.mean()):.1f} atoms) x {args.confs} conformers, ETKDG embed (max attempts = "
                               f"10 x atoms, the API default) + MMFF94 200-iteration BFGS", "data": "synthetic",
                   "l2": f"term tables {h2d / 1e9:.2f} GB, inverse-Hessian slabs > L2"},
        "e2e": {"value": n3 / (ms_e2e * 1e-3), "unit": "mols/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": int(h2d),
                "d2h_bytes_per_step": int(h_pos.numel() * 8 + h_en.numel() * 8)},
        "roofline": roof.get("embed"), "roofline_mmff": roof.get("minimize"),
        "phases_ms": phases, "gpu_launches": int(launches),
        "conformers_embedded_frac": float(ok.mean()), "mean_attempts": float(raw.attempts.float().mean().item()),
        "stage_failures": raw.stage_failures.cpu().numpy().tolist(),
        "mmff_converged_frac": float((st[ok] == 0).mean()) if ok.any() else 0.0,
        "mmff_iters_hist": np.bincount(np.minimum(it[ok] // 50, 4), minlength=5).tolist() if ok.any() else [],
        "mmff_note": "200 iterations is BASELINE config 4's fixed budget; the CPU transcription of RDKit's BFGS needs 450-1000 "
                     "iterations to converge these 43-110 atom systems from an ETKDG geometry (DESIGN.md 6), so nearly every "
                     "conformer runs all 200",
    }

    # ---- the same path with the embedder's inverse Hessian in fp64 (the reference's storage type) beside the fp32 default,
    # on a bounded subset of config 3 (both timed on the same molecules)
    if world == 1 and args.hessian_compare_mols > 0:
        nh = min(n3, args.hessian_compare_mols)
        idsh = ids3[:nh]
        cmp_ = {"mols": int(nh), "confs": int(args.confs)}
        for name, flag in (("f32", 0), ("f64", 1)):
            _lib.set_option("etkdg_hessian_fp64", flag)
            msh, (rawh, _resh) = _event_timed(lambda: leg.step(idsh, args.confs), dev, world)
            cmp_[name] = {"mols_per_s": nh / (msh * 1e-3), "etkdg_ms": _lib.profile_read("etkdg"), "bfgs_ms": _lib.profile_read("bfgs"),
                          "embedded_frac": float(rawh.ok.float().mean().item()),
                          "mean_attempts": float(rawh.attempts.float().mean().item())}
        _lib.set_option("etkdg_hessian_fp64", 0)
        out["etkdg_mmff"]["embedder_hessian_f32_vs_f64"] = cmp_

    # ---- configs 4 and 5 (BASELINE: 8 GPUs)
    if world == 8 or args.all_configs:
        n4 = args.mmff_mols
        ids4 = (np.arange(n4) % n_pool).astype(np.int32)
        rng = np.random.default_rng(4)
        xyz4 = gen_xyz + rng.normal(0.0, 0.1, gen_xyz.shape)  # pre-embedded coordinates + N(0, 0.1 A), SURVEY.md 8d
        leg.step(ids4[:: max(1, n4 // max(1, 2048 * world))], 1, embed=False, start_xyz=(atom_offs, xyz4))
        _lib.stats_read(reset=True)
        ms4, (_r4, res4) = _event_timed(lambda: leg.step(ids4, 1, embed=False, start_xyz=(atom_offs, xyz4)), dev, world)
        st4 = _lib.stats_read(reset=True)
        roof4 = _conformer_roofline(st4, {"bfgs": _lib.profile_read("bfgs")}, peak, peak_src, {})
        out["config4_mmff"] = {
            "metric": "mmff_mols_per_s", "value": n4 / (ms4 * 1e-3), "unit": "mols/s", "ms_per_step": ms4, "n_gpus": world,
            "config": {"workload": f"config 4: {n4} mols ({min(n4, n_pool)} distinct) MMFF94 200-iteration BFGS from pre-embedded "
                                   "coordinates + N(0, 0.1 A), molecule-range sharded, results all-gathered", "data": "synthetic"},
            "roofline": roof4.get("minimize"), "converged_frac": float((res4.status == 0).float().mean().item())}
        n5 = args.e2e_mols
        ids5 = (np.arange(n5) % n_pool).astype(np.int32)
        _lib.stats_read(reset=True)
        ms5, (raw5, res5) = _event_timed(lambda: leg.step(ids5, 1), dev, world)
        st5 = _lib.stats_read(reset=True)
        roof5 = _conformer_roofline(st5, {"etkdg": _lib.profile_read("etkdg"), "bfgs": _lib.profile_read("bfgs")}, peak, peak_src, {})
        out["config5_etkdg_mmff"] = {
            "metric": "etkdg_mmff_mols_per_s", "value": n5 / (ms5 * 1e-3), "unit": "mols/s", "ms_per_step": ms5, "n_gpus": world,
            "config": {"workload": f"config 5: {n5} mols ({min(n5, n_pool)} distinct, config 3 generator cycled) x 1 conformer, ETKDG "
                                   "+ MMFF94 200 iterations, NCCL all-gather-v of coordinates and energies", "data": "synthetic"},
            "roofline": roof5.get("embed"), "roofline_mmff": roof5.get("minimize"),
            "conformers_embedded_frac": float(raw5.ok.float().mean().item())}
    return out


def _attach_conformer_cpu_baseline(leg: dict, pool, args) -> None:
    """CPU arm of the conformer leg: the oracle port with OpenMP on every host core, on one molecule per core x the
    leg's conformers (>= 10 s of CPU work on a 128-core box)."""
    import oracle

    cores = oracle.set_threads(os.cpu_count() or 1)
    nb = args.etkdg_cpu_mols or max(16, cores)
    nb = min(nb, len(pool[0]))
    v, dt_b, okf = run_conformers_cpu(pool, nb, args.confs)
    leg["cpu_baseline"] = {"value": v, "unit": "mols/s", "cores": cores, "kind": "port",
                           "sample": f"{nb} mols x {args.confs} conformers (the first molecules of the same pool), {dt_b:.1f} s, "
                                     f"embedded {okf:.2f}"}


def run_conformers_cpu(pool, n_mols: int, confs: int):
    """The same config-3 pipeline on the host cores with the oracle (OpenMP over conformer slots). Returns mols/s."""
    import oracle

    flat, mmff, _ = pool
    mol_ids = (np.arange(n_mols) % len(flat)).astype(np.int32)
    slot_mol = np.repeat(mol_ids, confs)
    starts = np.concatenate([[0], np.cumsum(flat.atom_counts[slot_mol])]).astype(np.int32)
    p = dict(ETKDG_PARAMS, maxAttempts=10 * int(flat.atom_counts[mol_ids].max()))
    t0 = time.perf_counter()
    coords, ok, att, en = oracle.etkdg_embed_batch((flat.dg.atom_counts, flat.dg.tables), (flat.etk.atom_counts, flat.etk.tables),
                                                  flat.checks.tables, flat.checks.num_impropers, p, slot_mol, starts)
    keep = np.nonzero(ok)[0]
    if len(keep):
        from nvmolkit_b200._hostutil import rows_of

        k_starts = np.concatenate([[0], np.cumsum(flat.atom_counts[slot_mol[keep]])]).astype(np.int32)
        oracle.ff_minimize("mmff", mmff.atom_counts, mmff.tables, slot_mol[keep], k_starts, coords[rows_of(starts, keep)], 200, 1e-4)
    dt = time.perf_counter() - t0
    return n_mols / dt, dt, float(ok.mean())


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="all", choices=["all", "butina", "conformers"],
                    help="all = the Butina headline + the conformer legs; conformers = the ETKDG+MMFF leg as the line")
    ap.add_argument("--n-centres", type=int, default=0, help="override the problem size (x50 fingerprints); testing only")
    ap.add_argument("--cross-n", type=int, default=32768, help="rows of the materialised cross-similarity leg (0 = skip)")
    ap.add_argument("--etkdg-mols", type=int, default=10000, help="molecules of the ETKDG+MMFF leg, config 3 (0 = skip)")
    ap.add_argument("--confs", type=int, default=10)
    ap.add_argument("--pool", type=int, default=10000, help="distinct pseudo-molecules generated (cycled beyond that)")
    ap.add_argument("--pool-procs", type=int, default=0, help="generator processes (0 = host cores / ranks, at most 48)")
    ap.add_argument("--etkdg-cpu-mols", type=int, default=0, help="molecules of that leg's CPU sample (0 = one per host core)")
    ap.add_argument("--tensor-cluster", type=int, default=-1, help="pair-pass tile variant override (testing; -1 = library default)")
    ap.add_argument("--superpose", type=int, default=-1, help="pair-pass row superposition override (testing; -1 = library default)")
    ap.add_argument("--bfgs-l2-persist", action="store_true", help="mark the minimisers' inverse-Hessian slabs persisting in L2 (experiment)")
    ap.add_argument("--pipeline-chunks", type=int, default=-1, help="chunks of the pipelined pass / verification (testing; -1 = library default, 1 = off)")
    ap.add_argument("--superpose-auto", type=int, default=-1, help="0: no pilot passes, run the configured factors (profiling; -1 = library default)")
    ap.add_argument("--superpose-cols", type=int, default=-1, help="pair-pass column superposition override (testing; -1 = library default)")
    ap.add_argument("--hessian-compare-mols", type=int, default=2000,
                    help="config-3 subset on which the fp64 embedder Hessian is timed beside the fp32 default (0 = skip)")
    ap.add_argument("--all-configs", action="store_true", help="run configs 4 and 5 on fewer than 8 GPUs too")
    ap.add_argument("--mmff-mols", type=int, default=100000, help="config 4 size")
    ap.add_argument("--e2e-mols", type=int, default=1000000, help="config 5 size")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step of each leg returned as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
