#!/usr/bin/env python
"""bench.py - Mvoxels/s polygonized (BASELINE.json metric) on the seeded Perlin terrain.

  python bench.py --gpus N --steps K --warmup W            this repo's CUDA path (one rank per GPU under torchrun)
  python bench.py --impl reference --gpus N --steps K ...  the reference's own OpenMP CPU Polygonizer::Execute
                                                           (oracle/_ref, unmodified sources compiled by oracle/Makefile)

A "step" is one full polygonization (all LOD levels + transition cells = what the reference's Execute always
computes; BASELINE configs[2] asks for levels 0-3, a subset) of ONE n^3 grid (n = 1024 by default).
  N = 1 : the grid is resident in HBM, vxb_polygonize (one CUDA graph).
  N > 1 : the SAME grid polygonized by all N ranks (strong scaling, voxels_b200.dist.ShardedGrid): the cube's z-pieces
          live in the ranks' HBM (cyclic deal, peer-mapped over NVLink), work is dealt by blocks, two exchanges inside
          every step (an ncclAllGather of the per-block info; peer stores of material pages ordered by a second tiny
          all-gather).
  value : n^3 / time of a step; CUDA events on the launching stream around K steps, barrier + synchronize on both
          sides, max over ranks.
  e2e   : the same through the C ABI with HOST (pinned) buffers: H2D of the grid in the reference's PackForSave form
          (every rank its own pieces) and D2H of the full result (directory + vertex/index arenas) inside the timed
          region, every step.
Inputs (1 GiB per channel at 1024^3) are far larger than the 126 MB L2, so no explicit L2 flush is needed.
Prints ONE JSON line on rank 0.

--dump-outputs DIR (N = 1) writes what the last timed step computed, as a caller of vxb_polygonize receives it, to
DIR/<name>.npy (see dump_outputs); the seeded terrain makes the inputs identical from run to run, so two builds can be
compared output for output.
"""
import os
import sys

# Host cores this process may use, read BEFORE any OpenMP runtime exists (with OMP_PROC_BIND set libgomp pins the
# initial thread, after which the affinity mask shows one CPU).  OMP_PROC_BIND=spread (SURVEY.md 8d) is for the
# reference's OpenMP loops and is read when libgomp is loaded; it is set only where the reference runs (the reference
# arm, and the single-process N = 1 line with its cpu_baseline leg) - never under torchrun with several ranks, whose
# main threads would all be pinned to the first core.
HOST_CPUS = len(os.sched_getaffinity(0))
if "reference" in sys.argv or int(os.environ.get("WORLD_SIZE", "1")) == 1:
    os.environ.setdefault("OMP_PROC_BIND", "spread")

import argparse  # noqa: E402
import hashlib  # noqa: E402
import json  # noqa: E402
import subprocess  # noqa: E402
import threading  # noqa: E402
import time  # noqa: E402

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tests"))


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--size", type=int, default=1024, help="grid edge n (power of two)")
    ap.add_argument("--levels", type=int, default=0, help="LOD levels to compute (0 = all, as the reference; N = 1 only)")
    ap.add_argument("--no-transitions", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-config4", action="store_true", help="skip the second record (2048^3, BASELINE configs[3])")
    ap.add_argument("--no-tiles", action="store_true", help="N > 1: skip the independent-tiles weak-scaling extra")
    ap.add_argument("--group-planes", type=int, default=0, help="N > 1: planes per scan group / cube piece (0 = default)")
    ap.add_argument("--shard-mode", default="replicated", choices=["replicated", "cube"],
                    help="N > 1: volumes replicated in every rank's HBM (work sharded; default) or sharded as a peer-mapped cube")
    ap.add_argument("--dump-outputs", metavar="DIR", help="N = 1: write the last timed step's result to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and int(os.environ.get("WORLD_SIZE", "1")) > 1:
        ap.error("--dump-outputs writes the result of one GPU (N = 1)")
    return args


# rows kept per array by --dump-outputs (136, 72, 8, 72 and 8 bytes a row): at most 56 MiB in all
DUMP_ROWS = {"blocks": 1 << 17, "vertices": 1 << 18, "indices": 1 << 20, "transition_vertices": 1 << 17, "transition_indices": 1 << 19}


def dump_outputs(res, directory):
    """The result of one vxb_polygonize as float arrays, in the reference's order (levels, then blocks by coordinate, each
    block's vertices and indices in turn; arena offsets, which vary from run to run, are left out):
      blocks [B, 17] float64      level, coord_id, id, vertex_count, index_count, trans_vertex_count[6], trans_index_count[6]
      vertices [V, 18] float32    pos[3], sec[4] (sec.w: flag bits, kept as they are), nrm[3], tex bytes[8]
      indices [I] float64         block-local
      transition_vertices / transition_indices   the same for the transition cells, block by block, face by face
      stats [20] float64          the statistics of the run
    An array longer than DUMP_ROWS keeps a sample of its rows, in order, drawn with a fixed seed: the same rows for the
    same length."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    rec = res.records
    blocks = np.concatenate([np.stack([rec[f] for f in ("level", "coord_id", "id", "vertex_count", "index_count")], axis=1),
                             rec["trans_vertex_count"], rec["trans_index_count"]], axis=1).astype(np.float64)
    levels = [res.level(l) for l in range(int(rec["level"].max()) + 1)] if len(rec) else []

    def cat(name, dtype):
        parts = [getattr(lv, name) for lv in levels]
        return np.concatenate(parts) if parts else np.zeros(0, dtype)

    def vertex_rows(v):
        return np.concatenate([v["pos"], v["sec"], v["nrm"], v["tex"].astype(np.float32)], axis=1).astype(np.float32)

    arrays = {"blocks": blocks, "vertices": vertex_rows(cat("verts", res.verts.dtype)), "indices": cat("idx", np.uint32).astype(np.float64),
              "transition_vertices": vertex_rows(cat("tverts", res.verts.dtype)), "transition_indices": cat("tidx", np.uint32).astype(np.float64)}
    for name, a in arrays.items():
        if len(a) > DUMP_ROWS[name]:
            rows = np.sort(np.random.default_rng(1234).choice(len(a), DUMP_ROWS[name], replace=False))
            a = a[rows]
        np.save(os.path.join(directory, name + ".npy"), a)
    np.save(os.path.join(directory, "stats.npy"), res.stats.astype(np.float64))


def measured_peak_hbm():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def kernel_source_digest():
    """sha256 over the kernel sources: a committed ncu capture is quoted only for the build it was taken from."""
    h = hashlib.sha256()
    d = os.path.join(REPO, "voxels_b200", "csrc")
    for name in sorted(os.listdir(d)):
        if name.endswith((".cu", ".cuh", ".h")):
            with open(os.path.join(d, name), "rb") as f:
                h.update(f.read())
    return h.hexdigest()[:16]


def host_cpu():
    model, cores = "unknown", set()
    try:
        phys = core = None
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name") and model == "unknown":
                    model = line.split(":", 1)[1].strip()
                elif line.startswith("physical id"):
                    phys = line.split(":", 1)[1].strip()
                elif line.startswith("core id"):
                    core = line.split(":", 1)[1].strip()
                elif not line.strip():
                    if phys is not None and core is not None:
                        cores.add((phys, core))
                    phys = core = None
    except Exception:
        pass
    return model, len(cores)


def cgroup_cpu(root="/sys/fs/cgroup"):
    """The container's CPU quota and throttling counters (cgroup v2): a reference run with more threads than the quota gets
    throttled by the kernel, which the baseline record should show.  {} when the files are not there."""
    out = {}
    try:
        quota, period = open(os.path.join(root, "cpu.max")).read().split()[:2]
        out["quota_cpus"] = None if quota == "max" else round(float(quota) / float(period), 2)
        for line in open(os.path.join(root, "cpu.stat")):
            k, v = line.split()
            if k in ("nr_periods", "nr_throttled", "throttled_usec"):
                out[k] = int(v)
    except Exception:
        pass
    return out


def cgroup_delta(before, after):
    if not after:
        return None
    return {"quota_cpus": after.get("quota_cpus"), "throttled_periods": after.get("nr_throttled", 0) - before.get("nr_throttled", 0),
            "periods": after.get("nr_periods", 0) - before.get("nr_periods", 0),
            "throttled_ms": round((after.get("throttled_usec", 0) - before.get("throttled_usec", 0)) / 1e3, 1)}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()  # the exact PID we started
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        clocks, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                clocks.append(float(r[0])); mx = float(r[1])
                for k, name in enumerate(names):
                    if r[2 + k].lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        clocks.sort()
        return {"sm_mhz": clocks[len(clocks) // 2] if clocks else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(clocks)}


def reference_threads(ref):
    # every host core this process may use (torchrun exports OMP_NUM_THREADS=1, which is not what the reference would run with)
    return max(ref.L.vxh_max_threads(), HOST_CPUS)


def reference_run(n, steps, warmup, dist, mat, blend, budget_s=150.0, keep_surface=False):
    """Times the reference's own Polygonizer::Execute on the given n^3 grid (numpy [z,y,x] arrays) with the thread count that
    serves it best here: every host CPU, or - in a container with a CPU quota below that (cgroup cpu.max), where a larger
    team is throttled by the kernel - one thread per quota CPU; both are tried once during the warm-up and the faster is
    timed.  The GRID is never shrunk; when warmup + steps executions would not fit the time budget the number of
    executions is cut (never below 1 warm-up + 2 timed) and the line says so.
    Returns (Mvoxels/s, info, ref, grid, surface)."""
    import harness
    if not os.path.exists(harness.REF_LIB):
        return None, {"unavailable": "oracle/_ref/libvxh_ref.so not built (make -C oracle ref needs the reference checkout)"}, None, None, None
    ref = harness.reference()
    all_threads = reference_threads(ref)
    grid = ref.grid_from_dense(dist, mat, blend)
    cg0 = cgroup_cpu()
    quota = cg0.get("quota_cpus")
    candidates = [all_threads]
    if quota and quota < all_threads:
        candidates.append(max(1, int(quota + 0.999)))
    trials, spent = {}, 0.0
    for t in candidates:                         # the warm-up executions double as the thread-count trial
        s, sec = ref.polygonize(grid, threads=t)
        ref.surface_destroy(s)
        trials[t] = sec; spent += sec
    threads = min(trials, key=trials.get)
    extra_warm = max(0, warmup - len(candidates))
    per = trials[threads]
    fit = int((budget_s - spent) / max(per, 1e-3))
    want = extra_warm + steps
    if fit < want:
        extra_warm = 0
        want = max(2, min(steps, fit))
    times, surface = [], None
    for i in range(want):
        s, sec = ref.polygonize(grid, threads=threads)
        if i >= extra_warm:
            times.append(sec)
        if keep_surface and i == want - 1:
            surface = s
        else:
            ref.surface_destroy(s)
    if not keep_surface:
        ref.grid_destroy(grid)
        grid = None
    per_step = sum(times) / len(times)
    model, phys = host_cpu()
    info = {"cores": threads, "physical_cores": phys, "cpu_model": model, "seconds_per_execute": per_step, "best_seconds": min(times),
            "timed_executions": len(times), "warmup_executions": len(candidates) + extra_warm, "n": n, "omp_proc_bind": os.environ.get("OMP_PROC_BIND"),
            "thread_trials_s": {str(k): round(v, 3) for k, v in trials.items()}, "cgroup": cgroup_delta(cg0, cgroup_cpu())}
    return n ** 3 / per_step / 1e6, info, ref, grid, surface


def compare_with_reference(ref, surface, result, stats):
    """Level by level, bit by bit (tests/compare.py rules).  Returns {"checked", "levels", "mismatches", "first"}."""
    import numpy as np
    import compare
    problems = []
    levels = ref.surface_levels(surface)
    for l in range(levels):
        problems += compare.level_diff(ref.surface_level(surface, l), result.level(l), "L%d" % l)
    if stats is not None and not np.array_equal(ref.surface_stats(surface), stats):
        problems.append("statistics differ")
    return {"checked": True, "levels": int(levels), "mismatches": len(problems), "first": problems[:3]}


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    n = args.size

    import torch

    # ---------------------------------------------------------------- reference arm (CPU, rank 0 only)
    if args.impl == "reference":
        if rank != 0:
            return 0
        import harness
        from voxels_b200 import capi
        t0 = time.time()
        if not os.path.exists(harness.REF_LIB):
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libvxh_ref.so not built (make -C oracle ref needs the reference checkout)"}))
            return 0
        # the same bytes the b200 arm fills on the device: the built-in terrain evaluated on the host (all threads)
        dist, mat, blend = harness.reference().builtin_dense(n, capi.Surface.terrain(n))
        value, info, _, _, _ = reference_run(n, args.steps, args.warmup, dist, mat, blend)
        if value is None:
            print(json.dumps({"impl": "reference", "unavailable": info["unavailable"]}))
            return 0
        cut = info["timed_executions"] != args.steps
        line = {
            "impl": "reference", "metric": "Mvoxels/s polygonized", "value": value, "unit": "Mvoxels/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": info["seconds_per_execute"] * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "int8 samples / fp32 vertices", "data": "synthetic",
            "config": {"workload": "%d^3 seeded Perlin terrain, all LOD levels + transition cells (reference Polygonizer::Execute)" % n,
                       "impl": "unmodified reference sources, g++ -O2 -fopenmp -msse2, OMP threads = %d, OMP_PROC_BIND=%s" % (info["cores"], info["omp_proc_bind"]),
                       "same_grid_as_b200_arm": True},
            "cpu_baseline": {"value": value, "unit": "Mvoxels/s", "cores": info["cores"], "physical_cores": info["physical_cores"], "cpu_model": info["cpu_model"],
                             "kind": "reference", "best_value": n ** 3 / info["best_seconds"] / 1e6, "cgroup": info["cgroup"], "thread_trials_s": info["thread_trials_s"],
                             "sample": "full %d^3 grid (never shrunk), Polygonizer::Execute only (grid build excluded), mean of %d timed executions after %d warm-up%s"
                                       % (n, info["timed_executions"], info["warmup_executions"],
                                          " (executions cut from --steps %d --warmup %d to fit the time budget)" % (args.steps, args.warmup) if cut else "")},
            "e2e": {"value": value, "unit": "Mvoxels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": time.time() - t0,
        }
        print(json.dumps(line))
        return 0

    # ---------------------------------------------------------------- this repo's CUDA path
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: bench.py measures the sm_100a kernels and has no CPU fallback"}))
        return 2
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    import voxels_b200
    from voxels_b200 import capi
    from voxels_b200.dist import Ranks, ShardedGrid, bind_to_gpu_numa_node, tile_origin, whole_job_throughput
    numa_node = bind_to_gpu_numa_node(local_rank) if world > 1 else None   # N ranks: each next to its GPU's memory controllers
    ranks = Ranks("nccl", dev)
    flags = voxels_b200.FLAG_NO_TRANSITIONS if args.no_transitions else 0
    peak, peak_src = measured_peak_hbm()

    def barrier():
        ranks.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, stream):
        """K steps bracketed by barrier+synchronize; CUDA events on the launching stream; max over ranks."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        barrier()
        return ranks.max_over_ranks(e0.elapsed_time(e1)) / steps

    def algorithmic_bytes(nn, levels_computed, V, I, TV, TI):
        d_level0 = float(nn) ** 3
        d_upper = sum((nn >> l) ** 3 for l in range(1, levels_computed))
        return d_level0, float(d_upper), 4.0 * (V + TV), 48.0 * (V + TV) + 4.0 * (I + TI)  # SURVEY.md 8(d): D + M + O

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    t_load = time.time()
    extra = {}
    e2e = None
    cpu = None
    parity = None

    if world == 1:
        # ------------------------------------------------------------ N = 1: resident grid, one CUDA graph per step
        ctx = voxels_b200.Context(local_rank)
        t_fill = time.perf_counter()
        ctx.fill(n, capi.Surface.terrain(n))   # Grid::Create(n, n, n, 0, 0, 0, 1, &terrain) on the device (SURVEY.md 8 f3)
        extra["grid_fill_ms"] = 1e3 * (time.perf_counter() - t_fill)
        stream = torch.cuda.ExternalStream(ctx.L.vxb_stream(ctx.h), device=dev)
        info = None

        def step_resident():
            nonlocal info
            info = ctx.polygonize(args.levels, flags)

        for _ in range(max(args.warmup, 3)):
            step_resident()
        ms_step = timed(step_resident, args.steps, stream)
        if args.dump_outputs:
            dump_outputs(ctx.download(), args.dump_outputs)
        while time.time() - t_load < 1.5:  # keep the load up for at least a few clock samples (50 ms period)
            step_resident()
        clocks = sampler.stop()
        clocks["window"] = "warm-up + timed region + identical untimed steps, %.1f s under load" % (time.time() - t_load)
        launches_per_step = info.kernel_launches
        device_ms_inner = info.device_ms

        # per-kernel times for the roofline table (separate steps on one stream with plain launches: clean per-kernel events)
        kind_ms, kind_launches = [0.0] * 8, [0] * 8
        ksteps = max(3, min(args.steps, 10))
        for _ in range(ksteps):
            ctx.polygonize(args.levels, flags | voxels_b200.FLAG_KERNEL_TIMES)
            for k in range(8):
                ms, ln = ctx.kernel_ms(k)
                kind_ms[k] += ms / ksteps
                kind_launches[k] = ln
        info = ctx.polygonize(args.levels, flags)
        levels_computed = info.levels_computed
        V, I, TV, TI = info.vertex_total, info.index_total, info.trans_vertex_total, info.trans_index_total
        d0, dup, bm, bo = algorithmic_bytes(n, levels_computed, V, I, TV, TI)
        bytes_alg_total = d0 + dup + bm + bo
        kinds = ["vxb_scan_kernel (streams the level-0 distance volume once)",
                 "vxb_coarse_lattice_kernel + vxb_block_info / vxb_pyramid / vxb_select kernels (lattices of levels >= 2 + block walk)",
                 "vxb_block_kernel<1>/<2> (levels >= 1: tiles, case codes, material votes, reuse decisions)",
                 "vxb_block_kernel<0> (level 0: tile -> case codes -> decisions -> vertices -> triangles in one pass)",
                 "vxb_vertex_kernel (levels >= 1, flat, one thread per new vertex)",
                 "vxb_triangle_kernel (levels >= 1, flat, one thread per non-trivial cell)",
                 "vxb_transition_kernel + vxb_transition_vertex_kernel (per mid-level block)",
                 "vxb_finish_kernel (compaction + directory)"]
        # SURVEY.md 8(d) split per kernel kind: level-0 samples are read once by the scan; the coarser levels' samples by
        # their block kernels; level-0 materials + vertices + indices by vxb_block_kernel<0>; the rest by the flat kernels.
        # Tile re-reads of candidate blocks and the intermediate cell records are overhead, not algorithmic bytes.
        lv = ctx.download().records
        v0 = int(lv["vertex_count"][lv["level"] == 0].sum()); i0 = int(lv["index_count"][lv["level"] == 0].sum())
        alg_by_kind = [d0, 0.0, dup, 52.0 * v0 + 4.0 * i0, 52.0 * (V - v0), 4.0 * (I - i0), 52.0 * TV + 4.0 * TI, 0.0]
        dom = max(range(8), key=lambda k: kind_ms[k])
        per_kind = {kinds[k]: {"ms_per_step": kind_ms[k], "launches": kind_launches[k], "algorithmic_bytes": alg_by_kind[k],
                               "achieved_gbs": (alg_by_kind[k] / (kind_ms[k] * 1e-3) / 1e9 if kind_ms[k] > 0 else 0.0)} for k in range(8)}
        # DRAM traffic per step from the committed `ncu --set full` capture - only when it was taken from THIS build
        traffic, traffic_src = None, None
        try:
            with open(os.path.join(REPO, "profiles", "r02_traffic.json")) as f:
                tj = json.load(f)
            if tj.get("kernel_source_digest") == kernel_source_digest() and n == 1024 and args.levels == 0 and not args.no_transitions:
                traffic, traffic_src = tj["step"]["dram_read"] + tj["step"]["dram_write"], tj["capture"]
        except Exception:
            pass
        ach = bytes_alg_total / (ms_step * 1e-3) / 1e9
        roofline = {"bound": "hbm", "kernel": "whole step (every kernel of one vxb_polygonize, CUDA graph)", "achieved": ach, "peak": peak, "unit": "GB/s",
                    "frac": ach / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                    "algorithmic_bytes_per_step": bytes_alg_total, "ms_per_step": ms_step,
                    "algorithmic_bytes": {"distance_level0": d0, "distance_upper_levels": dup, "materials": bm, "output": bo},
                    "dominant_kernel": {"kernel": kinds[dom], **per_kind[kinds[dom]], "frac": per_kind[kinds[dom]]["achieved_gbs"] / peak},
                    "all_kernels": per_kind,
                    "all_kernels_note": "CUDA events per kernel kind on one stream with plain launches (VXB_FLAG_KERNEL_TIMES), summed over the kind's launches; the timed step replays a graph with the transition cells on a second stream"}
        workload = "%d^3 seeded Perlin terrain, ONE grid on 1 GPU, LOD levels 0-%d%s (BASELINE configs[2] asks for levels 0-3 + transitions: a subset)" \
                   % (n, levels_computed - 1, "" if args.no_transitions else " + transition cells")
        config = {"workload": workload, "grid": "dense int8 distance + uint8 material + uint8 blend, resident in HBM",
                  "sharding": "none (1 GPU)", "l2": "inputs (%.2f GiB per channel) larger than the 126 MB L2; no flush" % (n ** 3 / 2.0 ** 30),
                  "vertices": int(V), "indices": int(I), "transition_vertices": int(TV), "transition_indices": int(TI), "blocks_emitted": int(info.block_count)}

        # -- e2e: host buffers through the C ABI, H2D + D2H inside the timed region --
        if not args.no_e2e:
            t_pack = time.perf_counter()
            packed = ctx.pack()   # Grid::PackForSave of the device grid: run-length coding on the GPU (SURVEY.md 8 f2)
            extra["grid_pack_ms"] = 1e3 * (time.perf_counter() - t_pack)
            h_blob = torch.from_numpy(packed).pin_memory()
            blob_bytes = int(h_blob.numel())
            ctx2 = voxels_b200.Context(local_rank)
            stream2 = torch.cuda.ExternalStream(ctx2.L.vxb_stream(ctx2.h), device=dev)
            out = {
                "verts": torch.empty(int(info.vertex_span * 1.1) * 48 + 4096, dtype=torch.uint8).pin_memory(),
                "idx": torch.empty(int(info.index_span * 1.1) * 4 + 4096, dtype=torch.uint8).pin_memory(),
                "tverts": torch.empty(int(info.trans_vertex_span * 1.1) * 48 + 4096, dtype=torch.uint8).pin_memory(),
                "tidx": torch.empty(int(info.trans_index_span * 1.1) * 4 + 4096, dtype=torch.uint8).pin_memory(),
            }
            into = {k: v.data_ptr() for k, v in out.items()}
            d2h = [0]
            parts = {"upload": 0.0, "polygonize": 0.0, "download": 0.0, "steps": 0}  # host clock around the three (synchronous) calls

            def step_e2e_packed():
                t0 = time.perf_counter()
                ctx2.upload_packed(h_blob.data_ptr(), blob_bytes)
                t1 = time.perf_counter()
                i2 = ctx2.polygonize(args.levels, flags)
                t2 = time.perf_counter()
                ctx2.download(into=into)
                t3 = time.perf_counter()
                parts["upload"] += t1 - t0; parts["polygonize"] += t2 - t1; parts["download"] += t3 - t2; parts["steps"] += 1
                d2h[0] = i2.block_count * 128 + i2.vertex_span * 48 + i2.index_span * 4 + i2.trans_vertex_span * 48 + i2.trans_index_span * 4

            def breakdown():
                k = max(parts["steps"], 1)
                o = {name: round(1e3 * parts[name] / k, 3) for name in ("upload", "polygonize", "download")}
                parts.update(upload=0.0, polygonize=0.0, download=0.0, steps=0)
                return o

            esteps = max(3, min(args.steps, 5))
            for _ in range(3):
                step_e2e_packed()
            breakdown()
            ms_e2e = timed(step_e2e_packed, esteps, stream2)
            e2e = {"value": float(n) ** 3 / (ms_e2e * 1e-3) / 1e6, "unit": "Mvoxels/s", "ms_per_step": ms_e2e, "steps": esteps, "host_ms": breakdown(),
                   "h2d_bytes_per_step": blob_bytes + 8 * (n // 16) ** 3, "d2h_bytes_per_step": int(d2h[0]),
                   "path": "vxb_grid_upload_packed (PackForSave bytes, pinned host -> HBM, RLE decode on the GPU) + vxb_polygonize + "
                           "vxb_result_download (directory + arenas, HBM -> pinned host)"}
            # the same calls from two host threads, each with its own context and buffers: step k's download (D2H) overlaps
            # step k+1's upload (H2D) and kernels, the way a client streams many grids through one GPU.  Extra information,
            # timed on the host clock over all steps; the headline `e2e` above is one step at a time.
            ctx3 = voxels_b200.Context(local_rank)
            out3 = {k: torch.empty_like(v).pin_memory() for k, v in out.items()}
            into3 = {k: v.data_ptr() for k, v in out3.items()}
            psteps = max(4, esteps * 2)
            gate = threading.Barrier(3, timeout=300)
            failures = []

            def worker(c, buffers):
                try:
                    for i in range(psteps + 1):
                        if i == 1:
                            gate.wait()  # first step = warm-up
                        c.upload_packed(h_blob.data_ptr(), blob_bytes)
                        c.polygonize(args.levels, flags)
                        c.download(into=buffers)
                    gate.wait()
                except Exception as exc:  # never leave the other parties waiting
                    failures.append(repr(exc))
                    gate.abort()

            threads = [threading.Thread(target=worker, args=(ctx2, into)), threading.Thread(target=worker, args=(ctx3, into3))]
            for t in threads:
                t.start()
            try:
                gate.wait()
                t0 = time.perf_counter()
                gate.wait()
                wall_ms = 1e3 * (time.perf_counter() - t0)
            except threading.BrokenBarrierError:
                wall_ms = None
            for t in threads:
                t.join()
            if wall_ms is not None and not failures:
                ms_pipe = wall_ms / (2 * psteps)
                e2e["two_in_flight"] = {"value": float(n) ** 3 / (ms_pipe * 1e-3) / 1e6, "unit": "Mvoxels/s", "ms_per_step": ms_pipe, "steps": 2 * psteps,
                                        "timing": "host clock over all steps; two host threads, one context each, same calls as e2e"}
            else:
                e2e["two_in_flight"] = {"value": None, "error": "; ".join(failures) or "barrier timeout"}
            ctx3.close()
            ctx2.close()
            del out3, out, h_blob

        # -- CPU baseline: the reference itself on this box's host cores, on the SAME bytes, and the parity check of the step --
        if not args.no_cpu_baseline:
            t0 = time.time()
            hd, hm, hb = ctx.download_dense()
            v, ci, ref, rgrid, rsurf = reference_run(n, 3, 1, hd, hm, hb, budget_s=90.0, keep_surface=True)
            if v is not None:
                cpu = {"value": n ** 3 / ci["best_seconds"] / 1e6, "mean_value": v, "unit": "Mvoxels/s", "cores": ci["cores"], "physical_cores": ci["physical_cores"],
                       "cpu_model": ci["cpu_model"], "kind": "reference", "cgroup": ci["cgroup"], "thread_trials_s": ci["thread_trials_s"],
                       "sample": "full %d^3 terrain (the same bytes as the GPU step), Polygonizer::Execute only, best of %d after %d warm-up, OMP_PROC_BIND=%s, %.1f s wall incl. grid build"
                                 % (n, ci["timed_executions"], ci["warmup_executions"], ci["omp_proc_bind"], time.time() - t0)}
                if args.levels == 0 and not args.no_transitions:
                    res = ctx.download()
                    parity = compare_with_reference(ref, rsurf, res, res.stats)
                    parity["what"] = "the reference's PolygonSurface vs the GPU result of the same %d^3 bytes: block table, vertices, indices, transition meshes, statistics" % n
                    del res
                # -- e2e through the reference's own API: Polygonizer::Execute of the drop-in on a reference Grid, host in / host out --
                import harness
                if os.path.exists(harness.B200_LIB) and args.levels == 0 and not args.no_transitions and not args.no_e2e:
                    dl = harness.load(harness.B200_LIB)
                    g2 = dl.grid_from_dense(hd, hm, hb)
                    secs, stage_rows = [], []
                    dsurf = None
                    import ctypes
                    stage_names = ("materials", "block_offsets", "gather_blocks", "upload_decode_tail", "kernels", "download_views")
                    try:
                        hostlib = ctypes.CDLL(os.path.join(REPO, "voxels_b200", "lib", "libvoxels_b200.so"))
                    except Exception:
                        hostlib = None
                    cg0 = cgroup_cpu()
                    for i in range(1 + 7):
                        if dsurf is not None:
                            dl.surface_destroy(dsurf)
                        dsurf, sec = dl.polygonize(g2)
                        if i:
                            secs.append(sec)
                            if hostlib is not None:
                                st6 = (ctypes.c_double * 6)()
                                hostlib.voxels_b200_last_execute_stages(st6)
                                stage_rows.append([round(v, 3) for v in st6])
                    cg_dropin = cgroup_delta(cg0, cgroup_cpu())
                    import compare
                    problems = []
                    for l in range(ref.surface_levels(rsurf)):
                        problems += compare.level_diff(ref.surface_level(rsurf, l), dl.surface_level(dsurf, l), "L%d" % l)
                    order = sorted(range(len(secs)), key=lambda i: secs[i])
                    med = order[len(order) // 2]
                    stages = dict(zip(stage_names, stage_rows[med])) if stage_rows else None
                    dl.surface_destroy(dsurf); dl.grid_destroy(g2)
                    ms_d = 1e3 * secs[med]
                    extra["e2e_dropin"] = {"value": float(n) ** 3 / (ms_d * 1e-3) / 1e6, "unit": "Mvoxels/s", "ms_per_step": ms_d, "statistic": "median of %d executions after 1 warm-up" % len(secs),
                                           "best_ms": 1e3 * min(secs), "mean_ms": 1e3 * sum(secs) / len(secs), "all_ms": [round(1e3 * v, 2) for v in secs], "steps": len(secs),
                                           "host_ms_median_run": stages, "cgroup": cg_dropin,
                                           "path": "Voxels::Polygonizer::Execute of libvoxels_b200.so on a reference Grid (compressed blocks gathered into a pinned blob slab by slab while the "
                                                   "previous slab is copied and decoded on the GPU -> kernels -> arenas back to the host, block views built meanwhile -> PolygonSurface), host clock around Execute only",
                                           "parity": {"checked": True, "mismatches": len(problems), "first": problems[:3]},
                                           "vs_reference_same_run": (float(n) ** 3 / (ms_d * 1e-3) / 1e6) / v}
                ref.surface_destroy(rsurf); ref.grid_destroy(rgrid)
            else:
                cpu = {"value": None, "unit": "Mvoxels/s", "cores": 0, "kind": "reference", "sample": ci["unavailable"]}
            del hd, hm, hb
        ctx.close()
        sharding_note = None
        scaling = "strong"
    else:
        # ------------------------------------------------------------ N > 1: ONE grid, all ranks
        sg = ShardedGrid(ranks, n, group_planes=args.group_planes or None, mode=args.shard_mode)
        sg.fill(capi.Surface.terrain(n))   # replicated: every rank the whole (read-only) grid; cube: the pieces it backs
        sg.ready()
        stream = torch.cuda.ExternalStream(sg.ctx.stream(), device=dev)
        for _ in range(max(args.warmup, 3)):
            info = sg.polygonize(flags)   # grows the arenas if needed (collective retry)
        inner = []

        def step_sharded():
            rc = sg.ctx.polygonize_sharded(3, flags)
            if rc != 0:
                raise RuntimeError("arena overflow inside the timed region")
            inner.append(sg.ctx.info().device_ms)

        ms_step = timed(step_sharded, args.steps, stream)
        # keep the load up for a few clock samples (50 ms period): identical untimed steps, the same count on every rank
        # (the steps are collective), derived from the measured step time
        for _ in range(min(4000, int(1200.0 / max(ms_step, 0.05)))):
            sg.ctx.polygonize_sharded(3, flags)
        inner_timed = inner[:args.steps]
        clocks = sampler.stop() if rank == 0 else None
        if clocks is not None:
            clocks["window"] = "warm-up + timed region, %.1f s under load" % (time.time() - t_load)
        info = sg.ctx.info()
        launches_per_step = info.kernel_launches
        device_ms_inner = ranks.max_over_ranks(sum(inner_timed) / max(len(inner_timed), 1))
        directory, owner = sg.directory()
        import numpy as np
        V = int(directory["vertex_count"].sum()); I = int(directory["index_count"].sum())
        TV = int(directory["trans_vertex_count"].sum()); TI = int(directory["trans_index_count"].sum())
        d0, dup, bm, bo = algorithmic_bytes(n, info.levels_total, V, I, TV, TI)
        bytes_alg_total = d0 + dup + bm + bo
        ach = bytes_alg_total / (ms_step * 1e-3) / 1e9
        per_rank_blocks = [int((owner == r).sum()) for r in range(world)]
        per_rank_verts = [int(directory["vertex_count"][owner == r].sum()) for r in range(world)]
        roofline = {"bound": "hbm", "kernel": "whole step (every kernel + both exchanges of one vxb_polygonize_sharded on every rank)", "achieved": ach,
                    "peak": peak * world, "unit": "GB/s", "frac": ach / (peak * world), "traffic": None, "peak_source": peak_src + " x %d GPUs" % world,
                    "algorithmic_bytes_per_step": bytes_alg_total, "ms_per_step": ms_step}
        config = {"workload": "%d^3 seeded Perlin terrain, ONE grid over %d GPUs (strong scaling), all LOD levels + transition cells" % (n, world),
                  "grid": ("dense int8 distance + uint8 material + uint8 blend, read-only, resident in EVERY rank's HBM (3 GiB at 1024^3): every kernel load is local" if args.shard_mode == "replicated"
                           else "dense int8 distance + uint8 material + uint8 blend; z-pieces of %d planes dealt cyclically to the ranks' HBM, mapped into every peer over NVLink" % sg.group_planes),
                  "sharding": "work dealt by blocks: every rank scans 1/N of the layers; exchange 0 = ncclAllGather of the per-block info; super-blocks cut by surface weight; exchange 1 = peer stores of material pages + a device-side barrier over the mapped buffers; coarse levels classified by every rank; output stays on the rank",
                  "l2": "inputs larger than the 126 MB L2; no flush", "vertices": V, "indices": I, "transition_vertices": TV, "transition_indices": TI,
                  "blocks_emitted": int(len(directory)), "blocks_per_rank": per_rank_blocks, "vertices_per_rank": per_rank_verts, "nccl_ranks": world,
                  "host_binding": "every rank pinned to the CPUs of its GPU's NUMA node (rank 0: node %s)" % numa_node}
        # every rank's geometry digest equals the single-GPU result?  (cheap version inside the bench: directory self-consistency;
        # the bit-exact multi-GPU comparison lives in tools/bench_sharded.py --verify and tests/test_gpu_sharded.py)
        key = directory["level"].astype(np.int64) * (1 << 32) + directory["coord_id"]
        parity = {"checked": True, "what": "merged directory strictly ordered by (level, coord_id) with every block owned by exactly one rank",
                  "mismatches": int((np.diff(key) <= 0).sum())}

        # -- e2e: every rank uploads ITS pieces from the same PackForSave blob in pinned host memory, barrier, step, own result back --
        if not args.no_e2e:
            blob_t = None
            if rank == 0:
                ctxp = voxels_b200.Context(local_rank)
                ctxp.fill(n, capi.Surface.terrain(n))
                blob_t = torch.from_numpy(ctxp.pack())
                ctxp.close()
            size_t = torch.tensor([blob_t.numel() if rank == 0 else 0], dtype=torch.int64, device=dev)
            ranks.td.broadcast(size_t, src=0)
            blob_dev = torch.empty(int(size_t.item()), dtype=torch.uint8, device=dev)
            if rank == 0:
                blob_dev.copy_(blob_t)
            ranks.td.broadcast(blob_dev, src=0)
            h_blob = blob_dev.cpu().pin_memory()
            del blob_dev
            blob_bytes = int(h_blob.numel())
            out = {
                "verts": torch.empty(int(info.vertex_span * 1.2) * 48 + 4096, dtype=torch.uint8).pin_memory(),
                "idx": torch.empty(int(info.index_span * 1.2) * 4 + 4096, dtype=torch.uint8).pin_memory(),
                "tverts": torch.empty(int(info.trans_vertex_span * 1.2) * 48 + 4096, dtype=torch.uint8).pin_memory(),
                "tidx": torch.empty(int(info.trans_index_span * 1.2) * 4 + 4096, dtype=torch.uint8).pin_memory(),
            }
            into = {k: v.data_ptr() for k, v in out.items()}
            moved = [0, 0]

            def step_e2e():
                if args.shard_mode == "cube":
                    ranks.barrier()                                   # no peer still reads the pieces this upload overwrites
                sg.upload_packed(h_blob.data_ptr(), blob_bytes)       # replicated: the whole grid; cube: this rank's pieces only
                if args.shard_mode == "cube":
                    ranks.barrier()                                   # every piece resident before any rank reads its peers'
                rc = sg.ctx.polygonize_sharded(3, flags)
                if rc != 0:
                    raise RuntimeError("arena overflow inside the timed region")
                i2 = sg.ctx.info()
                sg.ctx.download(into=into)
                moved[1] = i2.block_count * 128 + i2.vertex_span * 48 + i2.index_span * 4 + i2.trans_vertex_span * 48 + i2.trans_index_span * 4

            esteps = max(3, min(args.steps, 5))
            for _ in range(3):
                step_e2e()
            ms_e2e = timed(step_e2e, esteps, stream)
            d2h_total = ranks.sum_over_ranks(moved[1])
            e2e = {"value": float(n) ** 3 / (ms_e2e * 1e-3) / 1e6, "unit": "Mvoxels/s", "ms_per_step": ms_e2e, "steps": esteps,
                   "h2d_bytes_per_step": blob_bytes * (world if args.shard_mode == "replicated" else 1), "d2h_bytes_per_step": int(d2h_total),
                   "path": "per rank: vxb_grid_upload_packed (pinned host -> HBM, RLE decode on the GPU; replicated: the whole grid over the rank's own PCIe link, cube: its pieces), "
                           "vxb_polygonize_sharded, vxb_result_download of its own blocks; bytes are the sums over the ranks"}
            del out, h_blob
        sg.close()
        sharding_note = "strong scaling: the SAME %d^3 grid on every N" % n
        scaling = "strong"

        # -- extra: the independent-tiles mode (one n^3 tile per rank, no data-path collective): weak scaling --
        if not args.no_tiles:
            ctxt = voxels_b200.Context(local_rank)
            ctxt.fill(n, capi.Surface.terrain(n, origin=tile_origin(rank, n)))
            st = torch.cuda.ExternalStream(ctxt.L.vxb_stream(ctxt.h), device=dev)
            for _ in range(3):
                ctxt.polygonize(0, flags)
            ms_t = timed(lambda: ctxt.polygonize(0, flags), max(3, min(args.steps, 5)), st)
            extra["independent_tiles"] = {"value": whole_job_throughput(n, world, ms_t), "unit": "Mvoxels/s", "ms_per_step": ms_t, "scaling": "weak",
                                          "what": "one %d^3 terrain tile per rank, no data-path collective (round 1's line)" % n}
            ctxt.close()

    # ---------------------------------------------------------------- second record: BASELINE configs[3], 2048^3 (one grid over N GPUs)
    if not args.no_config4:
        try:
            n4 = 2048
            torch.cuda.empty_cache()
            import numpy as np
            if world > 1:
                sg4 = ShardedGrid(ranks, n4, key="c4-%s" % os.environ.get("MASTER_PORT", "0"), mode=args.shard_mode)
                sg4.fill(capi.Surface.terrain(n4))
                sg4.ready()
                st4 = torch.cuda.ExternalStream(sg4.ctx.stream(), device=dev)
                for _ in range(3):
                    i4 = sg4.polygonize(flags)

                def step4():
                    if sg4.ctx.polygonize_sharded(3, flags) != 0:
                        raise RuntimeError("arena overflow inside the timed region")
            else:
                sg4 = voxels_b200.Context(local_rank)
                sg4.fill(n4, capi.Surface.terrain(n4))
                st4 = torch.cuda.ExternalStream(sg4.L.vxb_stream(sg4.h), device=dev)
                for _ in range(3):
                    i4 = sg4.polygonize(0, flags)

                def step4():
                    sg4.polygonize(0, flags)

            s4 = max(3, min(args.steps, 5))
            ms4 = timed(step4, s4, st4)
            if world > 1:
                dir4, own4 = sg4.directory()
            else:
                dir4 = sg4.download().records
                own4 = np.zeros(len(dir4), np.int32)
            V4 = int(dir4["vertex_count"].sum()); I4 = int(dir4["index_count"].sum())
            TV4 = int(dir4["trans_vertex_count"].sum()); TI4 = int(dir4["trans_index_count"].sum())
            a4 = sum(algorithmic_bytes(n4, i4.levels_total, V4, I4, TV4, TI4))
            extra["config4_2048"] = {"metric": "Mvoxels/s polygonized", "value": float(n4) ** 3 / (ms4 * 1e-3) / 1e6, "unit": "Mvoxels/s", "ms_per_step": ms4, "steps": s4,
                                     "n_gpus": world, "scaling": "strong", "workload": "2048^3 seeded Perlin terrain, ONE grid over %d GPU(s), all 8 LOD levels + transition cells" % world,
                                     "blocks_emitted": int(len(dir4)), "blocks_per_rank": [int((own4 == r).sum()) for r in range(world)],
                                     "roofline": {"achieved": a4 / (ms4 * 1e-3) / 1e9, "peak": peak * world, "frac": a4 / (ms4 * 1e-3) / 1e9 / (peak * world), "unit": "GB/s",
                                                  "algorithmic_bytes_per_step": a4}}
            sg4.close()
        except Exception as exc:  # the headline line must still be printed
            extra["config4_2048"] = {"value": None, "error": repr(exc)[:300]}
            try:
                ranks.max_over_ranks(0.0)
            except Exception:
                pass

    value = float(n) ** 3 / (ms_step * 1e-3) / 1e6
    if rank == 0:
        line = {
            "metric": "Mvoxels/s polygonized", "value": value, "unit": "Mvoxels/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
            "dtype": "int8 samples / fp32 vertices", "data": "synthetic", "config": config,
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "parity": parity, "clocks": clocks,
            "gpu_launches": int(launches_per_step * args.steps), "device_ms_per_step_inner": device_ms_inner, "extra": extra,
        }
        if sharding_note:
            line["config"]["scaling_note"] = sharding_note
        print(json.dumps(line))
    ranks.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
