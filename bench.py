#!/usr/bin/env python
"""bench.py -- Mvoxels/s to converged min-cut (BASELINE.json metric) on the headline workload.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--size S] [--no-extras] [--dump-outputs DIR]

A "step" is one complete pass of the hot path over one synthetic volume: graph build (n-link stencil, regional
t-links, markers, solver state -- one fused kernel) -> max-flow to convergence -> mask + energy.  Workload
(config.workload): BASELINE config 3, a 512^3 fp32 two-blob volume with regional_probability_map t-links +
boundary_difference_exponential (sigma = RMS neighbour difference), fg ball / bg shell markers (SURVEY.md §8d).

  value    : N_voxels * K / t, inputs resident in HBM, t = CUDA events around the K timed steps (max over ranks)
  e2e      : same metric through the public API (medpy_b200.graphcut.graph_from_voxels -> maxflow -> get_mask)
             from pinned HOST buffers, H2D and D2H inside the timed region
  roofline : the dominant kernel by device time (k_build_tile, the fused graph build): algorithmic bytes per launch /
             its CUDA-event time, measured live; `traffic` = its DRAM bytes per launch from the committed ncu capture.
             `roofline_maxflow` = the max-flow phase (global relabels + push passes + stop tests): measured DRAM bytes
             of those kernels (same capture) / their live device time.  Same choice at every N (rank 0's slab).
  mask_sha256 : sha256 of the full uint8 mask of the last timed step, at every N, next to the committed hash of the
             REFERENCE solver's mask on this workload (tests/golden/bench_mask_sha256.json; pinned by
             tests/test_gpu_fullsize.py) -- `mask_matches_reference`
  config.extra : the other BASELINE configs, measured once each outside the timed region of the headline:
             N = 1: config 2 (256^3 boundary only), config 4 (256x256x128x4, 4-D), config 5 on ONE GPU (its oracle);
             N > 1: config 5 (1024^3) z-slab partitioned over the N GPUs
  cpu_baseline: the reference's BK solver (oracle/_ref, real reference sources) timed on a bounded 256^3 sample of the
             same generator on the host, 1 thread (BK is serial)

`--dump-outputs DIR` writes what the last timed step returned -- energy and mask -- as .npy files (see output_arrays); the
inputs are generated from a fixed seed, so two builds run with the same arguments can be compared output for output.

`--impl reference` times the reference's CPU path on the SAME 512^3 instance (numpy terms + C++ graph fill + BK maxflow +
read-out; ~40 s and ~40 GB of host memory per step, so at most 2 steps are measured whatever K says -- stated in the line).
N > 1: the volume is z-slab partitioned over the ranks (one process per GPU, NCCL halo exchange of border
heights / pushed flow); same total work => "scaling": "strong".
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time



def _cpu_quota():
    """CPUs this process may actually use: the cgroup quota (cpu.max) when there is one, else the affinity mask.  The GPU box
    shows 128 logical CPUs to a 16-CPU container; numpy / torch worker pools sized for 128 spin past the quota and the
    kernel's CFS throttling then stalls EVERY thread of the process for up to 100 ms (measured: e2e steps of 27 ms with
    outliers of 80-290 ms), so the pools are capped before those libraries are imported."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


CPU_QUOTA = _cpu_quota()
for _k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS"):
    os.environ.setdefault(_k, str(max(1, min(8, CPU_QUOTA // 2))))

import numpy  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "Mvoxels/sec to min-cut"
UNIT = "Mvoxels/s"
B_ALG = 11  # algorithmic bytes / voxel of config 3: image 4 + prob 4 + fg 1 + bg 1 + mask 1 (SURVEY.md §8d)
DUMP_SAMPLE = 1 << 22  # mask voxels --dump-outputs draws (float32 values + float64 indices: 48 MB at most)


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi sampled DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.path = tempfile.mktemp(suffix=".csv")
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=self.f,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        for line in open(self.path):
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1])); mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        note = "nvidia-smi -lms 20 from the start of the warm-up steps to the end of the timed steps"
        if not sm:
            # the whole region can be shorter than nvidia-smi's start-up: one query right after it, GPU still hot
            try:
                line = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                      capture_output=True, text=True, timeout=10).stdout.strip().splitlines()[0]
                parts = [x.strip() for x in line.split(",")]
                sm.append(float(parts[1])); mx.append(float(parts[2]))
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
                note = "timed region shorter than nvidia-smi's start-up; single query immediately after it"
            except Exception:
                pass
        return {"sm_mhz": float(numpy.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "how": note}


def make_volume(size):
    from medpy_b200 import synthetic
    shape = (size, size, size)
    t0 = time.time()
    vol = synthetic.two_blob_volume(shape, seed=0)
    vol["shape"] = shape
    vol["gen_s"] = time.time() - t0
    return vol


# ------------------------------------------------------------------------------------------------------
# CPU arm: the reference's BK on the host
# ------------------------------------------------------------------------------------------------------
def cpu_reference_run(size, repeats=1):
    """Times the reference's CPU path on a bounded sample: a `size`^3 volume from the same generator, same terms.
    Graph construction uses the oracle's vectorised numpy restatement + a bulk C fill (far faster than the
    reference's per-edge Python loop, ~1 us/edge, SURVEY.md §6), so the number flatters the reference."""
    from oracle import energy_terms as et
    from oracle import solvers
    vol = make_volume(size)
    n = int(numpy.prod(vol["shape"]))
    best = None
    for _ in range(repeats):
        t0 = time.time()
        prob = et.build_problem(vol["fg"], vol["bg"], regional=(vol["prob"], vol["alpha"]),
                                boundary=("difference_exponential", vol["image"], vol["sigma"], False))
        t1 = time.time()
        if solvers.have_ref():
            flow, mask, tm = solvers.solve_ref(prob)
            kind = "reference"
            fill, mf, ro = tm["fill_s"], tm["maxflow_s"], tm["readout_s"]
        else:
            flow, mask, tm = solvers.solve_port(prob)
            kind = "port"
            fill, mf, ro = tm["setup_s"], tm["maxflow_s"], 0.0
        total = (t1 - t0) + fill + mf + ro
        r = dict(kind=kind, n=n, terms_s=t1 - t0, fill_s=fill, maxflow_s=mf, readout_s=ro, total_s=total,
                 energy=flow, fg_voxels=int(mask.sum(dtype=numpy.int64)), mask_sha256=sha256_of(mask))
        if best is None or r["total_s"] < best["total_s"]:
            best = r
    return best


def workload_text(size, sigma=None):
    t = ("BASELINE config 3: %d^3 fp32 two-blob volume, regional_probability_map (alpha 0.1) + boundary_difference_exponential "
         "(sigma = RMS neighbour difference), fg balls / bg shell" % size)
    return t


def cpu_baseline_obj(r, size, workload_size):
    frac = (float(size) / workload_size) ** 3
    return {
        "value": r["n"] / r["total_s"] / 1e6, "unit": UNIT, "cores": 1, "kind": r["kind"],
        "sample": "%d^3 two-blob volume, same generator and terms as the workload (%s of its voxels); "
                  "numpy terms %.2fs + C++ graph fill %.2fs + BK maxflow() %.2fs + read-out %.2fs"
                  % (size, "all" if frac >= 1.0 else "1/%d" % round(1.0 / frac), r["terms_s"], r["fill_s"], r["maxflow_s"], r["readout_s"]),
        "maxflow_only_value": r["n"] / max(r["maxflow_s"], 1e-9) / 1e6,
        "host_cores_available": os.cpu_count(), "host_cpu_quota": CPU_QUOTA,
    }


def output_arrays(energy, mask):
    """The energy and the mask of one step as the arrays --dump-outputs writes, each to <name>.npy:
      energy.npy             float64 [1]   the min-cut energy maxflow() returned
      mask_fg_per_plane.npy  float64 [S0]  foreground voxels per index of the first axis (covers the whole mask)
      mask_sample.npy        float32 [k]   mask values (1 = foreground) at
      mask_sample_index.npy  float64 [k]   flat C-order voxel indices: every voxel of a mask of at most DUMP_SAMPLE voxels,
                                           else the sorted distinct draws of DUMP_SAMPLE uniform indices from a fixed seed"""
    mask = numpy.asarray(mask)
    flat = mask.reshape(-1)
    if flat.size <= DUMP_SAMPLE:
        idx = numpy.arange(flat.size)
    else:
        idx = numpy.unique(numpy.random.default_rng(0).integers(0, flat.size, size=DUMP_SAMPLE))
    return {"energy": numpy.asarray([energy], dtype=numpy.float64),
            "mask_fg_per_plane": mask.reshape(mask.shape[0], -1).sum(axis=1, dtype=numpy.int64).astype(numpy.float64),
            "mask_sample": flat[idx].astype(numpy.float32),
            "mask_sample_index": idx.astype(numpy.float64)}


def committed_mask_hash(key="config3_512"):
    try:
        return json.load(open(os.path.join(ROOT, "tests", "golden", "bench_mask_sha256.json")))[key]["sha256"]
    except Exception:
        return None


def sha256_of(arr):
    import hashlib
    return hashlib.sha256(numpy.ascontiguousarray(arr, dtype=numpy.uint8).tobytes()).hexdigest()


def run_reference_arm(args):
    """The reference's own CPU implementation of the path on the SAME instance as the GPU arm (same_config): numpy terms,
    C++ graph fill, BK maxflow(), what_segment read-out -- oracle/_ref = lib/maxflow/src compiled in place.  One step at
    512^3 is ~40 s and ~40 GB of host memory, so the number of measured steps is capped (config.steps_measured)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    size = args.cpu_size if args.cpu_size else args.size
    cap = 2 if size >= 384 else (5 if size >= 200 else args.steps)
    steps = max(1, min(args.steps, cap))
    warm = 0 if size >= 384 else max(0, min(args.warmup, 1))
    for _ in range(warm):
        cpu_reference_run(size)
    t0 = time.time()
    rs = [cpu_reference_run(size) for _ in range(steps)]
    dt = time.time() - t0
    n = rs[0]["n"]
    total = sum(r["total_s"] for r in rs)
    value = n * len(rs) / total / 1e6
    best = min(rs, key=lambda r: r["total_s"])
    cb = cpu_baseline_obj(best, size, args.size)
    cb["value"] = value
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / len(rs), "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_text(size), "shape": [size] * 3, "state_dtype": "float64", "parallelism": "single",
                   "solver": "reference BK (lib/maxflow/src, -O2 -DNDEBUG), 1 host thread (BK is serial)"
                             if best["kind"] == "reference" else "oracle BK port",
                   "steps_measured": len(rs), "warmup_measured": warm,
                   "steps_note": "one step = the whole %d^3 instance on one host core; capped at %d measured steps so the arm "
                                 "finishes within minutes" % (size, cap),
                   "energy": best["energy"], "fg_voxels": best["fg_voxels"], "mask_sha256": best.get("mask_sha256"),
                   "wall_s": dt},
        "cpu_baseline": cb,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out))
    return 0


# ------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------
def traffic_table():
    """DRAM bytes per launch / per step from the committed `ncu --set full` capture of this workload (profiles/)."""
    for name in ("r02_traffic_512cubed.json", "r01_traffic_512cubed.json"):
        try:
            t = json.load(open(os.path.join(ROOT, "profiles", name)))
            t["_file"] = "profiles/" + name
            return t
        except Exception:
            continue
    return {}


BUILD_BYTES_PER_VOXEL = 79    # k_build_tile: image 4 + prob 4 + fg 1 + bg 1 read; 6 caps 48 + tr 8 + excess 8 + label 4 + rmask 1 written
BUILD_BYTES_NOREG = 75        # ... without the regional term (no probability map)


def rooflines(stats_list, n_local, n_global, peak, peak_kind, regional=True):
    """`roofline`: k_build_tile (dominant kernel by device time).  `roofline_maxflow`: the max-flow phase."""
    k = max(len(stats_list), 1)
    tt = traffic_table()
    ms_build = sum(s["ms_boundary"] for s in stats_list) / k
    bpv = BUILD_BYTES_PER_VOXEL if regional else BUILD_BYTES_NOREG
    alg = n_local * bpv
    ach = alg / (ms_build * 1e-3) / 1e9 if ms_build > 0 else 0.0
    per_launch = tt.get("bytes_per_launch", {})
    traffic = per_launch.get("k_build_tile") if n_local == 512 ** 3 else None
    ms_rel = sum(s["ms_relabel"] for s in stats_list) / k
    ms_push = sum(s["ms_push"] for s in stats_list) / k
    ms_solve = sum(s["ms_solve"] for s in stats_list) / k
    ms_read = sum(s["ms_readout"] for s in stats_list) / k
    share = {"k_build_tile_ms": ms_build, "relabel_ms": ms_rel, "push_ms": ms_push, "solve_ms": ms_solve, "readout_ms": ms_read,
             "note": "device ms per step from the library's CUDA events (mgc_stats); solve = relabels + pushes + stop tests"}
    roof = {"bound": "hbm", "kernel": "k_build_tile (fused graph build: n-link stencil + t-links + markers + solver state)",
            "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic, "peak_kind": peak_kind,
            "launches": k, "avg_launch_ms": ms_build, "algorithmic_bytes_per_launch": alg,
            "algorithmic_bytes_per_voxel": bpv, "traffic_source": tt.get("_file"), "share_of_step": share}
    mf_bytes = tt.get("maxflow_phase_bytes_per_step") if n_global == 512 ** 3 and n_local == n_global else None
    mf = {"bound": "hbm", "kernel": "max-flow phase: k_bfs_coop / k_relabel_reset / k_sweep_* (global relabel) + k_push_tile_tma + k_count_active_tiles",
          "measured_dram_bytes_per_step": mf_bytes, "ms_per_step": ms_solve,
          "achieved": (mf_bytes / (ms_solve * 1e-3) / 1e9) if (mf_bytes and ms_solve > 0) else None, "peak": peak, "unit": "GB/s",
          "frac": (mf_bytes / (ms_solve * 1e-3) / 1e9 / peak) if (mf_bytes and ms_solve > 0) else None,
          "note": "worklist kernels touch only active tiles: the phase is latency-bound (grid barriers, tile visits), not bandwidth-bound; "
                  "bytes are MEASURED dram__bytes of those launches (ncu), time is live"}
    return roof, mf


def run_gpu_arm(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    torch.set_num_threads(max(1, min(8, CPU_QUOTA // max(1, min(world, 8)) // 2 or 1)))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    size = args.size
    shape = (size, size, size)
    n = int(numpy.prod(shape))
    peak, peak_kind = measured_peak()

    extras = {}
    if world > 1:
        from medpy_b200 import distributed as mdist
        result = mdist.bench_slab(shape, args, rank, world, local_rank)   # each rank builds only its own planes
        vol = {"sigma": result["sigma"]}
        if not args.no_extras:
            extras["config5_1024cubed_zslab%d" % world] = mdist.bench_config5(args, rank, world, local_rank)
    else:
        vol = make_volume(size)
        result = bench_single(vol, args, torch)
        del vol["image"], vol["prob"], vol["fg"], vol["bg"]
        if not args.no_extras:
            extras = run_extras_single(torch, peak)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    ref_hash = committed_mask_hash() if size == 512 else None
    out = {
        "metric": METRIC, "value": result["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": result["ms_per_step"], "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_text(size), "shape": list(shape), "state_dtype": "float64",
                   "parallelism": "zslab%d" % world if world > 1 else "single", "sigma": vol["sigma"],
                   "l2": "inputs (%.1f GB) and solver state (%.1f GB) exceed the 126 MB L2; no flush needed"
                         % (n * 10 / 1e9, n * 70 / 1e9),
                   "energy": result.get("energy"), "fg_voxels": result.get("fg_voxels"),
                   "mask_sha256": result.get("mask_sha256"), "reference_mask_sha256": ref_hash,
                   "mask_matches_reference": (result.get("mask_sha256") == ref_hash) if ref_hash else None,
                   "push_sweeps_per_step": result.get("push_sweeps"), "global_relabels_per_step": result.get("global_relabels"),
                   "relabel_sweeps_per_step": result.get("relabel_sweeps"),
                   "hbm_read_roofline_frac": (n * B_ALG / (result["ms_per_step"] * 1e-3)) / (peak * 1e9 * world),
                   "hbm_read_roofline_note": "N*%d B / t_step / (%s peak %.0f GB/s * n_gpus), SURVEY.md §8d" % (B_ALG, peak_kind, peak),
                   "extra": extras},
        "clocks": result["clocks"],
        "e2e": result["e2e"],
        "gpu_launches": result["gpu_launches"],
        "roofline": result["roofline"],
        "roofline_maxflow": result["roofline_maxflow"],
    }
    if world == 1 and not args.no_cpu_baseline:
        csize = args.cpu_size if args.cpu_size else 256
        r = cpu_reference_run(csize)
        out["cpu_baseline"] = cpu_baseline_obj(r, csize, size)
    if args.dump_outputs:
        outputs = result["outputs"] if world == 1 else output_arrays(result["energy"], result["mask"])
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in outputs.items():
            numpy.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()
    return 0


def resident_run(torch, vol, boundary, regional, steps, warmup):
    """One BASELINE configuration with its inputs resident in HBM: `warmup` untimed + `steps` timed passes (CUDA events).
    Returns (ms per step, energy, mask tensor, per-step stats)."""
    from medpy_b200.graphcut.device import graph_from_device_arrays
    stream = torch.cuda.current_stream()
    d_img = torch.from_numpy(vol["image"]).cuda()
    d_prob = torch.from_numpy(vol["prob"]).cuda() if regional else None
    d_fg = torch.from_numpy(vol["fg"].view(numpy.uint8)).cuda()
    d_bg = torch.from_numpy(vol["bg"].view(numpy.uint8)).cuda()
    d_mask = torch.empty(vol["image"].shape, dtype=torch.uint8, device="cuda")
    graph = None
    stats = []

    def step(record):
        nonlocal graph
        graph = graph_from_device_arrays(d_fg, d_bg, image=d_img, boundary=boundary, sigma=vol["sigma"],
                                         prob=d_prob, alpha=vol.get("alpha"), graph=graph, stream=stream.cuda_stream)
        e = graph.maxflow()
        graph._nat().get_mask_into(d_mask.data_ptr())
        if record:
            stats.append(graph.stats())
        return e

    for _ in range(warmup):
        step(False)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    energy = None
    for _ in range(steps):
        energy = step(True)
    ev1.record(stream)
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1) / steps, energy, d_mask, stats


def run_extras_single(torch, peak):
    """BASELINE configs 2, 4 and 5 (on one GPU: the oracle of the 8-GPU run), each once, outside the headline's timed region."""
    from medpy_b200 import synthetic
    out = {}
    todo = [("config2_256cubed_difference_exponential", (256, 256, 256), "difference_exponential", False),
            ("config4_256x256x128x4_maximum_exponential", (256, 256, 128, 4), "maximum_exponential", True),
            ("config5_1024cubed_single_gpu", (1024, 1024, 1024), "difference_exponential", False)]
    for name, shape, boundary, fourd in todo:
        try:
            t0 = time.time()
            vol = synthetic.multispectral_volume(shape, seed=0) if fourd else synthetic.two_blob_volume(shape, seed=0, with_prob=False)
            gen_s = time.time() - t0
            big = int(numpy.prod(shape)) >= 2 ** 29
            ms, energy, d_mask, stats = resident_run(torch, vol, boundary, False, steps=2, warmup=1)
            n = int(numpy.prod(shape))
            st = stats[-1]
            mask = d_mask.cpu().numpy()
            out[name] = {"shape": list(shape), "value": n / (ms * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": ms, "steps": 2, "warmup": 1,
                         "energy": energy, "fg_voxels": int(mask.sum(dtype=numpy.int64)), "mask_sha256": sha256_of(mask),
                         "hbm_read_roofline_frac": (n * 7 / (ms * 1e-3)) / (peak * 1e9),
                         "push_sweeps": st["push_sweeps"], "global_relabels": st["global_relabels"], "relabel_sweeps": st["relabel_sweeps"],
                         "ms_build": st["ms_boundary"], "ms_relabel": st["ms_relabel"], "ms_push": st["ms_push"], "ms_solve": st["ms_solve"],
                         "gen_s": gen_s, "sigma": vol["sigma"]}
            if name.startswith("config5"):
                ref5 = committed_mask_hash("config5_1024")
                out[name]["single_gpu_mask_sha256_committed"] = ref5
                out[name]["mask_matches_committed"] = (out[name]["mask_sha256"] == ref5) if ref5 else None
            del d_mask, mask, vol
            torch.cuda.empty_cache()
            if big:
                import gc as _gc
                _gc.collect()
        except Exception as exc:      # an extra must never take the headline line down with it
            out[name] = {"error": "%s: %s" % (type(exc).__name__, exc)}
            torch.cuda.empty_cache()
    return out


def bench_single(vol, args, torch):
    import medpy_b200.graphcut as gc
    shape = vol["shape"]
    n = int(numpy.prod(shape))
    peak, peak_kind = measured_peak()

    sampler = ClockSampler(torch.cuda.current_device())
    sampler.start()
    ms, energy, d_mask, stats = resident_run(torch, vol, "difference_exponential", True, steps=args.steps, warmup=args.warmup)
    clocks = sampler.stop()
    mask_host = d_mask.cpu().numpy()
    fg_vox = int(mask_host.sum(dtype=numpy.int64))
    mask_hash = sha256_of(mask_host)
    outputs = output_arrays(energy, mask_host) if args.dump_outputs else None
    del d_mask, mask_host
    value = n / (ms * 1e-3) / 1e6
    launches = int(sum(s["kernel_launches"] for s in stats))
    roof, roof_mf = rooflines(stats, n, n, peak, peak_kind)
    torch.cuda.empty_cache()

    # ---- end to end through the public API from pinned host buffers ----
    def pin(a):
        t = torch.from_numpy(numpy.ascontiguousarray(a)).pin_memory()
        return t, t.numpy()
    keep = [pin(vol["image"]), pin(vol["prob"]), pin(vol["fg"].view(numpy.uint8)), pin(vol["bg"].view(numpy.uint8))]
    h_img, h_prob, h_fg, h_bg = (k[1] for k in keep)
    h_fg = h_fg.view(numpy.bool_)
    h_bg = h_bg.view(numpy.bool_)

    def e2e_step():
        g = gc.graph_from_voxels(h_fg, h_bg, regional_term=gc.energy_voxel.regional_probability_map,
                                 regional_term_args=(h_prob, vol["alpha"]),
                                 boundary_term=gc.energy_voxel.boundary_difference_exponential,
                                 boundary_term_args=(h_img, vol["sigma"], False))
        e = g.maxflow()
        m = g.get_mask()
        return e, m

    # warm-up in the steady-state shape: the previous step's mask is still referenced while the next step runs (as in
    # the timed loop), so the pinned read-back pool already holds the two buffers that pattern needs
    e2e_warm = max(2, min(args.warmup, 3))
    for _ in range(e2e_warm):
        e_e2e, m_e2e = e2e_step()
    torch.cuda.synchronize()
    per_step = []
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ts = time.perf_counter()
        e_e2e, m_e2e = e2e_step()
        per_step.append(1e3 * (time.perf_counter() - ts))
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    e2e = {"value": n * args.steps / dt / 1e6, "unit": UNIT, "h2d_bytes_per_step": int(n * 10), "d2h_bytes_per_step": int(n + 8),
           "ms_per_step": 1e3 * dt / args.steps, "step_ms_min_median_max": [min(per_step), float(numpy.median(per_step)), max(per_step)],
           "api": "medpy_b200.graphcut.graph_from_voxels -> maxflow -> get_mask",
           "energy_matches_resident_run": bool(abs(e_e2e - energy) <= 1e-12 * abs(energy)),
           "mask_matches_resident_run": bool(sha256_of(m_e2e) == mask_hash),
           "timer": "host perf_counter around synchronised steps (the z-chunked H2D uploads and the D2H mask copy are inside)"}
    del m_e2e, keep
    return {"value": value, "ms_per_step": ms, "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
            "roofline": roof, "roofline_maxflow": roof_mf, "energy": energy, "fg_voxels": fg_vox, "mask_sha256": mask_hash,
            "outputs": outputs,
            "push_sweeps": stats[-1]["push_sweeps"], "global_relabels": stats[-1]["global_relabels"],
            "relabel_sweeps": stats[-1]["relabel_sweeps"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--size", type=int, default=int(os.environ.get("MEDPY_BENCH_SIZE", "512")))
    ap.add_argument("--cpu-size", type=int, default=int(os.environ.get("MEDPY_BENCH_CPU_SIZE", "0")),
                    help="edge of the CPU arm's volume; 0 = the workload's own size for --impl reference, 256 for the cpu_baseline object")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip config.extra (configs 2, 4, 5)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the energy and mask of the last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_gpu_arm(args)


if __name__ == "__main__":
    sys.exit(main())
