"""z-slab multi-GPU graph cut: one process per GPU, ``torch.distributed`` (NCCL over NVLink) for the plumbing.

The global lattice is split into contiguous slabs along axis 0; rank r owns planes ``[z0, z1)`` and keeps one
ghost plane per interior side.  Arcs crossing a slab border belong to their tail voxel; a push across the
border parks the flow in the ghost plane (the rank's outbox) and the neighbour receives, per exchange, the
border plane's labels (int32) and the parked flow (float64) -- one message per direction -- and adds the flow
to the excess of its border voxel and to the residual of the reverse arc (SURVEY.md §8e).  Labels used across a
border are one exchange stale, which keeps every push feasible but not the labelling valid; correctness rests
on the stop test only: after an EXACT distributed global relabel (local BFS to a fixed point <-> border label
exchange, repeated until no ghost label changes anywhere), no voxel with excess has a finite label.

The stepping primitives are the ``mgc_slab_*`` entry points of the C ABI; this module only sequences them and
moves the border messages.  ``handle_factory`` lets the CPU test-suite drive the same code over gloo with a
numpy stand-in for the device handle (tests/fake_slab.py).
"""
import math
import os

import numpy

KINDS = {
    "difference_linear": 0, "difference_exponential": 1, "difference_division": 2, "difference_power": 3,
    "maximum_linear": 4, "maximum_exponential": 5, "maximum_division": 6, "maximum_power": 7,
}


def slab_bounds(extent, world, rank):
    """Planes [z0, z1) of axis 0 owned by ``rank``: as even as possible, never empty for world <= extent."""
    return (rank * extent) // world, ((rank + 1) * extent) // world


def _native_factory(shape, z0, z1, device):
    from . import _lib
    return _lib.Graph(list(shape), int(z0), int(z1), int(device))


class SlabSolver:
    """One rank's share of a z-slab partitioned graph cut."""

    def __init__(self, shape, rank=None, world=None, device=None, handle_factory=None, group=None,
                 passes0=1, passes_max=8):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.group = group
        self.rank = dist.get_rank(group) if rank is None else rank
        self.world = dist.get_world_size(group) if world is None else world
        self.shape = tuple(int(s) for s in shape)
        if len(self.shape) < 3:
            raise ValueError("z-slab partitioning needs a lattice with at least 3 axes")
        if self.world > self.shape[0]:
            raise ValueError("more ranks than axis-0 planes")
        self.z0, self.z1 = slab_bounds(self.shape[0], self.world, self.rank)
        self.ghost_lo = self.z0 > 0
        self.ghost_hi = self.z1 < self.shape[0]
        self.lo_peer = self.rank - 1 if self.ghost_lo else None
        self.hi_peer = self.rank + 1 if self.ghost_hi else None
        self.native = handle_factory is None
        if self.native:
            self.device_index = torch.cuda.current_device() if device is None else int(device)
            self.tdev = torch.device("cuda", self.device_index)
            self.handle = _native_factory(self.shape, self.z0, self.z1, self.device_index)
            self.handle.set_stream(torch.cuda.current_stream(self.tdev).cuda_stream)
            # the solve runs inside the library over its own NCCL communicator (mgc_slab_solve); torch.distributed only
            # carries the 128-byte unique id.  MEDPY_GC_SLAB_HOST_LOOP=1 keeps the round-1 Python-sequenced loop (A/B).
            self.native_loop = self.world > 1 and os.environ.get("MEDPY_GC_SLAB_HOST_LOOP", "0") != "1"
            if self.native_loop:
                box = [type(self.handle).slab_comm_unique_id() if self.rank == 0 else None]
                dist.broadcast_object_list(box, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
                self.handle.slab_comm_init(self.rank, self.world, box[0])
        else:
            self.tdev = torch.device("cpu")
            self.handle = handle_factory(self.shape, self.z0, self.z1)
        self.plane = int(self.handle.slab_plane_elems())
        # one message per direction: [labels int32 x P | pad to 8 B | flow float64 x P]
        self.h_bytes = (self.plane * 4 + 7) // 8 * 8
        self.msg_bytes = self.h_bytes + self.plane * 8
        mk = lambda: torch.zeros(self.msg_bytes, dtype=torch.uint8, device=self.tdev)
        self.send_lo, self.send_hi, self.recv_lo, self.recv_hi = mk(), mk(), mk(), mk()
        # [ghost label changed in round A, ... in round B, active voxels]: written by the handle's kernels, all-reduced
        self.stat3 = torch.zeros(3, dtype=torch.int64, device=self.tdev)
        self.passes0, self.passes_max = int(passes0), int(passes_max)
        self.stats = {"exchanges": 0, "relabel_rounds": 0, "global_relabels": 0, "push_passes": 0}

    # ---------------------------------------------------------------------------------------------- data
    def local_slice(self, arr):
        """The part of a global array this rank needs: its planes plus the ghost planes (1-plane overlap, so the
        n-link stencil needs no communication)."""
        a = self.z0 - (1 if self.ghost_lo else 0)
        b = self.z1 + (1 if self.ghost_hi else 0)
        return arr[a:b]

    def owned_of_local(self, arr):
        a = 1 if self.ghost_lo else 0
        return arr[a:a + (self.z1 - self.z0)]

    def reset(self):
        self.handle.reset()

    def add_regional_probability(self, prob_local, alpha, compute_f32=True):
        self.handle.add_regional_probability(prob_local, float(alpha), bool(compute_f32))

    def add_boundary(self, kind, image_local, sigma=None, spacing=False, norm=math.nan):
        k = KINDS[kind] if isinstance(kind, str) else int(kind)
        sp = [float(s) for s in spacing] if spacing else None
        self.handle.add_boundary(k, image_local, 0.0 if sigma is None else float(sigma), sp, float(norm))

    def add_markers(self, fg_local, bg_local):
        self.handle.add_markers(fg_local, bg_local)

    def build(self, fg_local, bg_local, image_local=None, kind=None, sigma=None, spacing=False, prob_local=None, alpha=None,
              norm=math.nan, compute_f32=True):
        """Everything graph_from_voxels adds (regional term, boundary term, fg / bg markers) in one native call: the
        fused single-pass build of the slab (mgc_build_voxel_graph)."""
        k = -1 if kind is None else (KINDS[kind] if isinstance(kind, str) else int(kind))
        sp = [float(s) for s in spacing] if spacing else None
        self.handle.build_voxel_graph(prob_local, 0.0 if alpha is None else float(alpha), bool(compute_f32) and prob_local is not None,
                                      k, image_local, 0.0 if sigma is None else float(sigma), sp, float(norm), fg_local, bg_local)

    # ---------------------------------------------------------------------------------------------- messages
    def _views(self, buf):
        h = buf[: self.plane * 4].view(self.torch.int32)
        f = buf[self.h_bytes:].view(self.torch.float64)
        return h, f

    def _ptr(self, t):
        return t.data_ptr() if self.native else t

    def exchange(self, changed=None):
        """pack -> send/recv with both neighbours -> unpack; everything is enqueued on the stream, the host never
        waits.  ``changed``: one-element device tensor the unpack kernel sets to 1 if a ghost label changed."""
        torch, dist = self.torch, self.dist
        hl, fl = self._views(self.send_lo)
        hh, fh = self._views(self.send_hi)
        self.handle.slab_pack(self._ptr(hl) if self.ghost_lo else 0, self._ptr(fl) if self.ghost_lo else 0,
                              self._ptr(hh) if self.ghost_hi else 0, self._ptr(fh) if self.ghost_hi else 0)
        ops = []
        if self.ghost_lo:
            ops.append(dist.P2POp(dist.isend, self.send_lo, self.lo_peer, self.group))
            ops.append(dist.P2POp(dist.irecv, self.recv_lo, self.lo_peer, self.group))
        if self.ghost_hi:
            ops.append(dist.P2POp(dist.isend, self.send_hi, self.hi_peer, self.group))
            ops.append(dist.P2POp(dist.irecv, self.recv_hi, self.hi_peer, self.group))
        if ops:
            for req in dist.batch_isend_irecv(ops):
                req.wait()
        rhl, rfl = self._views(self.recv_lo)
        rhh, rfh = self._views(self.recv_hi)
        self.handle.slab_unpack(self._ptr(rhl) if self.ghost_lo else 0, self._ptr(rfl) if self.ghost_lo else 0,
                                self._ptr(rhh) if self.ghost_hi else 0, self._ptr(rfh) if self.ghost_hi else 0,
                                self._ptr(changed) if changed is not None else 0)
        self.stats["exchanges"] += 1

    def _allreduce(self, value, op):
        t = self.torch.tensor([value], dtype=self.torch.int64, device=self.tdev)
        self.dist.all_reduce(t, op=op, group=self.group)
        return int(t.item())

    # ---------------------------------------------------------------------------------------------- solve
    def global_relabel(self):
        """Exact distributed backward BFS + stop test.  Returns the global number of active voxels afterwards.

        A round = local BFS to a fixed point, then a border-label exchange whose unpack raises a device flag if a ghost
        label changed.  Almost every relabel needs exactly two rounds (one that moves labels across the borders, one that
        confirms nothing moves any more), so two rounds and the active count are enqueued speculatively and checked with
        ONE all-reduce + host synchronisation: [changed in round A, changed in round B, active voxels].  The count is
        valid iff round B changed nothing anywhere; otherwise two more rounds follow."""
        dist = self.dist
        self.handle.slab_relabel_begin()
        st = self.stat3
        while True:
            st.zero_()
            for k in (0, 1):
                self.handle.slab_relabel_relax(False)
                self.exchange(changed=st[k:k + 1])
                self.stats["relabel_rounds"] += 1
            self.handle.slab_count_active_dev(self._ptr(st[2:3]))
            if self.world > 1:
                dist.all_reduce(st, op=dist.ReduceOp.SUM, group=self.group)
            vals = st.tolist()                       # the one host synchronisation
            if vals[1] == 0:
                break
        self.stats["global_relabels"] += 1
        return int(vals[2])

    def solve(self, max_rounds=100000):
        """Run to a maximum preflow.  Returns this rank's energy share; use ``energy()`` for the total."""
        self.stats = {"exchanges": 0, "relabel_rounds": 0, "global_relabels": 0, "push_passes": 0}   # per solve
        self.energy_total = None
        if self.native and getattr(self, "native_loop", False):
            self.energy_total = float(self.handle.slab_solve())
            self.stats = dict(self.handle.slab_solve_stats())
            self.energy_part = None
            return self.energy_total
        self.handle.slab_begin()
        passes = self.passes0
        rounds = 0
        while True:
            if self.global_relabel() == 0:
                break
            rounds += 1
            if rounds > max_rounds:
                raise RuntimeError("push-relabel did not converge within the round cap")
            for _ in range(passes):
                self.handle.slab_push(1)
                self.exchange()
                self.stats["push_passes"] += 1
            passes = min(self.passes_max, passes * 2)
        self.energy_part = float(self.handle.slab_finish())
        return self.energy_part

    def energy(self):
        """Total min-cut energy (float64 all-reduce of the per-slab parts)."""
        if getattr(self, "energy_total", None) is not None:
            return self.energy_total
        t = self.torch.tensor([self.energy_part], dtype=self.torch.float64, device=self.tdev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM, group=self.group)
        return float(t.item())

    def mask(self):
        """uint8 mask of the OWNED planes (host array)."""
        return self.handle.get_mask()


def graphcut_slab(fg_markers, bg_markers, image=None, boundary=None, sigma=None, spacing=False, prob=None, alpha=None,
                  norm=math.nan, gather=True, group=None, handle_factory=None):
    """Public multi-GPU entry point: every rank passes the SAME global arrays (host or device); each takes its
    slab, the ranks solve one global min cut together.  Returns ``(energy, mask)``; with ``gather`` the full mask
    is assembled on every rank (all_gather of the slabs), otherwise only the rank's own planes are returned."""
    import torch
    import torch.distributed as dist
    shape = tuple(fg_markers.shape)
    s = SlabSolver(shape, group=group, handle_factory=handle_factory)
    if boundary is not None and boundary.endswith("linear") and (isinstance(norm, float) and math.isnan(norm)):
        raise ValueError("linear boundary terms need the GLOBAL normaliser `norm` in slab mode")
    s.build(s.local_slice(fg_markers), s.local_slice(bg_markers),
            image_local=s.local_slice(image) if boundary is not None else None, kind=boundary, sigma=sigma, spacing=spacing,
            prob_local=s.local_slice(prob) if prob is not None else None, alpha=alpha, norm=norm,
            compute_f32=prob is not None and "float32" in str(prob.dtype))
    s.solve()
    energy = s.energy()
    own = s.mask()
    if not gather or s.world == 1:
        return energy, own
    # slabs may differ by one plane: pad to the largest, gather, trim
    counts = [slab_bounds(shape[0], s.world, r) for r in range(s.world)]
    pmax = max(b - a for a, b in counts)
    dev = s.tdev
    pad = torch.zeros((pmax,) + shape[1:], dtype=torch.uint8, device=dev)
    pad[: own.shape[0]] = torch.from_numpy(numpy.ascontiguousarray(own)).to(dev)
    parts = [torch.empty_like(pad) for _ in range(s.world)]
    dist.all_gather(parts, pad, group=group)
    full = numpy.concatenate([p[: b - a].cpu().numpy() for p, (a, b) in zip(parts, counts)], axis=0)
    return energy, full


# ------------------------------------------------------------------------------------------------------
# bench support (bench.py --gpus N, launched with torchrun)
# ------------------------------------------------------------------------------------------------------
def slab_volume(shape, rank, world, seed=0, with_prob=True):
    """This rank's planes (+ ghost planes) of the synthetic two-blob workload and the GLOBAL sigma: every rank
    generates only what it needs (the generator seeds each plane separately) and the per-plane partial sums of the
    RMS neighbour difference are all-gathered and added with fsum, so sigma is bit-identical to the single-process
    value whatever the partition."""
    import torch
    import torch.distributed as dist
    from . import synthetic
    z0, z1 = slab_bounds(shape[0], world, rank)
    a = z0 - (1 if z0 > 0 else 0)
    b = z1 + (1 if z1 < shape[0] else 0)
    vol = synthetic.two_blob_volume(shape, seed=seed, planes=(a, b), with_prob=with_prob)
    own = vol["image"][z0 - a: z0 - a + (z1 - z0)]
    nxt = vol["image"][z1 - a] if z1 < shape[0] else None
    parts = synthetic.neighbour_difference_partials(own, next_plane=nxt)
    pmax = max(slab_bounds(shape[0], world, r)[1] - slab_bounds(shape[0], world, r)[0] for r in range(world))
    dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu")
    buf = torch.zeros(pmax, dtype=torch.float64, device=dev)
    buf[: parts.size] = torch.from_numpy(parts).to(dev)
    allp = [torch.empty_like(buf) for _ in range(world)]
    dist.all_gather(allp, buf)
    vals = []
    for r, t in enumerate(allp):
        c0, c1 = slab_bounds(shape[0], world, r)
        vals.extend(t[: c1 - c0].cpu().tolist())
    vol["sigma"] = float(math.sqrt(math.fsum(vals) / synthetic.neighbour_pair_count(shape)))
    vol["shape"] = tuple(shape)
    return vol


def gather_mask(s, d_mask_own, shape):
    """Full uint8 mask on rank 0 (None elsewhere): the owned planes of every rank, gathered over NCCL."""
    import torch
    import torch.distributed as dist
    counts = [slab_bounds(shape[0], s.world, r) for r in range(s.world)]
    pmax = max(b - a for a, b in counts)
    pad = torch.zeros((pmax,) + tuple(shape[1:]), dtype=torch.uint8, device=d_mask_own.device)
    pad[: d_mask_own.shape[0]] = d_mask_own
    parts = [torch.empty_like(pad) for _ in range(s.world)] if s.rank == 0 else None
    dist.gather(pad, parts, dst=0)
    if s.rank != 0:
        return None
    return numpy.concatenate([p[: b - a].cpu().numpy() for p, (a, b) in zip(parts, counts)], axis=0)


def _slab_resident(shape, rank, world, local_rank, regional, steps, warmup, sampler=None):
    """z-slab run with the slab inputs resident in HBM: every timed step rebuilds the graph (fused build), solves and
    extracts the mask.  Timing: CUDA events between barriers, max over ranks."""
    import torch
    import torch.distributed as dist
    dev = torch.device("cuda", local_rank)
    vol = slab_volume(shape, rank, world, with_prob=regional)
    s = SlabSolver(shape, rank=rank, world=world, device=local_rank)
    d_img = torch.from_numpy(numpy.ascontiguousarray(vol["image"])).to(dev)
    d_prob = torch.from_numpy(numpy.ascontiguousarray(vol["prob"])).to(dev) if regional else None
    d_fg = torch.from_numpy(numpy.ascontiguousarray(vol["fg"]).view(numpy.uint8)).to(dev)
    d_bg = torch.from_numpy(numpy.ascontiguousarray(vol["bg"]).view(numpy.uint8)).to(dev)
    d_mask = torch.empty((s.z1 - s.z0,) + tuple(shape[1:]), dtype=torch.uint8, device=dev)
    launches, build_ms = [], []

    def step():
        s.reset()
        s.build(d_fg, d_bg, image_local=d_img, kind="difference_exponential", sigma=vol["sigma"], prob_local=d_prob,
                alpha=vol.get("alpha"))
        s.solve()
        s.handle.get_mask_into(d_mask.data_ptr())
        return s.energy()

    if sampler is not None and rank == 0:
        sampler.start()
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    dist.barrier()
    stream = torch.cuda.current_stream()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    dist.barrier()
    ev0.record(stream)
    energy = None
    for _ in range(steps):
        energy = step()
        st = s.handle.stats()
        launches.append(st["kernel_launches"])
        build_ms.append(st["ms_boundary"])
    ev1.record(stream)
    torch.cuda.synchronize()
    dist.barrier()
    ms = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item()) / steps
    clocks = sampler.stop() if (sampler is not None and rank == 0) else None
    fgv = torch.tensor([int(d_mask.sum().item())], dtype=torch.int64, device=dev)
    dist.all_reduce(fgv)
    nl = torch.tensor([int(sum(launches))], dtype=torch.int64, device=dev)
    dist.all_reduce(nl)
    full = gather_mask(s, d_mask, shape)
    return dict(s=s, vol=vol, ms=ms, energy=energy, clocks=clocks, fg_voxels=int(fgv.item()), launches=int(nl.item()),
                build_ms=build_ms, mask=full, d_mask=d_mask)


def bench_slab(shape, args, rank, world, local_rank):
    """Strong-scaling run of bench.py's workload: the volume is partitioned once, the slab inputs stay resident
    in HBM, each timed step rebuilds the graph, solves and extracts the mask.  Returns the dict bench.py prints
    (meaningful on rank 0), with the last timed step's full host mask under "mask" (rank 0; None elsewhere)."""
    import time
    import torch
    import torch.distributed as dist
    from bench import ClockSampler, measured_peak, rooflines, sha256_of, UNIT  # noqa
    dev = torch.device("cuda", local_rank)
    n = int(numpy.prod(shape))
    r = _slab_resident(shape, rank, world, local_rank, True, args.steps, args.warmup, sampler=ClockSampler(local_rank))
    s, vol, ms, energy = r["s"], r["vol"], r["ms"], r["energy"]
    mask_hash = sha256_of(r["mask"]) if rank == 0 else None
    peak, peak_kind = measured_peak()
    del r["d_mask"]
    torch.cuda.empty_cache()

    # ---- end to end: pinned host slabs -> device -> solve -> host mask ----
    def pin(a):
        t = torch.from_numpy(numpy.ascontiguousarray(a)).pin_memory()
        return t, t.numpy()
    keep = [pin(vol["image"]), pin(vol["prob"]), pin(vol["fg"].view(numpy.uint8)), pin(vol["bg"].view(numpy.uint8))]
    h_img, h_prob, h_fg, h_bg = (k[1] for k in keep)

    def e2e_step():
        s.reset()
        s.build(h_fg, h_bg, image_local=h_img, kind="difference_exponential", sigma=vol["sigma"], prob_local=h_prob, alpha=vol["alpha"])
        s.solve()
        m = s.mask()
        return s.energy(), m

    for _ in range(2):
        e_e2e, _m = e2e_step()
    torch.cuda.synchronize()
    dist.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e_e2e, _m = e2e_step()
    torch.cuda.synchronize()
    dist.barrier()
    dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    dt = float(dt.item())
    local_bytes = int(numpy.prod(h_img.shape)) * 10
    e2e = {"value": n * args.steps / dt / 1e6, "unit": UNIT, "h2d_bytes_per_step": int(n * 10 + (world - 1) * 2 * s.plane * 10),
           "d2h_bytes_per_step": int(n + 8 * world), "ms_per_step": 1e3 * dt / args.steps,
           "api": "medpy_b200.distributed.SlabSolver (reset/build/solve/mask) per rank", "energy_matches_resident_run": bool(e_e2e == energy),
           "timer": "host perf_counter between barriers, max over ranks", "rank0_h2d_bytes": local_bytes}
    # same kernel choice as at N = 1: the fused build, here on rank 0's slab (library CUDA events around each launch)
    n_local = int(numpy.prod(vol["image"].shape))
    stats_like = [{"ms_boundary": b, "ms_relabel": 0.0, "ms_push": 0.0, "ms_solve": 0.0, "ms_readout": 0.0} for b in r["build_ms"]]
    roof, roof_mf = rooflines(stats_like, n_local, n, peak, peak_kind)
    roof["kernel"] += " on rank 0's slab"
    phases_all = [None] * world
    dist.all_gather_object(phases_all, s.stats.get("phase_ms"))
    roof["share_of_step"] = {"k_build_tile_ms": roof["avg_launch_ms"], "step_ms": ms, "exchanges_cumulative": s.stats["exchanges"],
                             "phase_ms_last_step_per_rank": phases_all,
                             "rank0_phase_ms_last_step": s.stats.get("phase_ms"),
                             "note": "phase_ms: device time of rank 0's last solve per phase (CUDA events inside mgc_slab_solve): local BFS, "
                                     "border exchanges (pack + ncclSend/Recv + unpack), stop test (count + all-reduce), push passes, read-out; "
                                     "host_blocked_ms = host time in the per-round stream synchronisations"}
    roof_mf["ms_per_step"] = None
    return {"value": n / (ms * 1e-3) / 1e6, "ms_per_step": ms, "clocks": r["clocks"], "e2e": e2e,
            "gpu_launches": r["launches"], "roofline": roof, "roofline_maxflow": roof_mf, "energy": energy, "fg_voxels": r["fg_voxels"],
            "mask_sha256": mask_hash, "mask": r["mask"],
            "push_sweeps": s.stats["push_passes"], "global_relabels": s.stats["global_relabels"],
            "relabel_sweeps": s.stats["relabel_rounds"], "sigma": vol["sigma"]}


def bench_config5(args, rank, world, local_rank, shape=(1024, 1024, 1024)):
    """BASELINE config 5: 1024^3 fp32, boundary_difference_exponential, z-slab partitioned over the ranks.  One warm-up
    and two timed steps; the gathered mask is hashed on rank 0 (compare with the single-GPU run's config.extra)."""
    import torch
    from bench import measured_peak, sha256_of, committed_mask_hash, UNIT  # noqa
    try:
        r = _slab_resident(shape, rank, world, local_rank, False, 2, 1)
    except Exception as exc:
        return {"error": "%s: %s" % (type(exc).__name__, exc)}
    n = int(numpy.prod(shape))
    peak, _ = measured_peak()
    s = r["s"]
    out = {"shape": list(shape), "value": n / (r["ms"] * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": r["ms"], "steps": 2, "warmup": 1,
           "energy": r["energy"], "fg_voxels": r["fg_voxels"], "mask_sha256": sha256_of(r["mask"]) if rank == 0 else None,
           "hbm_read_roofline_frac": (n * 7 / (r["ms"] * 1e-3)) / (peak * 1e9 * world), "n_gpus": world,
           "push_passes": s.stats["push_passes"], "global_relabels": s.stats["global_relabels"], "exchanges": s.stats["exchanges"],
           "sigma": r["vol"]["sigma"]}
    ref5 = committed_mask_hash("config5_1024") if tuple(shape) == (1024, 1024, 1024) else None
    out["single_gpu_mask_sha256_committed"] = ref5
    out["mask_matches_single_gpu"] = (out["mask_sha256"] == ref5) if (ref5 and rank == 0) else None
    del r
    torch.cuda.empty_cache()
    return out
