#!/usr/bin/env python
"""Headline benchmark: particle-segments/s of the MoveToNextLocation hot path.

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA engine
  python bench.py --impl reference --gpus N --steps K ...  # CPU reference arm (oracle port)

A "step" is one MoveToNextLocation over one synthetic batch of BASELINE.json's
config c2 (998,250-tet Kuhn box, 10M particles per GPU; SURVEY.md section 8d).
Per-GPU work is fixed as N grows (weak scaling); every rank holds the whole
mesh (full-buffer picpart) and its own particle stripe, and the per-rank
tallies are summed once at batch end inside the timed region (ncclAllReduce, or
ncclReduceScatter to the owners of the element shares with the gather deferred
to read time -- whichever the engine measured to be quicker on this mesh when
the communicator was set up).  One JSON line is printed by rank 0.

`value` is device-resident throughput; `e2e` is the same metric through the
reference-facing call on pageable host arrays (host->device copies inside the
timed region).  At N = 2, 4, 8 the line also carries `extra` blocks for the
multi-GPU configurations BASELINE.json names: `c4_x4` (1 M long tracks on 4
GPUs), `c5_x8` (100 M particles on the 9.86 M-tet mesh, 8 GPUs) and
`c5_strong_x2/4` (the same 100 M particles on fewer GPUs: strong scaling).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

T_START = time.time()
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "particle_segments_per_sec"
UNIT = "segments/s"
# algorithmic bytes (SURVEY.md section 8d): per tallied segment 96 B tet geometry + 16 B
# neighbour ids + 16 B flux read-modify-write; per flying track 61 B read + 28 B written
BYTES_PER_SEGMENT = 128
BYTES_PER_TRACK = 89
# --dump-outputs writes at most this many flux entries and particles (52 MiB of float64 with their
# indices); larger meshes and batches are sampled
DUMP_ELEMENTS = 1 << 21
DUMP_PARTICLES = 1 << 19


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def workload_description(cfg_name, cfg, n):
    c = cfg["cells"]
    return (f"{cfg_name}: Kuhn box {c[0]}x{c[1]}x{c[2]} = {6 * c[0] * c[1] * c[2]} tets, {n} particles/GPU, "
            f"isotropic exp(mean {cfg['mean_length']}) tracks, 95% flying, weights U[0.5,1]")


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def recorded_traffic():
    """DRAM bytes per launch of the walk kernel from the committed ncu capture (not measured in this
    run: dram__bytes needs ncu), with the capture it comes from; or None."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        return {"dram_bytes_per_launch": t["dram_bytes_per_launch"],
                "source": "profiles/traffic.json (%s)" % t.get("source", "ncu capture")}
    except Exception:
        return None


def dump_outputs(out_dir, flux, elem_ids, positions):
    """What a caller reads after the last timed move -- the flux tally and each particle's parent element
    and position -- as float64 DIR/<name>.npy, so that two builds can be compared output for output.
    Arrays longer than DUMP_ELEMENTS / DUMP_PARTICLES are cut to a fixed seeded sample whose indices
    are written beside them."""
    import numpy as np

    def sample(n, k, seed):
        return np.arange(n) if n <= k else np.sort(np.random.default_rng(seed).choice(n, k, replace=False))

    e = sample(len(flux), DUMP_ELEMENTS, 1)
    p = sample(len(elem_ids), DUMP_PARTICLES, 2)
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"flux": flux[e], "flux_element_index": e, "elem_ids": elem_ids[p], "positions": positions[p],
              "particle_index": p}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def bind_to_gpu_node(torch, index):
    """Run this rank (and allocate its host arrays) on the CPUs local to its GPU -- what
    `numactl --cpunodebind` does in an HPC launch line.  Returns the CPU list or None."""
    try:
        p = torch.cuda.get_device_properties(index)
        bus = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        cpus = set()
        for tok in open(f"/sys/bus/pci/devices/{bus}/local_cpulist").read().strip().split(","):
            a, _, b = tok.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if len(cpus) * 4 >= len(os.sched_getaffinity(0)):
            os.sched_setaffinity(0, cpus)
            return sorted(cpus)
    except Exception:
        pass
    return None


def cpu_thread_candidates():
    """Thread counts worth trying for the CPU arm: every hardware thread, one per core, and what the
    container's CPU quota allows (more threads than that only get throttled)."""
    logical = os.cpu_count() or 1
    try:
        import psutil

        physical = psutil.cpu_count(logical=False) or logical
    except Exception:
        physical = logical
    quota = logical
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            quota = max(1, int(round(float(q) / float(per))))
    except Exception:
        pass
    return sorted({logical, physical, min(quota, logical), min(2 * quota, logical)}, reverse=True)


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.thread = index, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=lambda: self.rows.extend(self.proc.stdout), daemon=True)
        self.thread.start()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": "nvidia-smi unavailable"}
        time.sleep(0.15)
        self.proc.terminate()
        self.thread.join(timeout=2)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nme, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------ CPU reference arm

def run_reference(args, rank):
    """Times the reference algorithm's CPU restatement (oracle, OpenMP, all host threads) on a
    bounded sample of the same workload.  The real reference cannot be built offline (needs
    Kokkos/Omega_h/pumi-pic), hence kind = "port"."""
    if rank != 0:
        return
    import numpy as np
    from oracle.oracle import OraclePumiTally, num_threads, set_num_threads
    from pumiumtally_b200.mesh import kuhn_box
    from pumiumtally_b200.workload import CONFIGS, SyntheticWorkload

    cfg = CONFIGS[args.config]
    n = min(args.ref_sample, cfg["particles"])
    coords, t2v = kuhn_box(*cfg["cells"])
    wl = SyntheticWorkload(box=tuple(float(c) for c in cfg["cells"]), num_particles=n,
                           mean_length=cfg["mean_length"], mu_min=cfg["mu_min"])
    orc = OraclePumiTally(coords, t2v, n, per_particle=True)
    orc.CopyInitialPosition(wl.initial_positions().reshape(-1))
    # give the CPU arm the thread count it runs fastest with
    best = None
    for nt in cpu_thread_candidates():
        set_num_threads(nt)
        o, d, f, w = wl.next_step()
        s_before, t0 = orc.n_segments, time.perf_counter()
        orc.MoveToNextLocation(o.reshape(-1), d.reshape(-1), f, w)
        rate = (orc.n_segments - s_before) / (time.perf_counter() - t0)
        if best is None or rate > best[0]:
            best = (rate, nt)
    set_num_threads(best[1])
    for _ in range(max(args.warmup - 2, 0)):
        o, d, f, w = wl.next_step()
        orc.MoveToNextLocation(o.reshape(-1), d.reshape(-1), f, w)
    batches = [wl.next_step() for _ in range(args.steps)]
    s0 = orc.n_segments
    t0 = time.perf_counter()
    for o, d, f, w in batches:
        orc.MoveToNextLocation(o.reshape(-1), d.reshape(-1), f, w)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, orc.flux, orc.elem_ids, orc.positions)
    segs = orc.n_segments - s0
    value = segs / dt
    sample = (f"first {n} particles of the {args.config} batch per step ({args.steps} steps, "
              f"{segs} segments) on the full {len(t2v)}-tet mesh")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(args.steps, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": workload_description(args.config, cfg, cfg["particles"]),
                   "note": "reference-algorithm restatement (OpenMP); the Kokkos/pumi-pic reference cannot be built offline"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": num_threads(), "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------- GPU arm

def exchange_description(eng):
    rs = eng.get_option("exchange_choice") == 1
    return {"collective": "ncclReduceScatter (shares gathered once when the result is read)" if rs else "ncclAllReduce",
            "measured_at_comm_init_ms": {"allreduce": eng.get_option("exchange_allreduce_us") / 1e3,
                                         "reduce_scatter": eng.get_option("exchange_reduce_scatter_us") / 1e3}}


class GpuArm:
    """One rank of the CUDA arm: measures one configuration at a time (device-resident `value`,
    end-to-end `e2e`) with every rank taking part; rank 0 assembles the JSON line."""

    def __init__(self, args, rank, local_rank, world):
        import numpy as np
        import torch

        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the tally engine has no CPU path "
                             "(use --impl reference for the CPU arm)")
        self.np, self.torch = np, torch
        self.args, self.rank, self.local_rank, self.world = args, rank, local_rank, world
        torch.cuda.set_device(local_rank)
        self.dev = torch.device("cuda", local_rank)
        self.all_cpus = os.sched_getaffinity(0)
        self.bound = None if args.no_bind else bind_to_gpu_node(torch, local_rank)
        self.dist = None
        if world > 1:
            import torch.distributed as dist

            dist.init_process_group("nccl", device_id=self.dev)
            self.dist = dist
        self.nccl_id = None

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def reduce(self, values, op):
        t = self.torch.tensor(values, dtype=self.torch.float64, device=self.dev)
        if self.dist is not None:
            self.dist.all_reduce(t, op=getattr(self.dist.ReduceOp, op))
        return [float(x) for x in t]

    def measure(self, cfg_name, n, steps, warmup, e2e=True, e2e_modes=False, clocks=False, scaling="weak",
                dump_dir=None):
        """Device-resident and end-to-end throughput of `cfg_name` with n particles on this rank; with
        dump_dir, rank 0 writes the device-resident engine's results there (dump_outputs)."""
        from pumiumtally_b200.tally import PumiTally
        from pumiumtally_b200.workload import CONFIGS, SyntheticWorkload

        np, torch, args, rank, world, dev = self.np, self.torch, self.args, self.rank, self.world, self.dev
        cfg = CONFIGS[cfg_name]
        cells = cfg["cells"]
        box = tuple(float(c) for c in cells)
        spec = f"box:{cells[0]},{cells[1]},{cells[2]}"
        nsteps = warmup + steps

        def new_engine():
            e = PumiTally.from_spec(spec, n, device=self.local_rank)
            e.set_option("variant", args.variant)  # -1 = the engine's own choice for this mesh
            e.set_option("block", args.block)
            for kv in args.opt:
                k, v = kv.split("=")
                e.set_option(k, int(v))
            return e

        def new_workload():
            w = SyntheticWorkload(box=box, num_particles=n, mean_length=cfg["mean_length"], mu_min=cfg["mu_min"],
                                  backend="torch", device=dev, id_offset=rank * n)
            return w, w.initial_positions().contiguous()

        # identical batches for both arms, generated on the device
        wl, init = new_workload()
        bytes_per_step = n * 57
        pregen = nsteps * bytes_per_step <= args.pregen_gb * (1 << 30)
        # default (c2): all batches are generated up front and the K timed steps run back to back.
        # Configs whose batches do not fit (100M particles) generate each batch just before its step,
        # outside the timed region, and the per-step device times are summed.
        batches = [tuple(x.contiguous() for x in wl.next_step()) for _ in range(nsteps)] if pregen else None
        stream = torch.cuda.current_stream().cuda_stream
        state = {"wl": wl}

        def batch(k):
            return batches[k] if pregen else tuple(x.contiguous() for x in state["wl"].next_step())

        # ---------------- device-resident arm: `value` ------------------------------
        eng = new_engine()
        if world > 1:
            from pumiumtally_b200.distributed import broadcast_unique_id

            eng.comm_init(rank, world, broadcast_unique_id(self.dist, PumiTally.nccl_unique_id, device=dev))
        eng.copy_initial_position_device(init.data_ptr(), stream)
        for k in range(warmup):
            o, d, f, w = batch(k)
            eng.move_device(o.data_ptr(), d.data_ptr(), f.data_ptr(), w.data_ptr(), stream)
        if world > 1 and warmup:
            torch.cuda.current_stream().synchronize()
            eng.exchange_tally()  # the warm-up steps are a batch too: its exchange is outside the timed region
        self.barrier()
        st0 = eng.stats()
        launches0 = eng.get_option("launches")
        sampler = ClockSampler(self.local_rank) if (clocks and rank == 0) else None
        if sampler:
            sampler.start()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        if pregen:
            ev0.record()
            for k in range(warmup, nsteps):
                o, d, f, w = batches[k]
                eng.move_device(o.data_ptr(), d.data_ptr(), f.data_ptr(), w.data_ptr(), stream)
            if world > 1:
                torch.cuda.current_stream().synchronize()
                eng.exchange_tally()  # batch-end exchange of the ghost tallies over NVLink
            ev1.record()
            self.barrier()
            ms = ev0.elapsed_time(ev1)
        else:
            ms = 0.0
            for k in range(warmup, nsteps):
                o, d, f, w = batch(k)
                self.barrier()
                ev0.record()
                eng.move_device(o.data_ptr(), d.data_ptr(), f.data_ptr(), w.data_ptr(), stream)
                if world > 1 and k == nsteps - 1:
                    torch.cuda.current_stream().synchronize()
                    eng.exchange_tally()
                ev1.record()
                torch.cuda.synchronize()
                ms += ev0.elapsed_time(ev1)
                del o, d, f, w
            self.barrier()
        clocks_out = sampler.stop() if sampler else None
        st1 = eng.stats()
        segs, tracks = st1["segments"] - st0["segments"], st1["tracks"] - st0["tracks"]
        kernel_ms = st1["kernel_ms"] - st0["kernel_ms"]
        ms_max = self.reduce([ms], "MAX")[0]
        total_segs, total_tracks = self.reduce([float(segs), float(tracks)], "SUM")
        flux = eng.flux  # collective after a reduce-scatter exchange: every rank reads it
        if dump_dir and rank == 0:
            dump_outputs(dump_dir, flux, eng.elem_ids, eng.positions)
        out = {
            "config": cfg_name, "particles_per_gpu": n, "n_gpus": world, "scaling": scaling, "steps": steps,
            "value": total_segs / (ms_max * 1e-3), "ms_per_step": ms_max / steps,
            "segments_per_track": total_segs / max(total_tracks, 1.0), "lost": int(st1["lost"]),
            "relocation_crossings_per_step": (st1["relocations"] - st0["relocations"]) / max(steps, 1),
            "flux_sum": float(flux.sum()), "variant": eng.get_option("variant"),
            "gpu_launches": eng.get_option("launches") - launches0,  # kernels the engine launched in the timed region
            "allreduce_ms": (eng.get_option("allreduce_us") / 1e3) if world > 1 else None,  # the batch-end exchange
            "allreduce_bytes": 8 * eng.num_elements if world > 1 else None,
            "exchange": exchange_description(eng) if world > 1 else None,
            "pregen": pregen, "clocks": clocks_out, "bytes_per_step": bytes_per_step,
        }
        peak, peak_src = measured_peak()
        alg_bytes = BYTES_PER_SEGMENT * segs + BYTES_PER_TRACK * tracks  # this rank, whole timed region
        achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9 if kernel_ms > 0 else None
        out["roofline"] = {
            "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": (achieved / peak) if achieved else None,
            "kernel": "walk kernel (variant %d%s), %d launches, %.3f ms each" % (
                out["variant"], " incl. binning pass" if out["variant"] in (15, 16, 17, 21, 24, 25, 26) else "", steps,
                kernel_ms / max(steps, 1)),
            "algorithmic_bytes_per_launch": alg_bytes / max(steps, 1), "peak_source": peak_src}
        del eng

        # ---------------- end-to-end arm through the host-pointer C ABI: `e2e` ------
        # Headline: the call a user of the reference makes (PumiTally.h:87-89) on ordinary pageable host
        # arrays that the caller reuses for every move, as OpenMC does with its std::vectors, with the
        # engine's default settings.  Side numbers: the same from pinned buffers, and the direct path
        # (host_path=0) from pageable memory with and without cudaHostRegister.
        def run_e2e(kind, opts, ksteps, kwarm):
            """kind: 'pageable' | 'pinned' caller buffers."""
            if not pregen:  # replay the same counter-based stream from the start
                state["wl"], init2 = new_workload()
            else:
                init2 = init
            if kind == "pinned":
                bufs = [torch.empty(s_, dtype=d_, pin_memory=True).numpy() for s_, d_ in
                        ((3 * n, torch.float64), (3 * n, torch.float64), (n, torch.int8), (n, torch.float64))]
            else:
                bufs = [np.empty(3 * n), np.empty(3 * n), np.empty(n, dtype=np.int8), np.empty(n)]
            O, D, F, W = bufs
            eng2 = new_engine()
            for k_, v_ in opts.items():
                eng2.set_option(k_, v_)
            eng2.CopyInitialPosition(init2.cpu().numpy().reshape(-1))

            def fill(k):  # untimed: the transport code producing its next batch in its own arrays
                o, d, f, w = batch(k)
                for dst, src in zip((O, D, F, W), (o, d, f, w)):
                    dst[:] = src.reshape(-1).cpu().numpy()

            for k in range(kwarm):
                fill(k)
                eng2.MoveToNextLocation(O, D, F, W)
                eng2.stats()
            self.barrier()
            st_a = eng2.stats()
            dt, ret = 0.0, 0.0
            for k in range(kwarm, kwarm + ksteps):
                fill(k)
                t0 = time.perf_counter()
                eng2.MoveToNextLocation(O, D, F, W)
                t1 = time.perf_counter()
                st_b = eng2.stats()  # device->host read of the step's result (synchronises)
                dt += time.perf_counter() - t0
                ret += t1 - t0
            secs = self.reduce([dt], "MAX")[0]
            sg = self.reduce([float(st_b["segments"] - st_a["segments"])], "SUM")[0]
            res = {"value": sg / secs, "ms_per_step": 1e3 * secs / ksteps,
                   "h2d_bytes_per_step": int((st_b["h2d_bytes"] - st_a["h2d_bytes"]) / ksteps),
                   "call_return_ms": 1e3 * ret / ksteps, "host_threads": eng2.get_option("host_threads")}
            del eng2
            return res

        if e2e:
            r = run_e2e("pageable", {}, steps, warmup)
            out["e2e"] = {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": r["h2d_bytes_per_step"],
                          "d2h_bytes_per_step": 56, "ms_per_step": r["ms_per_step"],
                          "call_return_ms": r["call_return_ms"],
                          "caller_buffers": "pageable numpy arrays, reused for every move",
                          "host_threads": r["host_threads"],
                          "note": "MoveToNextLocation(host pointers) with default options + per-step stats read-back; "
                                  "staged path: pinned per-particle slots refilled by the engine's worker pool, "
                                  "only changed origins travel"}
            if e2e_modes and pregen:
                # side numbers: caller arrays the engine may page-lock (register_host=1, what an OpenMC
                # integration sets: its vectors live for the whole run) with the engine choosing between
                # staged and direct uploads; pinned caller arrays; and the direct paths on their own
                kw = min(5, max(nsteps - 1, 0))  # the automatic choice has probed both upload paths after 4 moves
                ks = max(1, min(6, nsteps - kw))
                modes = [("registered_auto", "pageable", {"register_host": 1})]
                if world == 1:
                    modes += [("pinned_buffers", "pinned", {}),
                              ("direct_registered", "pageable", {"host_path": 0, "register_host": 1}),
                              ("direct_pageable", "pageable", {"host_path": 0})]
                out["e2e"]["other_modes"] = {
                    name: {k: v for k, v in run_e2e(kind, opts, ks, kw).items() if k != "host_threads"}
                    for name, kind, opts in modes}
        return out

    def cpu_baseline(self, cfg_name, n, nsteps):
        """The oracle (OpenMP) beside it on a bounded sample (rank 0, N=1 only)."""
        from oracle.oracle import OraclePumiTally, num_threads
        from pumiumtally_b200.mesh import kuhn_box
        from pumiumtally_b200.workload import CONFIGS, SyntheticWorkload

        args = self.args
        os.sched_setaffinity(0, self.all_cpus)  # the CPU arm gets every core of the box
        cfg = CONFIGS[cfg_name]
        cells = cfg["cells"]
        ns = min(args.cpu_sample, n)
        coords, t2v = kuhn_box(*cells)
        orc = OraclePumiTally(coords, t2v, ns, per_particle=True)
        # counter-based generator: the numpy stream of ids [0, ns) is the GPU batch's first ns particles
        wl_cpu = SyntheticWorkload(box=tuple(float(c) for c in cells), num_particles=ns,
                                   mean_length=cfg["mean_length"], mu_min=cfg["mu_min"])
        orc.CopyInitialPosition(wl_cpu.initial_positions().reshape(-1))
        cpu_steps = min(args.cpu_steps, nsteps)
        from oracle.oracle import set_num_threads

        best = None  # the thread count the oracle runs fastest with on this box (untimed trial moves)
        for nt in cpu_thread_candidates():
            set_num_threads(nt)
            o, d, f, w = wl_cpu.next_step()
            s_before, t0 = orc.n_segments, time.perf_counter()
            orc.MoveToNextLocation(o.reshape(-1), d.reshape(-1), f, w)
            rate = (orc.n_segments - s_before) / (time.perf_counter() - t0)
            if best is None or rate > best[0]:
                best = (rate, nt)
        set_num_threads(best[1])
        s0, t_cpu = orc.n_segments, 0.0
        for _ in range(cpu_steps):
            o, d, f, w = wl_cpu.next_step()
            t0 = time.perf_counter()
            orc.MoveToNextLocation(o.reshape(-1), d.reshape(-1), f, w)
            t_cpu += time.perf_counter() - t0
        segs_cpu = orc.n_segments - s0
        return {"value": segs_cpu / t_cpu, "unit": UNIT, "cores": num_threads(), "kind": "port",
                "sample": f"first {ns} particles of {cpu_steps} batches ({segs_cpu} segments, "
                          f"{t_cpu:.1f} s) on the full mesh; reference-algorithm restatement, OpenMP"}


def run_gpu(args, rank, local_rank, world):
    from pumiumtally_b200.workload import CONFIGS

    arm = GpuArm(args, rank, local_rank, world)
    cfg = CONFIGS[args.config]
    # per-GPU particle count: the config's total divided by the GPU count it is quoted on
    n = args.particles or cfg["particles"] // (cfg.get("gpus", 1) if world > 1 else 1)
    if world == 1 and cfg.get("gpus", 1) > 1 and not args.particles:
        n = cfg["particles"] // cfg["gpus"] if args.per_gpu_share else cfg["particles"]
    main = arm.measure(args.config, n, args.steps, args.warmup, e2e=not args.no_e2e,
                       e2e_modes=not args.no_e2e_modes, clocks=True, dump_dir=args.dump_outputs)

    # ---- the multi-GPU configurations BASELINE.json names, measured beside the headline ----------
    # c4 on 4 GPUs (1 M particles / 4), c5 on 8 GPUs (100 M particles / 8), and c5 strong scaling
    # (100 M particles / N on the 9.86 M-tet mesh) at every N > 1.
    extra = {}
    over_budget = arm.reduce([time.time() - T_START], "MAX")[0] > args.extra_after_s
    if over_budget:
        extra["skipped"] = f"headline run took more than {args.extra_after_s} s; extras skipped to stay inside the driver's limit"
    if not args.no_extra and args.config == "c2" and not args.particles and not over_budget:
        ks, kw = min(args.steps, 10), min(args.warmup, 3)
        if world == 4:
            extra["c4_x4"] = arm.measure("c4", CONFIGS["c4"]["particles"] // 4, ks, kw)
        if world in (2, 4, 8):
            tag = "c5_x8" if world == 8 else f"c5_strong_x{world}"
            extra[tag] = arm.measure("c5", CONFIGS["c5"]["particles"] // world, ks, kw, scaling="strong")

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = arm.cpu_baseline(args.config, n, args.warmup + args.steps)
    if arm.dist is not None:
        arm.dist.barrier()
        arm.dist.destroy_process_group()
    if rank != 0:
        return
    traffic = recorded_traffic() if (args.config == "c2" and not args.particles) else None
    roof = dict(main["roofline"])
    roof["traffic"] = traffic["dram_bytes_per_launch"] if traffic else None
    roof["traffic_source"] = traffic["source"] if traffic else None
    line = {
        "metric": METRIC, "value": main["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": main["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_description(args.config, cfg, n), "variant": main["variant"],
                   "block": args.block, "cpu_binding": (f"{len(arm.bound)} CPUs local to the GPU" if arm.bound else "none"),
                   "l2": f"inputs larger than L2 ({main['bytes_per_step'] / 1e6:.0f} MB of fresh particle data per step)",
                   "timing": "K steps back to back between two CUDA events" if main["pregen"] else
                             "per-step CUDA-event times summed (batches generated between steps, untimed)",
                   "parallelism": f"particle stripes x{world}, full-buffer picparts, 1 NCCL exchange of the flux per batch",
                   "segments_per_track": main["segments_per_track"], "lost": main["lost"],
                   "relocation_crossings_per_step": main["relocation_crossings_per_step"],
                   "flux_sum": main["flux_sum"], "allreduce_ms": main["allreduce_ms"],
                   "allreduce_bytes": main["allreduce_bytes"], "exchange": main["exchange"]},
        "roofline": roof,
        "cpu_baseline": cpu,
        "e2e": main.get("e2e"),
        # kernels of this repo inside the timed region: one fused walk kernel per move, plus the five
        # binning kernels (count, 3-kernel scan, scatter) when the binned variant is in use
        "gpu_launches": main["gpu_launches"],
        "clocks": main["clocks"],
    }
    if extra:
        for blk in extra.values():
            blk.pop("clocks", None)
            blk.pop("pregen", None)
        line["extra"] = extra
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2")
    ap.add_argument("--particles", type=int, default=0, help="override particles per GPU (debug only)")
    ap.add_argument("--variant", type=int, default=env_int("PUMITALLY_VARIANT", -1))
    ap.add_argument("--block", type=int, default=env_int("PUMITALLY_BLOCK", 128))
    ap.add_argument("--cpu-sample", type=int, default=2_000_000)
    ap.add_argument("--ref-sample", type=int, default=2_000_000, help="particles per step of the --impl reference arm")
    ap.add_argument("--cpu-steps", type=int, default=5)
    ap.add_argument("--pregen-gb", type=float, default=24.0, help="pre-generate all batches if they fit in this many GiB")
    ap.add_argument("--per-gpu-share", action="store_true",
                    help="on one GPU, run only the per-GPU share of a multi-GPU config")
    ap.add_argument("--opt", action="append", default=[], help="engine option name=value (repeatable)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-e2e-modes", action="store_true", help="skip the e2e side numbers (pinned / direct paths)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-bind", action="store_true", help="do not bind the rank to its GPU's NUMA node")
    ap.add_argument("--extra-after-s", type=float, default=360.0,
                    help="skip the extra blocks when the headline measurement has already taken this long")
    ap.add_argument("--no-extra", action="store_true",
                    help="N>1: skip the extra blocks (c4 on 4 GPUs, c5 on 8 GPUs, c5 strong scaling)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the flux and the particles' elements and positions "
                         "(float64 .npy, seeded samples of large arrays, at most 64 MiB) to DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 0)
    rank, local_rank, world = env_int("RANK", 0), env_int("LOCAL_RANK", 0), env_int("WORLD_SIZE", 1)
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world != args.gpus and args.gpus > 1:
        raise SystemExit(f"--gpus {args.gpus} needs torchrun with {args.gpus} ranks (WORLD_SIZE={world})")
    run_gpu(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
