"""End-to-end MoveToNextLocation from host memory (config c2): staged path (default) for several
worker counts and chunk sizes, pageable vs pinned caller buffers, vs the direct path.
Usage: python scripts/exp_e2e.py [mode ...]   mode = staged:<threads>:<chunk> | pinned_staged:<threads>:<chunk> |
                                                     direct_registered | direct_pageable | direct_pinned"""
import sys, os, json, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from pumiumtally_b200.tally import PumiTally
from pumiumtally_b200.workload import CONFIGS, SyntheticWorkload

if os.environ.get("EXP_BIND") == "1":  # like `numactl --cpunodebind=<GPU's node>`: host arrays end up next to the GPU
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from bench import bind_to_gpu_node
    print("bound to", len(bind_to_gpu_node(torch, 0) or []), "CPUs", flush=True)
cfgname = os.environ.get("EXP_CONFIG", "c2")
cfg = CONFIGS[cfgname]; cells = cfg["cells"]; n = int(os.environ.get("EXP_PARTICLES", cfg["particles"]))
box = tuple(float(c) for c in cells)
wl = SyntheticWorkload(box=box, num_particles=n, mean_length=cfg["mean_length"], mu_min=cfg["mu_min"], backend="torch", device="cuda")
init = wl.initial_positions().cpu().numpy()
NB = int(os.environ.get("EXP_STEPS", 8))
batches = [tuple(x.cpu().numpy() for x in wl.next_step()) for _ in range(NB)]
modes = sys.argv[1:] or ["staged:0:0", "pinned_staged:0:0", "direct_registered", "direct_pinned"]
for mode in modes:
    parts = mode.split(":")
    kind = parts[0]
    eng = PumiTally.from_spec(f"box:{cells[0]},{cells[1]},{cells[2]}", n, device=0)
    if kind in ("staged", "pinned_staged"):
        if len(parts) > 1 and int(parts[1]) > 0: eng.set_option("host_threads", int(parts[1]))
        if len(parts) > 2 and int(parts[2]) > 0: eng.set_option("chunk", int(parts[2]))
    else:
        eng.set_option("host_path", 0)
        eng.set_option("register_host", 1 if kind == "direct_registered" else 0)
    t0 = time.perf_counter()
    eng.CopyInitialPosition(init.reshape(-1))
    t_init = time.perf_counter() - t0
    if kind in ("pinned_staged", "direct_pinned"):
        bufs = [torch.empty(s, dtype=d, pin_memory=True) for s, d in ((3 * n, torch.float64), (3 * n, torch.float64), (n, torch.int8), (n, torch.float64))]
        O, D, F, W = (b.numpy() for b in bufs)
    else:
        O, D, F, W = np.empty(3 * n), np.empty(3 * n), np.empty(n, dtype=np.int8), np.empty(n)
    times, ret, host_us, sent, copy_us = [], [], [], [], []
    s0 = eng.stats()["segments"]
    for o, d, f, w in batches:
        O[:], D[:], F[:], W[:] = o.reshape(-1), d.reshape(-1), f, w
        t0 = time.perf_counter()
        eng.MoveToNextLocation(O, D, F, W)
        t1 = time.perf_counter()
        segs = eng.stats()["segments"]
        times.append(time.perf_counter() - t0); ret.append(t1 - t0)
        host_us.append(eng.get_option("stage_host_us")); sent.append(eng.get_option("stage_sent_bytes")); copy_us.append(eng.get_option("stage_copy_us"))
    ms = 1e3 * np.median(times[2:])
    print(json.dumps({"mode": mode, "config": cfgname, "n": n, "ms_per_move_median": round(ms, 2), "ms_all": [round(1e3 * t, 2) for t in times],
                      "call_return_ms": round(1e3 * np.median(ret[2:]), 2), "init_ms": round(1e3 * t_init, 1),
                      "stage_host_us": int(np.median(host_us[2:])), "stage_copy_us": int(np.median(copy_us[2:])), "sent_MB": round(np.median(sent[2:]) / 1e6, 1),
                      "threads": eng.get_option("host_threads"), "host_node": eng.get_option("host_node"), "chunk": eng.get_option("chunk"),
                      "gseg_s": round((segs - s0) / len(batches) / ms / 1e6, 2)}), flush=True)
    del eng
