"""Cost of the batch statistics on one GPU: device time of end_batch, kernel time and achieved bytes/s of its
accumulate pass (48 B of algorithmic traffic per bin-major tally entry: batch value read, zero written back,
S1 and S2 read and written), and whether the move after end_batch is slower than a move after a move (the
pass streams its arrays with L2::evict_first so the tet records stay in L2).  Device-resident moves, fixed
kernel (auto-tuner off), c2 with 1 bin and the c5 per-GPU share with 8 score bins.
Usage: python scripts/exp_batch_stats.py OUTDIR [pairs]   (writes OUTDIR/exp_batch_stats.jsonl)"""
import json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from pumiumtally_b200.tally import PumiTally
from pumiumtally_b200.workload import CONFIGS, SyntheticWorkload

outdir = sys.argv[1]
pairs = int(sys.argv[2]) if len(sys.argv) > 2 else 12
os.makedirs(outdir, exist_ok=True)
out = open(os.path.join(outdir, "exp_batch_stats.jsonl"), "w")


def emit(rec):
    print(json.dumps(rec), flush=True)
    out.write(json.dumps(rec) + "\n")
    out.flush()


assert torch.cuda.is_available(), "needs a CUDA device"
hw = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                    capture_output=True, text=True).stdout.strip()
emit({"hardware": hw, "torch_device": torch.cuda.get_device_name(0)})
dev = torch.device("cuda", 0)
stream = torch.cuda.current_stream().cuda_stream

for cfg_name, n, nbins in (("c2", CONFIGS["c2"]["particles"], 1),
                           ("c5", CONFIGS["c5"]["particles"] // CONFIGS["c5"]["gpus"], 8)):
    cfg = CONFIGS[cfg_name]
    cells = cfg["cells"]
    wl = SyntheticWorkload(box=tuple(float(c) for c in cells), num_particles=n, mean_length=cfg["mean_length"],
                           mu_min=cfg["mu_min"], backend="torch", device=dev)
    eng = PumiTally.from_spec(f"box:{cells[0]},{cells[1]},{cells[2]}", n, device=0)
    eng.set_option("autotune", 0)
    if nbins > 1:
        eng.set_score_bins(nbins)
    eng.copy_initial_position_device(wl.initial_positions().contiguous().data_ptr(), stream)
    gen = torch.Generator(device=dev)
    gen.manual_seed(5)

    def move():
        o, d, f, w = (x.contiguous() for x in wl.next_step())
        if nbins > 1:
            b = torch.randint(-1, nbins, (n,), dtype=torch.int32, device=dev, generator=gen)
            eng.move_device_binned(o.data_ptr(), d.data_ptr(), f.data_ptr(), w.data_ptr(), b.data_ptr(), stream)
        else:
            eng.move_device(o.data_ptr(), d.data_ptr(), f.data_ptr(), w.data_ptr(), stream)
        torch.cuda.synchronize()

    def timed_move():
        k0 = eng.stats()["kernel_ms"]
        move()
        return eng.stats()["kernel_ms"] - k0

    flux_len = nbins * eng.num_elements
    for _ in range(3):  # warm-up: kernels, the first end_batch allocates the accumulators
        move()
        eng.end_batch()
    after_batch, after_move, end_ms = [], [], []
    for k in range(pairs):
        for order in ((0, 1) if k % 2 == 0 else (1, 0)):  # alternate which of the two comes first
            move()
            if order == 0:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                eng.end_batch()  # returns after its pass has finished on the device
                end_ms.append(1e3 * (time.perf_counter() - t0))
                after_batch.append(timed_move())
            else:
                after_move.append(timed_move())
    # kernel time of the accumulate pass, from a profiled window of its own
    from torch.profiler import ProfilerActivity, profile
    move()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            eng.end_batch()
    acc = [e for e in prof.key_averages() if "batch_accumulate_kernel" in e.key]
    acc_us = (acc[0].device_time_total / acc[0].count) if acc else float("nan")
    med = lambda v: round(float(np.median(v)), 4)
    spread = lambda v: round(float(np.percentile(v, 90) - np.percentile(v, 10)), 4)
    emit({"config": cfg_name, "particles": n, "score_bins": nbins, "tets": eng.num_elements, "flux_len": flux_len,
          "variant": eng.get_option("variant"), "pairs": pairs,
          "end_batch_ms_median": med(end_ms), "end_batch_ms_min": round(min(end_ms), 4),
          "accumulate_kernel_us": round(acc_us, 2),
          "accumulate_algorithmic_bytes": 48 * flux_len,
          "accumulate_achieved_TBps": round(48 * flux_len / (acc_us * 1e-6) / 1e12, 3) if acc else None,
          "move_kernel_ms_after_end_batch_median": med(after_batch), "move_kernel_ms_after_move_median": med(after_move),
          "move_kernel_ms_after_end_batch_p10_p90_spread": spread(after_batch),
          "move_kernel_ms_after_move_p10_p90_spread": spread(after_move),
          "move_kernel_ms_after_end_batch": [round(x, 4) for x in after_batch],
          "move_kernel_ms_after_move": [round(x, 4) for x in after_move]})
    del eng, wl
    torch.cuda.empty_cache()
out.close()
