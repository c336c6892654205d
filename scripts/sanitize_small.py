"""Small end-to-end run of every shipped kernel variant and host path for compute-sanitizer:
   compute-sanitizer --tool memcheck python scripts/sanitize_small.py [variant ...]"""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import numpy as np
from helpers import box_case, run_workload
from oracle.oracle import OraclePumiTally
from pumiumtally_b200.tally import PumiTally

variants = [int(v) for v in sys.argv[1:]] or [8, 16, 24, 0]
for v in variants:
    coords, t2v, wl = box_case((6, 6, 5), 6000)
    e = PumiTally.from_arrays(coords, t2v, wl.n)
    e.set_option("variant", v)
    e.set_option("chunk", 2048)  # several upload/compute ranges, ragged last chunk
    run_workload(e, OraclePumiTally(coords, t2v, wl.n), wl, steps=2, label=f"sanitize v{v}")
    print("variant", v, "staged host path ok", e.stats()["segments"], flush=True)
    # direct host path, device-side state accessors, weight sum, normalisation, page-locked caller arrays
    import torch
    for opts, pinned in (({"host_path": 0}, False), ({}, True)):
        coords, t2v, wl = box_case((6, 6, 5), 5003)
        e, orc = PumiTally.from_arrays(coords, t2v, wl.n), OraclePumiTally(coords, t2v, wl.n)
        e.set_option("variant", v)
        e.set_option("chunk", 1024)
        for k_, v_ in opts.items():
            e.set_option(k_, v_)
        e.set_source_normalization(3)
        init = wl.initial_positions()
        for x in (e, orc):
            x.CopyInitialPosition(init.reshape(-1).copy())
        n = wl.n
        if pinned:
            O, D, F, W = [torch.empty(s_, dtype=d_, pin_memory=True).numpy() for s_, d_ in
                          ((3 * n, torch.float64), (3 * n, torch.float64), (n, torch.int8), (n, torch.float64))]
        else:
            O, D, F, W = np.empty(3 * n), np.empty(3 * n), np.empty(n, dtype=np.int8), np.empty(n)
        for _ in range(3):
            o, d, f, w = wl.next_step()
            O[:], D[:], F[:], W[:] = o.reshape(-1), d.reshape(-1), f, w
            e.MoveToNextLocation(O, D, F, W)
            orc.MoveToNextLocation(o.reshape(-1).copy(), d.reshape(-1).copy(), f.copy(), w.copy())
        np.testing.assert_array_equal(e.elem_ids, orc.elem_ids)
        np.testing.assert_allclose(e.flux, orc.flux, rtol=1e-9, atol=1e-12)
        pos = torch.empty((n, 3), dtype=torch.float64, device="cuda"); el = torch.empty(n, dtype=torch.int32, device="cuda")
        e.get_state_device(pos.data_ptr(), el.data_ptr(), 0, n)
        e.set_state_device(pos.data_ptr(), el.data_ptr(), 0, n)
        fl = torch.empty(e.num_elements, dtype=torch.float64, device="cuda")
        e.get_flux_device(fl.data_ptr())
        torch.cuda.synchronize()
        np.testing.assert_allclose(fl.cpu().numpy(), e.flux, rtol=0, atol=0)
        e.normalized_flux()
        print("variant", v, opts, "ok", flush=True)

# score filter: per-bin masked passes (mask kernel + the unfiltered walk kernels), host and device entry points
import torch
from helpers import oracle_binned_move
coords, t2v, wl = box_case((5, 5, 4), 4001)
e, orc = PumiTally.from_arrays(coords, t2v, wl.n), OraclePumiTally(coords, t2v, wl.n)
e.set_option("chunk", 1024)
e.set_score_bins(3)
init = wl.initial_positions()
for x in (e, orc):
    x.CopyInitialPosition(init.reshape(-1).copy())
want = np.zeros((3, len(t2v)))
for step in range(2):
    o, d, f, w = wl.next_step()
    bins = (np.arange(wl.n, dtype=np.int32) * 7 + step) % 5 - 1  # -1 .. 3: some outside [0, 3)
    if step == 0:
        e.MoveToNextLocationBinned(o.reshape(-1).copy(), d.reshape(-1).copy(), f.copy(), w.copy(), bins)
    else:
        t = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (o, d, f, w, bins)]
        e.move_device_binned(*(x.data_ptr() for x in t), None)
        torch.cuda.synchronize()
    oracle_binned_move(orc, want, o, d, f, w, bins)
np.testing.assert_allclose(e.flux_bins, want, rtol=1e-9, atol=1e-12)
np.testing.assert_array_equal(e.elem_ids, orc.elem_ids)
print("score bins ok", flush=True)
