"""Small run of the batch-statistics path for compute-sanitizer:
   compute-sanitizer --tool memcheck python scripts/sanitize_batch_stats.py
Odd tally lengths (scalar tail of the 256-bit accumulate pass), score bins with an unreported bin, every
normalisation mode, the statistics read-out, the trigger and the VTK fields."""
import os, sys, tempfile
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import numpy as np
import torch
from helpers import box_case
from pumiumtally_b200.tally import PumiTally

for cells, n, nbins, mode in (((3, 3, 3), 3001, 1, 0), ((5, 4, 3), 4001, 3, 3), ((2, 3, 5), 999, 2, 1)):
    coords, t2v, wl = box_case(cells, n)
    e = PumiTally.from_arrays(coords, t2v, wl.n)
    e.set_option("chunk", 1024)
    if nbins > 1:
        e.set_score_bins(nbins)
    e.set_source_normalization(mode, 7.0)
    e.CopyInitialPosition(wl.initial_positions().reshape(-1))
    vals = []
    for b in range(3):
        o, d, f, w = wl.next_step()
        if nbins > 1:
            bins = (np.arange(wl.n, dtype=np.int32) * 7 + b) % (nbins + 2) - 1
            if b == 1:
                t = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (o, d, f, w, bins)]
                e.move_device_binned(*(x.data_ptr() for x in t), None)
                torch.cuda.synchronize()
            else:
                e.MoveToNextLocationBinned(o.reshape(-1).copy(), d.reshape(-1).copy(), f.copy(), w.copy(), bins)
            vals.append(e.normalized_flux_bins()[0])
        else:
            e.MoveToNextLocation(o.reshape(-1).copy(), d.reshape(-1).copy(), f.copy(), w.copy())
            vals.append(e.normalized_flux()[0])
        e.end_batch()
    mean, sd = e.tally_statistics()
    v = np.asarray(vals)
    np.testing.assert_allclose(mean, v.mean(axis=0), rtol=1e-13)
    np.testing.assert_allclose(sd, v.std(axis=0, ddof=1) / np.sqrt(3), rtol=1e-9, atol=1e-12 * np.abs(mean).max())
    print(cells, nbins, mode, "trigger", e.max_relative_error(0.1), flush=True)
    e.WriteTallyResults(os.path.join(tempfile.mkdtemp(), "fluxresult.vtk"))
print("batch statistics ok", flush=True)
