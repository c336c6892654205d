"""Batch statistics on the device (csrc/batch_stats.cu, Engine::end_batch): per-element mean and standard
deviation of the mean over the ended batches, the relative-error trigger and the VTK fields, against numpy
statistics of the engine's own per-batch normalised tallies (and those against the oracle)."""
import os
import subprocess

import numpy as np
import pytest

from helpers import ROOT, assert_flux_close, box_case, oracle_binned_move
from oracle.oracle import OraclePumiTally
from pumiumtally_b200.mesh import jitter_interior, kuhn_box
from pumiumtally_b200.tally import PumiTally
from pumiumtally_b200.workload import CONFIGS, SyntheticWorkload
from test_gpu_parity import _bins_for_step
from vtk_reader import read_vtu_cell_data

pytestmark = pytest.mark.gpu


def _numpy_stats(values):
    """values[batch, ...] -> (mean, standard deviation of the mean) over the batches"""
    v = np.asarray(values)
    return v.mean(axis=0), v.std(axis=0, ddof=1) / np.sqrt(v.shape[0])


def _assert_stats(eng, values, label=""):
    mean, sd = eng.tally_statistics()
    want_m, want_s = _numpy_stats(values)
    # the mean sums the batches in another order than numpy; the standard deviation comes from plain running
    # sums of squares, whose cancellation costs digits where the batches hardly differ
    np.testing.assert_allclose(mean, want_m, rtol=1e-13, atol=0, err_msg=label)
    bad = np.abs(sd - want_s) > 1e-9 * want_s + 1e-12 * np.abs(want_m)
    assert not bad.any(), f"{label}: {int(bad.sum())} std-dev values off, e.g. {sd[bad][:3]} vs {want_s[bad][:3]}"
    return mean, sd


def _jitter_case(n):
    c, t = jitter_interior(*kuhn_box(8, 7, 6), amplitude=0.18)
    return c, t, SyntheticWorkload(box=(8.0, 7.0, 6.0), num_particles=n, mean_length=3.0, seed=3)


@pytest.mark.parametrize("mesh", ["box", "jitter"])
def test_statistics_of_the_engines_own_batches(mesh):
    """6 batches x 2 host moves: every batch's raw tally matches the oracle's (reset per batch), and the
    statistics are numpy's over the normalised tallies read just before each end_batch."""
    if mesh == "box":
        coords, t2v, wl = box_case((6, 6, 5), 20_000)
    else:
        coords, t2v, wl = _jitter_case(30_000)
    eng, orc = PumiTally.from_arrays(coords, t2v, wl.n), OraclePumiTally(coords, t2v, wl.n)
    init = wl.initial_positions().reshape(-1)
    eng.CopyInitialPosition(init.copy())
    orc.CopyInitialPosition(init.copy())
    values = []
    for batch in range(6):
        orc.reset_flux()
        for _ in range(2):
            o, d, f, w = wl.next_step()
            for x in (eng, orc):
                x.MoveToNextLocation(o.reshape(-1).copy(), d.reshape(-1).copy(), f.copy(), w.copy())
        assert_flux_close(eng.flux, orc.flux, f"{mesh} batch {batch}")
        np.testing.assert_array_equal(eng.elem_ids, orc.elem_ids)
        values.append(eng.normalized_flux()[0])
        eng.end_batch()
        assert eng.get_option("batches") == batch + 1
        assert not eng.flux.any()  # the batch tally starts over
    _assert_stats(eng, values, mesh)
    assert eng.stats()["moves"] == 12  # the counters keep running
    with pytest.raises(ValueError):
        eng.set_option("batches", 0)  # read-only


@pytest.mark.parametrize("mode,value", [(0, 0.0), (1, 0.0), (2, 250.0), (3, 0.0)])
def test_source_normalisation_modes(mode, value):
    coords, t2v, wl = box_case((5, 5, 4), 8000)
    eng = PumiTally.from_arrays(coords, t2v, wl.n)
    eng.set_source_normalization(mode, value)
    eng.CopyInitialPosition(wl.initial_positions().reshape(-1))
    values, divs = [], []
    for _ in range(4):
        for k in range(2):
            o, d, f, w = wl.next_step()
            if k == 0:
                first = float(w[f == 1].sum())
            eng.MoveToNextLocation(o.reshape(-1).copy(), d.reshape(-1).copy(), f.copy(), w.copy())
        div = eng.source_normalization()
        want = {0: 1.0, 1: float(wl.n), 2: value, 3: first}[mode]
        np.testing.assert_allclose(div, want, rtol=1e-12)
        divs.append(div)
        values.append(eng.normalized_flux()[0])
        eng.end_batch()
    if mode == 3:
        assert len(set(divs)) == len(divs)  # a new first-track weight every batch
    _assert_stats(eng, values, f"mode {mode}")
    if mode != 3:
        return
    # a batch whose first move has no flying particle has no source weight: end_batch fails and changes nothing
    before = eng.tally_statistics()
    o, d, f, w = wl.next_step()
    eng.MoveToNextLocation(o.reshape(-1).copy(), d.reshape(-1).copy(), np.zeros_like(f), w.copy())
    o, d, f, w = wl.next_step()
    eng.MoveToNextLocation(o.reshape(-1).copy(), d.reshape(-1).copy(), f.copy(), w.copy())
    raw_before = eng.flux
    assert raw_before.any() and eng.source_normalization() == 0.0
    with pytest.raises(RuntimeError):
        eng.end_batch()
    assert eng.get_option("batches") == 4
    np.testing.assert_array_equal(eng.flux, raw_before)
    after = eng.tally_statistics()
    np.testing.assert_array_equal(after[0], before[0])
    np.testing.assert_array_equal(after[1], before[1])


def _binned_run(tmp_path, batches=4, moves=2, nbins=3):
    coords, t2v, wl = box_case((6, 6, 5), 20_000)
    eng, orc = PumiTally.from_arrays(coords, t2v, wl.n), OraclePumiTally(coords, t2v, wl.n)
    eng.set_score_bins(nbins)
    init = wl.initial_positions().reshape(-1)
    eng.CopyInitialPosition(init.copy())
    orc.CopyInitialPosition(init.copy())
    values, step = [], 0
    for _ in range(batches):
        want = np.zeros((nbins, len(t2v)))
        for _ in range(moves):
            o, d, f, w = wl.next_step()
            bins = _bins_for_step(wl.n, nbins, step)
            step += 1
            eng.MoveToNextLocationBinned(o.reshape(-1).copy(), d.reshape(-1).copy(), f.copy(), w.copy(), bins)
            oracle_binned_move(orc, want, o, d, f, w, bins)
        got = eng.flux_bins
        for b in range(nbins):
            assert_flux_close(got[b], want[b], f"bin {b}")
        values.append(eng.normalized_flux_bins()[0])
        eng.end_batch()
    return eng, values


def test_score_bins_statistics_and_vtk_fields(tmp_path):
    eng, values = _binned_run(tmp_path)
    mean, sd = _assert_stats(eng, values, "3 bins")
    assert mean.shape == (3, eng.num_elements)
    out = str(tmp_path / "fluxresult.vtk")
    eng.WriteTallyResults(out)
    cells = read_vtu_cell_data(os.path.join(out, "pieces", "piece_0.vtu"))
    for b in range(3):
        np.testing.assert_array_equal(cells[f"flux_bin{b}"], mean[b])
        np.testing.assert_array_equal(cells[f"flux_bin{b}_std_dev"], sd[b])
    np.testing.assert_allclose(cells["flux"], mean.sum(axis=0), rtol=1e-14)
    assert "flux_std_dev" not in cells  # the sum over the bins gets none (it would need covariances)
    pvtu = open(os.path.join(out, "pieces.pvtu")).read()
    assert 'Name="flux_bin2_std_dev"' in pvtu


def test_trigger_query_against_numpy(tmp_path):
    eng, values = _binned_run(tmp_path, batches=3, moves=1)
    mean, sd = eng.tally_statistics()
    rel = np.where(mean != 0, sd / np.where(mean != 0, np.abs(mean), 1.0), -1.0).reshape(-1)  # bin-major
    thr = float(np.median(rel[rel >= 0]))
    got_max, got_idx, got_count = eng.max_relative_error(thr)
    assert got_max == rel.max() and got_idx == int(np.argmax(rel))  # argmax: the lowest index on ties
    assert got_count == int((rel > thr).sum())
    assert eng.max_relative_error(1e300)[2] == 0 and eng.max_relative_error(-1.0)[2] == int((rel >= 0).sum())
    one, _ = _binned_run(tmp_path, batches=1, moves=1)
    with pytest.raises(RuntimeError):
        one.max_relative_error(0.1)  # needs two batches


def test_one_batch_and_no_batch_vtk_output(tmp_path):
    coords, t2v, wl = box_case((4, 3, 2), 5000)
    eng = PumiTally.from_arrays(coords, t2v, wl.n)
    eng.set_source_normalization(3)
    eng.CopyInitialPosition(wl.initial_positions().reshape(-1))
    o, d, f, w = wl.next_step()
    eng.MoveToNextLocation(o.reshape(-1), d.reshape(-1), f, w)
    # no batch ended: the output is the normalised flux and nothing else
    out0 = str(tmp_path / "none.vtk")
    eng.WriteTallyResults(out0)
    nf, vol = eng.normalized_flux()
    cells = read_vtu_cell_data(os.path.join(out0, "pieces", "piece_0.vtu"))
    np.testing.assert_array_equal(cells["flux"], nf)
    assert not any(k.startswith("flux_") for k in cells) and "std_dev" not in open(os.path.join(out0, "pieces.pvtu")).read()
    with pytest.raises(RuntimeError):
        eng.tally_statistics()
    # one batch: the written flux is what get_normalized_flux returned just before end_batch
    eng.end_batch()
    out1 = str(tmp_path / "one.vtk")
    eng.WriteTallyResults(out1)
    cells = read_vtu_cell_data(os.path.join(out1, "pieces", "piece_0.vtu"))
    np.testing.assert_allclose(cells["flux"], nf, rtol=1e-14, atol=0)
    np.testing.assert_array_equal(cells["volume"], vol)
    assert "flux_std_dev" not in cells
    mean, sd = eng.tally_statistics()
    assert np.isnan(sd).all()


def test_partial_batch_reset_and_score_bins_discard(tmp_path):
    coords, t2v, wl = box_case((5, 4, 4), 6000)
    eng = PumiTally.from_arrays(coords, t2v, wl.n)
    eng.CopyInitialPosition(wl.initial_positions().reshape(-1))
    for _ in range(3):
        o, d, f, w = wl.next_step()
        eng.MoveToNextLocation(o.reshape(-1), d.reshape(-1), f, w)
        eng.end_batch()
    mean, sd = eng.tally_statistics()
    o, d, f, w = wl.next_step()
    eng.MoveToNextLocation(o.reshape(-1), d.reshape(-1), f, w)  # a batch that never ends
    assert eng.flux.any()
    m2, s2 = eng.tally_statistics()
    np.testing.assert_array_equal(m2, mean)
    np.testing.assert_array_equal(s2, sd)
    out = str(tmp_path / "partial.vtk")
    eng.WriteTallyResults(out)
    cells = read_vtu_cell_data(os.path.join(out, "pieces", "piece_0.vtu"))
    np.testing.assert_array_equal(cells["flux"], mean)
    np.testing.assert_array_equal(cells["flux_std_dev"], sd)
    eng.reset_tally()
    assert eng.get_option("batches") == 0
    with pytest.raises(RuntimeError):
        eng.tally_statistics()
    # after the reset the sums start over: one batch, std NaN
    o, d, f, w = wl.next_step()
    eng.MoveToNextLocation(o.reshape(-1), d.reshape(-1), f, w)
    want = eng.normalized_flux()[0]
    eng.end_batch()
    m3, s3 = eng.tally_statistics()
    np.testing.assert_allclose(m3, want, rtol=1e-14, atol=0)
    assert np.isnan(s3).all()
    eng.set_score_bins(2)
    assert eng.get_option("batches") == 0


def test_end_batch_is_ordered_with_device_moves_on_a_side_stream():
    """Device-pointer moves enqueued on a torch side stream right before and after end_batch, without any
    host synchronisation, give the statistics of the same run synchronised after every call."""
    import torch

    coords, t2v, wl = box_case((6, 6, 6), 200_000)
    init = torch.from_numpy(wl.initial_positions()).cuda()
    steps = [[torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in wl.next_step()] for _ in range(6)]
    torch.cuda.synchronize()
    results = []
    for synced in (False, True):
        eng = PumiTally.from_arrays(coords, t2v, wl.n)
        side = torch.cuda.Stream()
        with torch.cuda.stream(side):
            s = side.cuda_stream
            eng.copy_initial_position_device(init.data_ptr(), s)
            for k, t in enumerate(steps):
                eng.move_device(*(x.data_ptr() for x in t), s)
                if synced:
                    torch.cuda.synchronize()
                if k % 2 == 1:
                    eng.end_batch()
        torch.cuda.synchronize()
        results.append(eng.tally_statistics())
    np.testing.assert_allclose(results[0][0], results[1][0], rtol=1e-12, atol=0)
    np.testing.assert_allclose(results[0][1], results[1][1], rtol=1e-9, atol=1e-12 * np.abs(results[1][0]).max())


def test_config_c2_full_size_statistics():
    """BASELINE configs[1] (998,250 tets, 10 M particles), device-resident, default engine: 4 batches x 2 moves."""
    import torch

    cfg = CONFIGS["c2"]
    cells, n = cfg["cells"], cfg["particles"]
    wl = SyntheticWorkload(box=tuple(float(c) for c in cells), num_particles=n, mean_length=cfg["mean_length"],
                           backend="torch", device="cuda")
    eng = PumiTally(f"box:{cells[0]},{cells[1]},{cells[2]}", n)
    s = torch.cuda.current_stream().cuda_stream
    init = wl.initial_positions().contiguous()
    eng.copy_initial_position_device(init.data_ptr(), s)
    values = []
    for _ in range(4):
        for _ in range(2):
            o, d, f, w = (x.contiguous() for x in wl.next_step())
            eng.move_device(o.data_ptr(), d.data_ptr(), f.data_ptr(), w.data_ptr(), s)
        torch.cuda.synchronize()
        values.append(eng.normalized_flux()[0])
        eng.end_batch()
    mean, _ = _assert_stats(eng, values, "c2")
    assert (mean > 0).mean() > 0.99
    r, idx, cnt = eng.max_relative_error(0.01)
    assert 0 < r < 1 and 0 <= idx < eng.num_elements and cnt > 0


def _two_gpu_batch_worker(rank, world, port, q, choice, mode):
    import sys

    import torch
    import torch.distributed as dist

    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from pumiumtally_b200.distributed import broadcast_unique_id, particle_stripe

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    n_total = 40_000
    b, e = particle_stripe(n_total, rank, world)
    eng = PumiTally.from_spec("box:8,8,8", e - b, device=rank)
    eng.comm_init(rank, world, broadcast_unique_id(dist, PumiTally.nccl_unique_id, device=torch.device("cuda", rank)))
    eng.set_option("exchange_choice", choice)
    eng.set_source_normalization(mode)
    wl = SyntheticWorkload(box=(8.0, 8.0, 8.0), num_particles=e - b, mean_length=2.0, id_offset=b)
    eng.CopyInitialPosition(wl.initial_positions().reshape(-1))
    for _ in range(4):
        for _ in range(2):
            o, d, f, w = wl.next_step()
            eng.MoveToNextLocation(o.reshape(-1), d.reshape(-1), f, w)
        eng.end_batch()
    stats = eng.tally_statistics()
    q.put((rank, stats if rank == 0 else None, eng.max_relative_error(0.05)))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("choice", [0, 1])
@pytest.mark.parametrize("mode", [1, 3])
def test_two_gpu_statistics_equal_single_gpu(choice, mode):
    """Particle stripes on two GPUs, both batch-end exchanges: the statistics are those of one GPU with all
    particles -- the batch divisor counts the particles / first-track weight of every rank."""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29800 + os.getpid() % 100 + 100 * choice + 200 * mode
    procs = [ctx.Process(target=_two_gpu_batch_worker, args=(r, 2, port, q, choice, mode)) for r in range(2)]
    for p in procs:
        p.start()
    got = dict((r, (st, trig)) for r, st, trig in (q.get(timeout=300) for _ in range(2)))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert got[0][1] == got[1][1]  # every rank gets the same trigger answer
    coords, t2v, wl = box_case((8, 8, 8), 40_000, mean_length=2.0)
    one = PumiTally.from_spec("box:8,8,8", 40_000)
    one.set_source_normalization(mode)
    one.CopyInitialPosition(wl.initial_positions().reshape(-1))
    for _ in range(4):
        for _ in range(2):
            o, d, f, w = wl.next_step()
            one.MoveToNextLocation(o.reshape(-1), d.reshape(-1), f, w)
        one.end_batch()
    mean1, sd1 = one.tally_statistics()
    mean2, sd2 = got[0][0]
    np.testing.assert_allclose(mean2, mean1, rtol=1e-9, atol=0)
    assert (np.abs(sd2 - sd1) <= 1e-7 * sd1 + 1e-12 * np.abs(mean1)).all()


def test_openmc_like_driver_active_batches(tmp_path):
    """examples/openmc_like_driver.cpp with 8 active batches: the VTK output carries flux_std_dev, and the
    printed largest relative error is the one computed from the written fields."""
    from pumiumtally_b200 import build as pbuild

    lib = pbuild.build_library()
    exe = str(tmp_path / "driver")
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "examples", "openmc_like_driver.cpp"), "-o", exe,
                           "-L", os.path.dirname(lib), "-lpumitally", "-Wl,-rpath," + os.path.dirname(lib)])
    out = subprocess.check_output([exe, "box:8,8,8", "20000", "4", "0", "1", "8"], cwd=str(tmp_path), text=True)
    assert "DRIVER_OK 640000 flights" in out
    line = [l for l in out.splitlines() if l.startswith("TALLY_TRIGGER")][0]
    printed = float(line.split("max relative error")[1].split()[0])
    cells = read_vtu_cell_data(str(tmp_path / "fluxresult.vtk" / "pieces" / "piece_0.vtu"))
    flux, sd = cells["flux"], cells["flux_std_dev"]
    nz = flux != 0
    assert nz.mean() > 0.9
    rel = sd[nz] / np.abs(flux[nz])
    assert np.isfinite(rel).all() and (rel >= 0).all()
    np.testing.assert_allclose(printed, rel.max(), rtol=1e-15)
