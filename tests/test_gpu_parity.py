"""Parity tests proper: the CUDA path, called through the C ABI of
libpumitally.so, against the CPU oracle on the same seeded inputs
(tolerances: helpers.FLUX_RTOL = 1e-6 relative on flux, exact parent
elements, 1e-12 relative positions), plus size-independent properties at the
full BASELINE.json sizes."""
import os
import subprocess

import numpy as np
import pytest

from helpers import (ROOT, assert_flux_close, assert_positions_close, box_case, edge_case_scenario,
                     lattice_track_scenario, non_convex_relocation_scenario, non_finite_input_scenario,
                     oracle_binned_move, run_workload, unstructured_special_point_scenario)
from oracle.oracle import OraclePumiTally
from pumiumtally_b200.mesh import delaunay_box, jitter_interior, kuhn_box, save_raw_mesh, tet_volumes
from pumiumtally_b200.tally import PumiTally
from pumiumtally_b200.workload import CONFIGS, SyntheticWorkload
from test_oracle_golden import check_c1_fixture, golden_scenario

pytestmark = pytest.mark.gpu
# The product library holds four walk kernels (0 cross-check, 8 streaming, 16 binned gather, 24 packed
# rows).  The measured alternatives live in libpumitally_exp.so; they are only exercised when that
# library is selected (PUMITALLY_LIB=pumiumtally_b200/lib/libpumitally_exp.so).
PRODUCT_VARIANTS = [0, 8, 16, 24]
EXPERIMENTS = os.path.basename(os.environ.get("PUMITALLY_LIB", "")) == "libpumitally_exp.so"
EXP_VARIANTS = [1, 2, 3, 4, 5, 6, 7, 13, 15, 17, 20, 21, 22, 23, 25] if EXPERIMENTS else []
VARIANTS = PRODUCT_VARIANTS + EXP_VARIANTS
BIG_VARIANTS = [0, 8, 16, 24] + ([6, 20, 21] if EXPERIMENTS else [])
EDGE_VARIANTS = [20, 21, 22, 23] if EXPERIMENTS else []  # compact layout + edge-function exit test
_X = [20] if EXPERIMENTS else []


def gpu_engine(variant, block=128, chunk=None, seed_grid=True):
    def make(coords, t2v, n):
        e = PumiTally.from_arrays(coords, t2v, n)
        e.set_option("variant", variant)
        e.set_option("block", block)
        e.set_option("seed_grid", int(seed_grid))  # 0 never, 1 where the hull is convex, 2 always
        if chunk:
            e.set_option("chunk", chunk)
        return e
    return make


@pytest.mark.parametrize("variant", VARIANTS)
def test_reference_known_answers(variant):
    eng = golden_scenario(gpu_engine(variant))
    st = eng.stats()
    assert st["segments"] == 18 and st["tracks"] == 7 and st["lost"] == 0 and st["moves"] == 2


@pytest.mark.parametrize("variant", VARIANTS)
def test_committed_c1_fixture(variant):
    """CUDA path vs the committed oracle fixture tests/golden/c1_oracle.npz (BASELINE configs[0])."""
    eng, segs, tracks = check_c1_fixture(gpu_engine(variant))
    st = eng.stats()
    assert st["segments"] == segs and st["tracks"] == tracks and st["lost"] == 0


@pytest.mark.parametrize("variant", VARIANTS)
def test_edge_cases(variant):
    edge_case_scenario(gpu_engine(variant))


@pytest.mark.parametrize("seed_grid", [False, True])
def test_out_of_mesh_origin_falls_back_to_reference_walk(seed_grid):
    """Relocation targets outside the hull: clipped along the line from the OLD position
    (reference semantics); the seeded walk must detect this and fall back."""
    coords, t2v = kuhn_box(4, 4, 4)
    n = 4096
    rng = np.random.default_rng(5)
    init = rng.uniform(0.2, 3.8, size=(n, 3))
    eng, orc = gpu_engine(8, seed_grid=seed_grid)(coords, t2v, n), OraclePumiTally(coords, t2v, n)
    for e in (eng, orc):
        e.CopyInitialPosition(init.reshape(-1).copy())
    np.testing.assert_array_equal(eng.elem_ids, orc.elem_ids)
    origin = rng.uniform(-3.0, 7.0, size=(n, 3))
    dest = rng.uniform(0.2, 3.8, size=(n, 3))
    w = rng.uniform(0.5, 1.0, size=n)
    for e in (eng, orc):
        e.MoveToNextLocation(origin.reshape(-1).copy(), dest.reshape(-1).copy(), np.ones(n, dtype=np.int8), w.copy())
    assert_flux_close(eng.flux, orc.flux, "outside-origin")
    np.testing.assert_array_equal(eng.elem_ids, orc.elem_ids)
    np.testing.assert_allclose(eng.positions, orc.positions, atol=1e-12)
    assert eng.stats()["lost"] == 0


@pytest.mark.parametrize("variant", [0, 8, 16, 24])
def test_non_convex_mesh_relocation_is_the_reference_walk_unless_the_shortcut_is_forced(variant):
    """On a mesh whose hull is not convex the engine does not take the seed-grid shortcut on its own
    (ADVICE r01): relocation across the notch of an L-shaped mesh stops at the hull exactly like the
    reference's straight walk; seed_grid=2 forces the shortcut and the particles arrive."""
    eng, _ = non_convex_relocation_scenario(gpu_engine(variant, seed_grid=1))
    assert eng.get_option("hull_convex") == 0 and eng.get_option("seed_grid_active") == 0
    eng2, _ = non_convex_relocation_scenario(gpu_engine(variant, seed_grid=2), expect_reference=False)
    assert eng2.get_option("seed_grid_active") == 1
    convex = gpu_engine(variant)(*kuhn_box(2, 2, 2), 4)
    assert convex.get_option("hull_convex") == 1 and convex.get_option("seed_grid_active") == 1


def test_binning_groups_flying_particles_by_cell():
    """The per-move counting sort: order[] holds exactly the flying particles, grouped by the
    seed-grid cell of their origin in ascending cell order."""
    cells = (12, 10, 8)
    coords, t2v, wl = box_case(cells, 200_000)
    e = gpu_engine(16)(coords, t2v, wl.n)
    e.set_option("morton", 1)
    e.CopyInitialPosition(wl.initial_positions().reshape(-1))
    o, d, f, w = wl.next_step()
    fly = f == 1
    e.MoveToNextLocation(o.reshape(-1), d.reshape(-1), f, w)
    order = e.debug_order()
    assert len(order) == int(fly.sum())
    assert np.array_equal(np.sort(order), np.flatnonzero(fly))
    # recompute the cell of every origin with the grid geometry of csrc/seed_grid.hpp
    ncell_target = max(len(t2v) / 4.0, 1.0)
    h = (np.prod(cells) / ncell_target) ** (1.0 / 3.0)
    dims = np.minimum(np.maximum(np.ceil(np.array(cells) / h), 1), 1024).astype(int)
    h = max(h, *(np.array(cells) / dims))
    c = np.minimum((o[order] / h).astype(int), dims - 1)

    def spread(v):  # Morton bit interleave, as csrc/seed_grid.hpp::morton_cell_ranks
        v = v.astype(np.uint64) & np.uint64(0x1fffff)
        for sh, m in ((32, 0x1f00000000ffff), (16, 0x1f0000ff0000ff), (8, 0x100f00f00f00f00f),
                      (4, 0x10c30c30c30c30c3), (2, 0x1249249249249249)):
            v = (v | (v << np.uint64(sh))) & np.uint64(m)
        return v

    key = spread(c[:, 0]) | (spread(c[:, 1]) << np.uint64(1)) | (spread(c[:, 2]) << np.uint64(2))
    assert (np.diff(key.astype(np.int64)) >= 0).all(), f"{int((np.diff(key.astype(np.int64)) < 0).sum())} order inversions"


def test_seed_grid_cuts_relocation_work_not_results():
    coords, t2v, wl = box_case((12, 12, 12), 100_000)
    res = []
    for sg in (False, True):
        wl_i = SyntheticWorkload(box=(12.0, 12.0, 12.0), num_particles=wl.n)
        e = gpu_engine(8, seed_grid=sg)(coords, t2v, wl.n)
        e.CopyInitialPosition(wl_i.initial_positions().reshape(-1))
        for _ in range(3):
            o, d, f, w = wl_i.next_step()
            e.MoveToNextLocation(o.reshape(-1), d.reshape(-1), f, w)
        res.append((e.flux, e.elem_ids, e.positions, e.stats()))
    assert_flux_close(res[1][0], res[0][0], "seeded vs reference walk")
    np.testing.assert_array_equal(res[1][1], res[0][1])
    np.testing.assert_array_equal(res[1][2], res[0][2])
    assert res[1][3]["segments"] == res[0][3]["segments"]
    assert res[1][3]["relocations"] < 0.3 * res[0][3]["relocations"]


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("block", [64, 256])
def test_config_c1_parity(variant, block):
    coords, t2v, wl = box_case(CONFIGS["c1"]["cells"], CONFIGS["c1"]["particles"])
    eng = gpu_engine(variant, block)(coords, t2v, wl.n)
    orc = OraclePumiTally(coords, t2v, wl.n)
    run_workload(eng, orc, wl, steps=4, label=f"c1 v{variant}")
    st = eng.stats()
    assert st["segments"] == orc.n_segments and st["tracks"] == orc.n_tracks and st["lost"] == 0
    assert st["kernel_ms"] > 0


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("mesh", ["jitter", "delaunay"])
def test_unstructured_parity(variant, mesh):
    if mesh == "jitter":
        c, t = jitter_interior(*kuhn_box(8, 7, 6), amplitude=0.18)
        box = (8.0, 7.0, 6.0)
    else:
        c, t = delaunay_box(3000)
        box = (1.0, 1.0, 1.0)
    n = 50_000
    wl = SyntheticWorkload(box=box, num_particles=n, mean_length=0.4 * min(box), seed=3)
    eng, orc = gpu_engine(variant)(c, t, n), OraclePumiTally(c, t, n)
    run_workload(eng, orc, wl, steps=3, label=f"{mesh} v{variant}")
    assert eng.stats()["segments"] == orc.n_segments


@pytest.mark.parametrize("variant", VARIANTS)
def test_long_axial_tracks(variant):
    coords, t2v, wl = box_case((8, 8, 80), 20_000, mean_length=120.0, mu_min=0.9)
    eng, orc = gpu_engine(variant)(coords, t2v, wl.n), OraclePumiTally(coords, t2v, wl.n)
    run_workload(eng, orc, wl, steps=2, label="c4-mini")
    assert eng.stats()["segments"] == orc.n_segments


def test_contention_many_particles_few_tets():
    """Config c3 in miniature: thousands of particles per tet hammer the same flux words."""
    coords, t2v, wl = box_case((3, 3, 3), 400_000, mean_length=1.5)
    eng, orc = gpu_engine(0)(coords, t2v, wl.n), OraclePumiTally(coords, t2v, wl.n)
    run_workload(eng, orc, wl, steps=2, check_each_step=False, label="c3-mini")


@pytest.mark.parametrize("variant", EDGE_VARIANTS)
def test_edge_walk_takes_the_plane_records_only_for_coplanar_rays(variant):
    """Generic rays never leave the compact layout; rays coplanar with a mesh edge (axis-parallel
    tracks in a Kuhn mesh, tracks inside a face plane) are finished on the plane records and still
    match the oracle element for element (walk_compact.cuh)."""
    coords, t2v, wl = box_case((6, 6, 5), 20_000)
    eng, orc = gpu_engine(variant)(coords, t2v, wl.n), OraclePumiTally(coords, t2v, wl.n)
    run_workload(eng, orc, wl, steps=3, label=f"generic v{variant}")
    assert eng.stats()["plane_fallbacks"] == 0
    deg = edge_case_scenario(gpu_engine(variant))
    assert deg.stats()["plane_fallbacks"] > 0
    golden = golden_scenario(gpu_engine(variant))  # T1: axis-parallel tracks through the 6-tet cube
    assert golden.stats()["plane_fallbacks"] > 0


@pytest.mark.parametrize("variant", [0, 8, 16, 24] + _X)
def test_chunked_upload_pipeline_equals_single_range(variant):
    """Host-pointer path cut into many upload/compute ranges (the binned variant bins each range)."""
    coords, t2v, wl = box_case((6, 6, 5), 50_000)
    a = gpu_engine(variant, chunk=4096)(coords, t2v, wl.n)
    orc = OraclePumiTally(coords, t2v, wl.n)
    run_workload(a, orc, wl, steps=3, label="chunked")
    assert a.stats()["segments"] == orc.n_segments


@pytest.mark.parametrize("resample", [0.05, 0.9])
def test_staged_upload_of_origins_is_exact(resample):
    """Host-pointer path, staged (the default): origins equal to the previous call's destinations are
    not sent again (the device still holds them); the changed ones travel as a patch list, or the
    whole slice when most of a chunk changed.  Results must be identical to direct uploads of all
    four arrays (host_path=0), bytes must drop."""
    coords, t2v = kuhn_box(6, 6, 5)
    n = 40_000
    rng = np.random.default_rng(11)
    engs = []
    for mode in (0, 1):
        e = gpu_engine(8, chunk=8192)(coords, t2v, n)
        e.set_option("host_path", mode)
        engs.append(e)
    orc = OraclePumiTally(coords, t2v, n)
    pos = rng.uniform(0.05, 4.95, size=(n, 3))
    for e in engs + [orc]:
        e.CopyInitialPosition(pos.reshape(-1).copy())
    prev_dest = pos.copy()
    for step in range(4):
        origin = prev_dest.copy()
        moved = rng.random(n) < resample                 # re-sourced particles get a fresh origin
        origin[moved] = rng.uniform(0.05, 4.95, size=(int(moved.sum()), 3))
        # per-axis bounds: equal clipped coordinates would put particles exactly on a diagonal face plane
        dest = np.clip(origin + rng.normal(0, 1.0, size=(n, 3)), [0.011, 0.013, 0.017], [4.987, 4.983, 4.979])
        fly = (rng.random(n) < 0.9).astype(np.int8)
        w = rng.uniform(0.5, 1.0, n)
        for e in engs + [orc]:
            e.MoveToNextLocation(origin.reshape(-1).copy(), dest.reshape(-1).copy(), fly.copy(), w.copy())
        prev_dest = dest
    off, on = engs
    np.testing.assert_array_equal(on.elem_ids, off.elem_ids)
    np.testing.assert_array_equal(on.positions, off.positions)
    np.testing.assert_allclose(on.flux, off.flux, rtol=1e-12)
    assert_flux_close(on.flux, orc.flux, "staged upload")
    np.testing.assert_array_equal(on.elem_ids, orc.elem_ids)
    assert on.stats()["h2d_bytes"] < (0.75 if resample < 0.4 else 1.01) * off.stats()["h2d_bytes"]


def test_staged_upload_survives_interleaved_device_moves():
    import torch

    coords, t2v, wl = box_case((6, 6, 5), 20_000)
    a, b = gpu_engine(8)(coords, t2v, wl.n), gpu_engine(8)(coords, t2v, wl.n)
    a.set_option("host_path", 1)
    b.set_option("host_path", 0)
    init = wl.initial_positions().reshape(-1)
    for e in (a, b):
        e.CopyInitialPosition(init.copy())
    for step in range(5):
        o, d, f, w = wl.next_step()
        for e in (a, b):
            if step == 2:  # a device-pointer move in between: the particles move, the staging mirror does not
                t = [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (o, d, f, w)]
                e.move_device(*(x.data_ptr() for x in t), torch.cuda.current_stream().cuda_stream)
                torch.cuda.synchronize()
            else:
                e.MoveToNextLocation(o.reshape(-1).copy(), d.reshape(-1).copy(), f.copy(), w.copy())
    np.testing.assert_array_equal(a.elem_ids, b.elem_ids)
    np.testing.assert_array_equal(a.positions, b.positions)
    np.testing.assert_allclose(a.flux, b.flux, rtol=1e-12)


def test_pageable_buffers_with_host_registration():
    """Direct path with register_host=1: the caller's pageable numpy buffers are page-locked once and reused."""
    coords, t2v, wl = box_case((6, 6, 5), 60_000)
    eng = gpu_engine(8)(coords, t2v, wl.n)
    eng.set_option("host_path", 0)
    eng.set_option("register_host", 1)
    orc = OraclePumiTally(coords, t2v, wl.n)
    init = wl.initial_positions()
    eng.CopyInitialPosition(init.reshape(-1).copy())
    orc.CopyInitialPosition(init.reshape(-1).copy())
    # the same four buffers are reused for every move, as OpenMC does
    O, D, W = np.empty(3 * wl.n), np.empty(3 * wl.n), np.empty(wl.n)
    F = np.empty(wl.n, dtype=np.int8)
    for _ in range(3):
        o, d, f, w = wl.next_step()
        O[:], D[:], W[:], F[:] = o.reshape(-1), d.reshape(-1), w, f
        f2 = f.copy()
        eng.MoveToNextLocation(O, D, F, W)
        orc.MoveToNextLocation(o.reshape(-1), d.reshape(-1), f2, w)
        assert not F.any()
    assert_flux_close(eng.flux, orc.flux, "registered host buffers")
    np.testing.assert_array_equal(eng.elem_ids, orc.elem_ids)


@pytest.mark.parametrize("threads", [1, 3, 8])
def test_staged_path_reused_buffers_ragged_sizes_and_flag_values(threads):
    """The staged host path with the caller reusing its four buffers (as OpenMC does), a particle
    count that is not a multiple of anything, flying values other than 0/1 (only 1 flies,
    PumiTallyImpl.cpp:95), unaligned array addresses and 1..8 staging workers."""
    coords, t2v, wl = box_case((6, 6, 5), 50_003)
    n = wl.n
    e = PumiTally.from_arrays(coords, t2v, n)
    e.set_option("host_threads", threads)
    e.set_option("chunk", 4096)
    orc = OraclePumiTally(coords, t2v, n)
    init = wl.initial_positions()
    e.CopyInitialPosition(init.reshape(-1).copy())
    orc.CopyInitialPosition(init.reshape(-1).copy())
    assert e.get_option("staged") == 1 and e.get_option("host_threads") == threads
    # odd offsets: the caller's arrays are only 8-byte (flying: 1-byte) aligned
    O, D, W = np.empty(3 * n + 1)[1:], np.empty(3 * n + 1)[1:], np.empty(n + 1)[1:]
    F = np.empty(n + 3, dtype=np.int8)[3:]
    rng = np.random.default_rng(5)
    for step in range(4):
        o, d, f, w = wl.next_step()
        f = f.copy()
        odd = rng.random(n) < 0.02
        f[odd] = rng.choice(np.array([2, -1, 127, -128], dtype=np.int8), int(odd.sum()))
        O[:], D[:], W[:], F[:] = o.reshape(-1), d.reshape(-1), w, f
        f_ref = f.copy()
        e.MoveToNextLocation(O, D, F, W)
        orc.MoveToNextLocation(o.reshape(-1).copy(), d.reshape(-1).copy(), f_ref, w.copy())
        assert not F.any()
        # (particles with odd flag values did not fly although the generator thinks they did: their
        # next origin differs from where they are, which both sides handle by relocating them)
        assert_flux_close(e.flux, orc.flux, f"staged step {step}")
        np.testing.assert_array_equal(e.elem_ids, orc.elem_ids)
    st = e.stats()
    assert st["segments"] == orc.n_segments and st["lost"] == 0
    # origins travelled only for re-sourced particles (many in this small box): under the 57 B/particle
    # of a direct upload; test_staged_path_every_origin_changed_and_none_changed pins the byte counts
    assert st["h2d_bytes"] < 24 * n + 4 * 57 * n


def _host_buffers(n, kind):
    """The caller's four arrays: 'pinned' = page-locked by the caller (torch), else ordinary numpy."""
    if kind == "pinned":
        import torch

        return [torch.empty(s_, dtype=d_, pin_memory=True).numpy() for s_, d_ in
                ((3 * n, torch.float64), (3 * n, torch.float64), (n, torch.int8), (n, torch.float64))]
    return [np.empty(3 * n), np.empty(3 * n), np.empty(n, dtype=np.int8), np.empty(n)]


def _every_origin_changed_and_none_changed(buffers):
    """Patch-list overflow (every origin differs from the previous destination -> the slice travels
    whole) and the opposite extreme (no origin changed -> no origin bytes at all), staged from the
    caller's `buffers` (_host_buffers kind)."""
    coords, t2v = kuhn_box(6, 6, 5)
    n = 30_000
    rng = np.random.default_rng(3)
    e = gpu_engine(8, chunk=4096)(coords, t2v, n)
    e.set_option("host_path", 1)  # staged also for page-locked arrays, not the automatic choice
    orc = OraclePumiTally(coords, t2v, n)
    pos = rng.uniform(0.05, 4.95, size=(n, 3))
    for x in (e, orc):
        x.CopyInitialPosition(pos.reshape(-1).copy())
    O, D, F, W = _host_buffers(n, buffers)
    sent = [e.stats()["h2d_bytes"]]
    prev = pos
    for step in range(4):
        origin = prev.copy() if step % 2 == 0 else rng.uniform(0.05, 4.95, size=(n, 3))
        dest = np.clip(origin + rng.normal(0, 0.8, size=(n, 3)), [0.011, 0.013, 0.017], [4.987, 4.983, 4.979])
        w = rng.uniform(0.5, 1.0, n)
        O[:], D[:], W[:], F[:] = origin.reshape(-1), dest.reshape(-1), w, 1
        e.MoveToNextLocation(O, D, F, W)
        orc.MoveToNextLocation(origin.reshape(-1).copy(), dest.reshape(-1).copy(), np.ones(n, dtype=np.int8), w.copy())
        prev = dest
        sent.append(e.stats()["h2d_bytes"])
    per_move = np.diff(sent) / n
    assert abs(per_move[0] - 33) < 0.01 and abs(per_move[2] - 33) < 0.01   # nothing changed: no origin bytes
    assert abs(per_move[1] - 57) < 0.01 and abs(per_move[3] - 57) < 0.01   # everything changed: slices sent whole
    assert_flux_close(e.flux, orc.flux, f"overflow / no-change extremes, {buffers} buffers")
    np.testing.assert_array_equal(e.elem_ids, orc.elem_ids)
    np.testing.assert_array_equal(e.positions, orc.positions)


def test_staged_path_every_origin_changed_and_none_changed():
    _every_origin_changed_and_none_changed("pageable")


def test_page_locked_caller_arrays_every_origin_changed_and_none_changed():
    """Page-locked caller arrays go through the staging slots as well (host_path=1): the same 33 B /
    57 B per particle as from pageable arrays."""
    _every_origin_changed_and_none_changed("pinned")


@pytest.mark.parametrize("kind", ["pinned", "registered"])
@pytest.mark.parametrize("variant", [-1, 16, 24])
def test_page_locked_caller_arrays_match_oracle(kind, variant):
    """Host-pointer moves through the default staged path on page-locked caller arrays (pinned by the
    caller, or by register_host=1).  Re-sourcing, hull clipping, non-flying particles, odd flag values,
    a device-pointer move in between and non-finite origins included."""
    import torch

    coords, t2v, wl = box_case((6, 6, 5), 60_007)
    n = wl.n
    e = gpu_engine(variant, chunk=8192)(coords, t2v, n)
    e.set_option("host_path", 1)  # not the automatic choice between staged and direct uploads
    if kind == "registered":
        e.set_option("register_host", 1)
    orc = OraclePumiTally(coords, t2v, n)
    init = wl.initial_positions()
    e.CopyInitialPosition(init.reshape(-1).copy())
    orc.CopyInitialPosition(init.reshape(-1).copy())
    O, D, F, W = _host_buffers(n, kind)
    rng = np.random.default_rng(9)
    lost = 0
    for step in range(6):
        o, d, f, w = wl.next_step()
        o, f = o.copy(), f.copy()
        odd = rng.random(n) < 0.01
        f[odd] = rng.choice(np.array([2, -1, 127], dtype=np.int8), int(odd.sum()))
        f_ref = f.copy()
        if step == 3:  # a device-pointer move: the staging slots do not see it
            t = [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (o, d, f, w)]
            e.move_device(*(x.data_ptr() for x in t), torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
        else:
            if step == 4:  # unusable origins: those particles sit the move out and are counted
                bad = np.flatnonzero(f == 1)[:25]
                o[bad[:10], 1] = np.nan
                o[bad[10:], 2] = np.inf
                f_ref[bad] = 0
                lost += len(bad)
            O[:], D[:], W[:], F[:] = o.reshape(-1), d.reshape(-1), w, f
            e.MoveToNextLocation(O, D, F, W)
            assert not F.any()
        orc.MoveToNextLocation(np.nan_to_num(o, nan=0.5, posinf=0.5).reshape(-1).copy(), d.reshape(-1).copy(), f_ref, w.copy())
        assert_flux_close(e.flux, orc.flux, f"page-locked caller arrays, step {step}")
        ok = np.ones(n, dtype=bool)
        if step == 4:
            ok[bad] = False  # the oracle was told they do not fly; here they were skipped: same state either way
        np.testing.assert_array_equal(e.elem_ids, orc.elem_ids)
        np.testing.assert_allclose(e.positions, orc.positions, rtol=0, atol=1e-9)
    st = e.stats()
    assert st["segments"] == orc.n_segments and st["lost"] == lost


def test_page_locked_caller_arrays_get_the_faster_of_staged_and_direct_uploads():
    """host_path=2 (default): with page-locked caller arrays moves 2-3 of every 256 are uploaded directly,
    the rest staged, and the faster path is kept; results are the oracle's whichever path a move took."""
    coords, t2v, wl = box_case((6, 6, 5), 80_000)
    n = wl.n
    e = gpu_engine(8, chunk=16384)(coords, t2v, n)
    orc = OraclePumiTally(coords, t2v, n)
    init = wl.initial_positions()
    for x in (e, orc):
        x.CopyInitialPosition(init.reshape(-1).copy())
    O, D, F, W = _host_buffers(n, "pinned")
    paths = []
    for step in range(8):
        o, d, f, w = wl.next_step()
        O[:], D[:], W[:], F[:] = o.reshape(-1), d.reshape(-1), w, f
        e.MoveToNextLocation(O, D, F, W)
        paths.append(e.get_option("host_path_last"))
        orc.MoveToNextLocation(o.reshape(-1).copy(), d.reshape(-1).copy(), f.copy(), w.copy())
        assert not F.any()
        assert_flux_close(e.flux, orc.flux, f"auto host path, step {step}")
        np.testing.assert_array_equal(e.elem_ids, orc.elem_ids)
    assert paths[:4] == [1, 1, 0, 0]  # staged, staged, direct, direct; then whichever was faster
    assert e.stats()["segments"] == orc.n_segments


def test_error_behaviour():
    coords, t2v = kuhn_box(1, 1, 1)
    e = PumiTally.from_arrays(coords, t2v, 5)
    xyz = np.tile([0.1, 0.4, 0.5], 5)
    fly = np.ones(5, dtype=np.int8)
    with pytest.raises(RuntimeError):  # move before CopyInitialPosition (assert Impl.cpp:437)
        e.MoveToNextLocation(xyz, xyz, fly, np.ones(5))
    with pytest.raises(RuntimeError):  # size must be 3N (assert Impl.cpp:57)
        e.CopyInitialPosition(xyz, 5)
    e.CopyInitialPosition(xyz, 15)
    with pytest.raises(RuntimeError):  # only once (PumiTally.h:63-64)
        e.CopyInitialPosition(xyz, 15)
    with pytest.raises(RuntimeError):
        e.MoveToNextLocation(xyz, xyz, fly, np.ones(5), 5)
    with pytest.raises(RuntimeError):
        PumiTally("does/not/exist.osh", 5)
    with pytest.raises(RuntimeError):  # degenerate tet
        PumiTally.from_arrays(np.zeros((4, 3)), np.array([[0, 1, 2, 3]], dtype=np.int32), 1)


def test_raw_mesh_file_and_box_spec(tmp_path):
    coords, t2v = kuhn_box(3, 2, 2)
    path = str(tmp_path / "mesh.ptm")
    save_raw_mesh(path, coords, t2v)
    a, b = PumiTally(path, 100), PumiTally("box:3,2,2", 100)
    assert a.num_elements == b.num_elements == 72
    np.testing.assert_array_equal(a.adjacency, b.adjacency)
    wl = SyntheticWorkload(box=(3.0, 2.0, 2.0), num_particles=100, mean_length=1.0)
    init = wl.initial_positions().reshape(-1)
    o, d, f, w = wl.next_step()
    for e in (a, b):
        e.CopyInitialPosition(init.copy())
        e.MoveToNextLocation(o.reshape(-1).copy(), d.reshape(-1).copy(), f.copy(), w.copy())
    np.testing.assert_allclose(a.flux, b.flux, rtol=1e-13)


@pytest.mark.parametrize("fmt", ["osh", "osh_uncompressed", "msh"])
def test_mesh_file_formats_drive_the_engine_like_the_oracle(tmp_path, fmt):
    """The ctor's mesh argument as a user would pass it (PumiTally.h:40-47): an Omega_h .osh
    directory or the Gmsh file it was converted from.  Unstructured mesh, three moves, parity
    against the oracle built from the same arrays."""
    from pumiumtally_b200.mesh import save_gmsh, save_osh

    coords, t2v = delaunay_box(400)
    if fmt == "msh":
        path = str(tmp_path / "mesh.msh")
        save_gmsh(path, coords, t2v, version="4.1")
    else:
        path = str(tmp_path / "mesh.osh")
        save_osh(path, coords, t2v, compressed=(fmt == "osh"))
    n = 20_000
    eng, orc = PumiTally(path, n), OraclePumiTally(coords, t2v, n)
    assert eng.num_elements == len(t2v)
    wl = SyntheticWorkload(box=(1.0, 1.0, 1.0), num_particles=n, mean_length=0.3)
    run_workload(eng, orc, wl, steps=3, label=fmt)


def test_device_pointer_entry_points_match_host_path():
    import torch

    coords, t2v, wl = box_case((6, 6, 5), 30_000)
    host = gpu_engine(0)(coords, t2v, wl.n)
    dev = gpu_engine(0)(coords, t2v, wl.n)
    init = wl.initial_positions()
    host.CopyInitialPosition(init.reshape(-1).copy())
    d_init = torch.from_numpy(init).cuda()
    dev.copy_initial_position_device(d_init.data_ptr(), torch.cuda.current_stream().cuda_stream)
    for _ in range(3):
        o, d, f, w = wl.next_step()
        host.MoveToNextLocation(o.reshape(-1).copy(), d.reshape(-1).copy(), f.copy(), w.copy())
        t = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (o, d, f, w)]
        dev.move_device(*(x.data_ptr() for x in t), torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
    np.testing.assert_allclose(dev.flux, host.flux, rtol=1e-12)
    np.testing.assert_array_equal(dev.elem_ids, host.elem_ids)
    np.testing.assert_array_equal(dev.positions, host.positions)


def test_normalized_flux_reset_and_vtk_output(tmp_path):
    coords, t2v, wl = box_case((4, 3, 2), 5000)
    e = gpu_engine(0)(coords, t2v, wl.n)
    e.CopyInitialPosition(wl.initial_positions().reshape(-1))
    o, d, f0, w = wl.next_step()
    f = f0.copy()
    e.MoveToNextLocation(o.reshape(-1), d.reshape(-1), f0, w)
    nf, vol = e.normalized_flux()
    np.testing.assert_allclose(vol, tet_volumes(coords, t2v), rtol=1e-13)
    np.testing.assert_allclose(nf, e.flux / vol, rtol=1e-14)
    out = str(tmp_path / "fluxresult.vtk")
    e.WriteTallyResults(out)
    from vtk_reader import read_vtu_cell_data

    cells = read_vtu_cell_data(os.path.join(out, "pieces", "piece_0.vtu"))
    np.testing.assert_array_equal(cells["flux"], nf)
    np.testing.assert_array_equal(cells["volume"], vol)
    conn = cells["connectivity"].reshape(-1, 4)
    np.testing.assert_array_equal(np.sort(conn, axis=1), np.sort(t2v, axis=1))  # same tets, caller's order ...
    v = coords[conn]
    assert (np.einsum("ij,ij->i", np.cross(v[:, 1] - v[:, 0], v[:, 2] - v[:, 0]), v[:, 3] - v[:, 0]) > 0).all()  # ... positively oriented
    assert os.path.exists(os.path.join(out, "pieces.pvtu"))
    # per-source normalisation of the normalised flux (the reference's unfinished total_initial_weight,
    # PumiTallyImpl.h:170-171): the raw flux never changes
    raw = e.flux.copy()
    for mode, value, div in ((1, 0.0, float(wl.n)), (2, 123.5, 123.5), (0, 0.0, 1.0)):
        e.set_source_normalization(mode, value)
        assert e.source_normalization() == div
        np.testing.assert_allclose(e.normalized_flux()[0], raw / vol / div, rtol=1e-14)
        np.testing.assert_array_equal(e.flux, raw)
    with pytest.raises(ValueError):
        e.set_source_normalization(2, 0.0)
    e.reset_tally()
    assert not e.flux.any() and e.stats()["segments"] == 0
    # mode 3: total weight of the first tracks after the reset, summed on the device
    e.set_source_normalization(3)
    o2, d2, f2, w2 = wl.next_step()
    want = float(w2[f2 == 1].sum())
    e.MoveToNextLocation(o2.reshape(-1), d2.reshape(-1), f2, w2)
    o3, d3, f3, w3 = wl.next_step()
    e.MoveToNextLocation(o3.reshape(-1), d3.reshape(-1), f3, w3)  # later moves do not add to it
    np.testing.assert_allclose(e.source_normalization(), want, rtol=1e-12)
    np.testing.assert_allclose(e.normalized_flux()[0], e.flux / vol / want, rtol=1e-13)


def _bins_for_step(n, nbins, step):
    rng = np.random.default_rng(1000 + step)
    bins = rng.integers(0, nbins, n, dtype=np.int32)
    bins[rng.random(n) < 0.07] = -1            # no bin matches: flies unscored
    bins[rng.random(n) < 0.03] = nbins + 5     # likewise
    return bins


@pytest.mark.parametrize("variant", [-1, 0, 8, 16, 24])
def test_score_bins_host_moves_match_the_oracle_bin_by_bin(variant, tmp_path):
    """Score filter (SURVEY 8 f4): particle i scores into flux array bins[i] of this move; the bins change
    from move to move; particles outside every bin move like the others and score nowhere."""
    nbins = 3
    coords, t2v, wl = box_case((6, 6, 5), 20_000)
    e = gpu_engine(variant, chunk=4096)(coords, t2v, wl.n)
    e.set_score_bins(nbins)
    assert e.score_bins == nbins
    orc = OraclePumiTally(coords, t2v, wl.n)
    init = wl.initial_positions()
    e.CopyInitialPosition(init.reshape(-1).copy())
    orc.CopyInitialPosition(init.reshape(-1).copy())
    want = np.zeros((nbins, len(t2v)))
    for step in range(3):
        o, d, f, w = wl.next_step()
        bins = _bins_for_step(wl.n, nbins, step)
        f1 = f.copy()
        e.MoveToNextLocationBinned(o.reshape(-1).copy(), d.reshape(-1).copy(), f1, w.copy(), bins)
        assert not f1.any()
        oracle_binned_move(orc, want, o, d, f, w, bins)
        got = e.flux_bins
        for b in range(nbins):
            assert_flux_close(got[b], want[b], f"bin {b} step {step}")
        np.testing.assert_array_equal(e.flux, got[0])  # n = num_elements: the first bin
        np.testing.assert_array_equal(e.elem_ids, orc.elem_ids)
        assert_positions_close(e.positions, orc.positions, f"step {step}")
    assert want.sum() < orc.flux.sum()  # the unscored particles did fly (the oracle tallied them)
    nf, vol = e.normalized_flux_bins()
    np.testing.assert_allclose(nf, got / vol, rtol=1e-14)
    out = str(tmp_path / "fluxresult.vtk")
    e.WriteTallyResults(out)
    from vtk_reader import read_vtu_cell_data

    cells = read_vtu_cell_data(os.path.join(out, "pieces", "piece_0.vtu"))
    for b in range(nbins):
        np.testing.assert_array_equal(cells[f"flux_bin{b}"], nf[b])
    np.testing.assert_allclose(cells["flux"], nf.sum(axis=0), rtol=1e-14)
    # a plain move on a binned engine scores into the first bin; bins=None is the plain move
    o, d, f, w = wl.next_step()
    before = e.flux_bins
    e.MoveToNextLocation(o.reshape(-1).copy(), d.reshape(-1).copy(), f.copy(), w.copy())
    after = e.flux_bins
    np.testing.assert_array_equal(after[1:], before[1:])
    assert after[0].sum() > before[0].sum()
    e.reset_tally()
    assert not e.flux_bins.any()


def test_score_bins_device_moves_and_single_bin():
    import torch

    nbins = 4
    coords, t2v, wl = box_case((5, 5, 5), 15_000)
    host, dev, plain, direct = (gpu_engine(-1)(coords, t2v, wl.n) for _ in range(4))
    host.set_score_bins(nbins)
    dev.set_score_bins(nbins)
    direct.set_score_bins(nbins)
    direct.set_option("host_path", 0)  # plain copies of the caller's arrays instead of the staging slots
    direct.set_option("chunk", 4096)
    plain.set_score_bins(1)  # one bin is the unfiltered tally
    init = wl.initial_positions()
    for x in (host, dev, plain, direct):
        x.CopyInitialPosition(init.reshape(-1).copy())
    s = torch.cuda.current_stream().cuda_stream
    for step in range(3):
        o, d, f, w = wl.next_step()
        bins = _bins_for_step(wl.n, nbins, step)
        inside = (bins >= 0) & (bins < nbins)
        host.MoveToNextLocationBinned(o.reshape(-1).copy(), d.reshape(-1).copy(), f.copy(), w.copy(), bins)
        direct.MoveToNextLocationBinned(o.reshape(-1).copy(), d.reshape(-1).copy(), f.copy(), w.copy(), bins)
        t = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (o, d, f, w, bins)]
        dev.move_device_binned(*(x.data_ptr() for x in t), s)
        torch.cuda.synchronize()
        # the unfiltered engine with the unscored particles' weights set to zero tallies the sum of the bins
        plain.MoveToNextLocationBinned(o.reshape(-1).copy(), d.reshape(-1).copy(), f.copy(), np.where(inside, w, 0.0), bins)
    np.testing.assert_allclose(dev.flux_bins, host.flux_bins, rtol=1e-12)
    np.testing.assert_allclose(direct.flux_bins, host.flux_bins, rtol=1e-12)
    np.testing.assert_array_equal(direct.positions, host.positions)
    np.testing.assert_array_equal(dev.elem_ids, host.elem_ids)
    np.testing.assert_array_equal(dev.positions, host.positions)
    np.testing.assert_array_equal(plain.elem_ids, host.elem_ids)
    assert_flux_close(host.flux_bins.sum(axis=0), plain.flux, "sum over bins vs unfiltered")
    d_out = torch.empty(nbins * len(t2v), dtype=torch.float64, device="cuda")
    host.get_flux_device(d_out.data_ptr(), s)
    torch.cuda.synchronize()
    np.testing.assert_array_equal(d_out.cpu().numpy().reshape(nbins, -1), host.flux_bins)
    with pytest.raises(ValueError):
        host.set_score_bins(0)


def test_cxx_facade_program(tmp_path):
    """Link a C++ caller against include/pumitally/PumiTally.h + libpumitally.so, the way the
    OpenMC fork does, and replay the reference's known-answer scenario."""
    from pumiumtally_b200 import build as pbuild

    lib = pbuild.build_library()
    exe = str(tmp_path / "facade_demo")
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "facade_demo.cpp"), "-o", exe,
                           "-L", os.path.dirname(lib), "-lpumitally", "-Wl,-rpath," + os.path.dirname(lib)])
    out = subprocess.check_output([exe], cwd=str(tmp_path), text=True)
    assert "[TIME] Total PUMI-Tally time" in out
    assert "FACADE_OK" in out
    from vtk_reader import read_vtu_cell_data

    cells = read_vtu_cell_data(str(tmp_path / "fluxresult.vtk" / "pieces" / "piece_0.vtu"))
    np.testing.assert_allclose(cells["flux"] * cells["volume"], [0, 0, 1.5, 0.5, 2.5, 0], atol=1e-8)


def test_openmc_like_driver_example(tmp_path):
    """examples/openmc_like_driver.cpp: the four OpenMC call sites against the C++ facade."""
    from pumiumtally_b200 import build as pbuild

    lib = pbuild.build_library()
    exe = str(tmp_path / "driver")
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "examples", "openmc_like_driver.cpp"), "-o", exe,
                           "-L", os.path.dirname(lib), "-lpumitally", "-Wl,-rpath," + os.path.dirname(lib)])
    out = subprocess.check_output([exe, "box:8,8,8", "20000", "4"], cwd=str(tmp_path), text=True)
    assert "DRIVER_OK 80000 flights" in out and "[TIME] Total time to tally" in out
    from vtk_reader import read_vtu_cell_data

    cells = read_vtu_cell_data(str(tmp_path / "fluxresult.vtk" / "pieces" / "piece_0.vtu"))
    total = float((cells["flux"] * cells["volume"]).sum())
    assert 0.5 * 80000 * 0.75 < total < 3.0 * 80000 * 0.75 * 1.5  # ~ flights * <w> * <in-box length>
    # with an inactive batch first (tally reset) and per-source normalisation by the total weight of the
    # active batch's first tracks (PumiTallyExtras.h): the written flux is the raw one over that weight
    out = subprocess.check_output([exe, "box:8,8,8", "20000", "4", "1"], cwd=str(tmp_path), text=True)
    assert "DRIVER_OK 80000 flights" in out
    norm = float(out.split("source normalisation")[1].split()[0])
    assert 0.7 * 20000 * 0.75 < norm < 1.3 * 20000 * 0.75  # ~ particles * <w>
    cells = read_vtu_cell_data(str(tmp_path / "fluxresult.vtk" / "pieces" / "piece_0.vtu"))
    total2 = float((cells["flux"] * cells["volume"]).sum()) * norm
    assert 0.5 * 80000 * 0.75 < total2 < 3.0 * 80000 * 0.75 * 1.5
    # three energy groups (score filter): every group gets about a third, the groups add up to "flux"
    out = subprocess.check_output([exe, "box:8,8,8", "20000", "4", "0", "3"], cwd=str(tmp_path), text=True)
    assert "DRIVER_OK 80000 flights" in out
    cells = read_vtu_cell_data(str(tmp_path / "fluxresult.vtk" / "pieces" / "piece_0.vtu"))
    groups = np.stack([cells[f"flux_bin{g}"] for g in range(3)])
    np.testing.assert_allclose(groups.sum(axis=0), cells["flux"], rtol=1e-13)
    share = (groups * cells["volume"]).sum(axis=1) / float((cells["flux"] * cells["volume"]).sum())
    assert (np.abs(share - 1 / 3) < 0.02).all(), share


def _two_gpu_bins_worker(rank, world, port, q):
    import torch
    import torch.distributed as dist

    sys_path = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    import sys
    sys.path.insert(0, sys_path)
    from pumiumtally_b200.distributed import broadcast_unique_id, particle_stripe

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    n_total, nbins = 30_000, 3
    b, e = particle_stripe(n_total, rank, world)
    eng = PumiTally.from_spec("box:7,7,7", e - b, device=rank)
    eng.set_score_bins(nbins)  # before comm_init: the exchange buffers are sized for all bins
    eng.comm_init(rank, world, broadcast_unique_id(dist, PumiTally.nccl_unique_id, device=torch.device("cuda", rank)))
    wl = SyntheticWorkload(box=(7.0, 7.0, 7.0), num_particles=e - b, mean_length=2.0, id_offset=b)
    eng.CopyInitialPosition(wl.initial_positions().reshape(-1))
    for k in range(2):
        o, d, f, w = wl.next_step()
        bins = _bins_for_step(n_total, nbins, k)[b:e].copy()
        eng.MoveToNextLocationBinned(o.reshape(-1), d.reshape(-1), f, w, bins)
        (eng.allreduce_tally if k == 0 else eng.reduce_tally_to_owners)()
    flux = eng.flux_bins
    if rank == 0:
        q.put(flux)
    dist.barrier()
    dist.destroy_process_group()


def test_two_gpu_score_bins_exchange_equals_single_gpu():
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29700 + os.getpid() % 1000
    procs = [ctx.Process(target=_two_gpu_bins_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    flux2 = q.get(timeout=180)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    n_total, nbins = 30_000, 3
    coords, t2v, wl = box_case((7, 7, 7), n_total, mean_length=2.0)
    one = PumiTally.from_spec("box:7,7,7", n_total)
    one.set_score_bins(nbins)
    one.CopyInitialPosition(wl.initial_positions().reshape(-1))
    for k in range(2):
        o, d, f, w = wl.next_step()
        one.MoveToNextLocationBinned(o.reshape(-1), d.reshape(-1), f, w, _bins_for_step(n_total, nbins, k))
    for b in range(nbins):
        assert_flux_close(flux2[b], one.flux_bins[b], f"2-GPU bin {b} vs 1 GPU")


def _two_gpu_worker(rank, world, port, q, outdir=None):
    import torch
    import torch.distributed as dist

    sys_path = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    import sys
    sys.path.insert(0, sys_path)
    from pumiumtally_b200.distributed import broadcast_unique_id, particle_stripe

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    cells, n_total = (8, 8, 8), 40_000
    b, e = particle_stripe(n_total, rank, world)
    eng = PumiTally.from_spec("box:8,8,8", e - b, device=rank)
    eng.comm_init(rank, world, broadcast_unique_id(dist, PumiTally.nccl_unique_id, device=torch.device("cuda", rank)))
    wl = SyntheticWorkload(box=(8.0, 8.0, 8.0), num_particles=e - b, mean_length=2.0, id_offset=b)
    eng.CopyInitialPosition(wl.initial_positions().reshape(-1))
    for k in range(3):
        o, d, f, w = wl.next_step()
        eng.MoveToNextLocation(o.reshape(-1), d.reshape(-1), f, w)
        # an exchange after every batch: each must give the sum over ranks of everything tallied so
        # far, never counting an earlier exchange's result again -- by all-reduce, or by the cheaper
        # reduce-scatter whose shares are gathered when somebody asks for the flux
        if k == 0:
            eng.allreduce_tally()
        elif k == 1:
            eng.reduce_tally_to_owners()
        else:
            assert eng.get_option("exchange_choice") in (0, 1) and eng.get_option("exchange_allreduce_us") >= 0
            eng.exchange_tally()  # whichever of the two comm_init measured to be quicker here
        if k == 1:
            part = eng.flux  # collective gather on every rank
            assert np.isfinite(part).all()
    if outdir:  # every rank writes its slice of the (global) result: pieces/piece_<rank>.vtu, rank 0 the .pvtu
        eng.WriteTallyResults(outdir)
    flux = eng.flux  # every rank: the accessor gathers the shares of the last reduce-scatter
    if rank == 0:
        q.put(flux)
    dist.barrier()
    dist.destroy_process_group()


def test_two_gpu_stripes_allreduce_equals_single_gpu(tmp_path):
    """Particle stripes on two GPUs + ncclAllReduce of the tally == one GPU with all particles; the two
    ranks' VTK pieces tile the mesh and hold the global normalised flux."""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29600 + os.getpid() % 1000
    outdir = str(tmp_path / "fluxresult.vtk")
    procs = [ctx.Process(target=_two_gpu_worker, args=(r, 2, port, q, outdir)) for r in range(2)]
    for p in procs:
        p.start()
    flux2 = q.get(timeout=180)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    coords, t2v, wl = box_case((8, 8, 8), 40_000, mean_length=2.0)
    one = PumiTally.from_spec("box:8,8,8", 40_000)
    one.CopyInitialPosition(wl.initial_positions().reshape(-1))
    for _ in range(3):
        o, d, f, w = wl.next_step()
        one.MoveToNextLocation(o.reshape(-1), d.reshape(-1), f, w)
    assert_flux_close(flux2, one.flux, "2-GPU allreduce vs 1 GPU")
    from vtk_reader import read_vtu_cell_data

    pieces = [read_vtu_cell_data(os.path.join(outdir, "pieces", f"piece_{r}.vtu")) for r in range(2)]
    nf, vol = one.normalized_flux()
    assert len(pieces[0]["flux"]) + len(pieces[1]["flux"]) == len(nf) and len(pieces[0]["flux"]) == len(nf) // 2
    np.testing.assert_allclose(np.concatenate([p["flux"] for p in pieces]), nf, rtol=1e-9, atol=1e-12 * nf.sum())
    np.testing.assert_array_equal(np.concatenate([p["volume"] for p in pieces]), vol)
    pvtu = open(os.path.join(outdir, "pieces.pvtu")).read()
    assert "pieces/piece_0.vtu" in pvtu and "pieces/piece_1.vtu" in pvtu


def test_two_gpu_spatial_partition_equals_replicas():
    """pumiumtally_b200/partition.py on two GPUs (RCB picparts, routing, hand-off, ghost exchange)
    against the replica scheme on the same particles: scripts/exp_partition.py reports the parity."""
    import json
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    out = subprocess.check_output(
        ["python", "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
         "--master-port", str(29900 + os.getpid() % 90), os.path.join(ROOT, "scripts", "exp_partition.py"),
         "c2", "400000", "2", "4"], text=True, cwd=ROOT, timeout=600)
    res = json.loads([l for l in out.splitlines() if l.startswith("{")][-1])
    assert res["parity"]["flux_elements_outside_1e-6"] == 0
    assert res["parity"]["parent_element_mismatches"] == 0 and res["parity"]["max_position_error"] < 1e-9
    assert res["partition"]["handoffs_per_move"] > 0
    assert res["partition"]["local_tets"] < 0.7 * res["tets"]


# ---------------------------------------------------------------- full sizes

def _box_clip_length(o, d, box):
    """Length of segment o->d inside [0,box] (torch, on device)."""
    import torch

    u = d - o
    t1 = torch.ones(o.shape[0], dtype=torch.float64, device=o.device)
    for k in range(3):
        uk = u[:, k]
        hi = torch.where(uk > 0, (box[k] - o[:, k]) / uk, torch.where(uk < 0, (0.0 - o[:, k]) / uk, t1 * float("inf")))
        t1 = torch.minimum(t1, hi)
    return t1.clamp(min=0.0) * u.norm(dim=1)


def _full_size_properties(cfg_name, variant, n=None, cross_check=None, steps=2):
    """What must hold at any size, checked at BASELINE.json's full sizes where the oracle would
    need minutes: total tally == sum of weighted in-box track lengths (conservation), every
    particle ends inside its parent tet, final positions equal the clipped destinations, and
    optionally a second kernel variant must reproduce flux, elements and segment count."""
    import torch

    cfg = CONFIGS[cfg_name]
    cells = cfg["cells"]
    n = n or cfg["particles"]
    box = tuple(float(c) for c in cells)
    kw = dict(box=box, num_particles=n, mean_length=cfg["mean_length"], backend="torch", device="cuda")
    if "mu_min" in cfg:
        kw["mu_min"] = cfg["mu_min"]
    eng = PumiTally(f"box:{cells[0]},{cells[1]},{cells[2]}", n)
    eng.set_option("variant", variant)
    wl = SyntheticWorkload(**kw)
    init = wl.initial_positions().contiguous()
    s = torch.cuda.current_stream().cuda_stream
    eng.copy_initial_position_device(init.data_ptr(), s)
    expect_total = 0.0
    for step in range(steps):
        o, d, f, w = (x.contiguous() for x in wl.next_step())
        eng.move_device(o.data_ptr(), d.data_ptr(), f.data_ptr(), w.data_ptr(), s)
        fly = f == 1
        expect_total += float((_box_clip_length(o[fly], d[fly], box) * w[fly]).sum())
    torch.cuda.synchronize()
    flux = eng.flux
    st = eng.stats()
    assert st["lost"] == 0 and st["tracks"] > 0.9 * steps * n
    np.testing.assert_allclose(flux.sum(), expect_total, rtol=1e-9)
    assert (flux >= 0).all()
    # containment of a 200k-particle sample: barycentric coordinates of the stored position
    # in the stored parent tet are all >= -1e-9
    coords, t2v = kuhn_box(*cells)
    elem, pos = eng.elem_ids, eng.positions
    assert elem.min() >= 0 and elem.max() < len(t2v)
    idx = np.random.default_rng(0).choice(n, min(n, 200_000), replace=False)
    v = coords[t2v[elem[idx]]]
    T = np.transpose(v[:, 1:] - v[:, :1], (0, 2, 1))
    lam = np.linalg.solve(T, (pos[idx] - v[:, 0])[..., None])[..., 0]
    lam0 = 1.0 - lam.sum(1)
    assert min(lam.min(), lam0.min()) > -1e-9
    # final positions: destination if it is inside the box, else on the hull
    d_np, fly_np = d.cpu().numpy(), fly.cpu().numpy()
    inside = ((d_np >= 0) & (d_np <= np.array(box))).all(1)
    sel = idx[fly_np[idx] & inside[idx]]
    np.testing.assert_array_equal(pos[sel], d_np[sel])
    out = idx[fly_np[idx] & ~inside[idx]]
    on_hull = (np.isclose(pos[out], 0.0, atol=1e-9) | np.isclose(pos[out], np.array(box), atol=1e-9)).any(1)
    assert on_hull.all()
    if cross_check is not None and cross_check != variant:
        ref = PumiTally(f"box:{cells[0]},{cells[1]},{cells[2]}", n)
        ref.set_option("variant", cross_check)
        wl2 = SyntheticWorkload(**kw)
        i2 = wl2.initial_positions().contiguous()
        ref.copy_initial_position_device(i2.data_ptr(), s)
        for step in range(steps):
            o, d, f, w = (x.contiguous() for x in wl2.next_step())
            ref.move_device(o.data_ptr(), d.data_ptr(), f.data_ptr(), w.data_ptr(), s)
        torch.cuda.synchronize()
        assert_flux_close(flux, ref.flux, f"{cfg_name}: variant {variant} vs {cross_check}")
        np.testing.assert_array_equal(elem, ref.elem_ids)
        assert st["segments"] == ref.stats()["segments"]
    return st


@pytest.mark.parametrize("variant", BIG_VARIANTS)
def test_config_c2_full_size_properties(variant):
    """BASELINE.json configs[1] (998,250 tets, 10 M particles); variant 0 (thread per particle,
    plain loads) is the cross-check for the others."""
    _full_size_properties("c2", variant, cross_check=0)


@pytest.mark.parametrize("variant", [-1] + _X)
def test_config_c4_full_size_properties(variant):
    """BASELINE.json configs[3]: ~1 M tets, 1 M particles, near-axial tracks crossing hundreds of tets."""
    st = _full_size_properties("c4", variant, cross_check=0)
    assert st["segments"] > 100 * st["tracks"]


def test_config_c5_per_gpu_share_full_size_properties():
    """BASELINE.json configs[4], one GPU's share: 9.86 M tets (1.26 GB of records, the binned kernel is
    chosen automatically), 12.5 M particles; cross-checked against the streaming kernel."""
    cfg = CONFIGS["c5"]
    _full_size_properties("c5", -1, n=cfg["particles"] // cfg["gpus"], cross_check=8, steps=1)


def test_config_c3_full_size_properties():
    """BASELINE.json configs[2]: 48,000 tets, 100 M particles (about 2,000 particles per tet and move
    hammering the same flux words)."""
    _full_size_properties("c3", -1, cross_check=0, steps=1)


def _full_size_oracle_parity(cfg_name, n, steps=2, engine_opts=None):
    """One BASELINE configuration at its full mesh size and `n` particles through the default engine
    and through the per-particle oracle (both exit rules): parent elements exact after localisation
    and after every move, flux 1e-6 element for element, positions, equal segment / track counts."""
    import torch

    cfg = CONFIGS[cfg_name]
    cells = cfg["cells"]
    coords, t2v = kuhn_box(*cells)
    box = tuple(float(c) for c in cells)
    wl = SyntheticWorkload(box=box, num_particles=n, mean_length=cfg["mean_length"], mu_min=cfg["mu_min"],
                           backend="torch", device="cuda")
    eng = PumiTally.from_arrays(coords, t2v, n)
    for k, v in (engine_opts or {}).items():
        eng.set_option(k, v)
    orc = OraclePumiTally(coords, t2v, n, per_particle=True)
    strict = OraclePumiTally(coords, t2v, n, per_particle=True, strict_exit=True)
    init = wl.initial_positions().cpu().numpy()
    for e in (eng, orc, strict):
        e.CopyInitialPosition(init.reshape(-1).copy())
    np.testing.assert_array_equal(eng.elem_ids, orc.elem_ids, err_msg=f"{cfg_name}: parent elements after localisation")
    np.testing.assert_array_equal(strict.elem_ids, orc.elem_ids)
    for step in range(steps):
        o, d, f, w = (x.cpu().numpy() for x in wl.next_step())
        for e in (eng, orc, strict):
            e.MoveToNextLocation(o.reshape(-1).copy(), d.reshape(-1).copy(), f.copy(), w.copy())
        flux = orc.flux
        assert_flux_close(eng.flux, flux, f"{cfg_name} full size, move {step}")
        np.testing.assert_allclose(strict.flux, flux, rtol=1e-12)
        np.testing.assert_array_equal(eng.elem_ids, orc.elem_ids, err_msg=f"{cfg_name}: parent elements after move {step}")
        np.testing.assert_array_equal(strict.elem_ids, orc.elem_ids)
        np.testing.assert_allclose(eng.positions, orc.positions, rtol=0, atol=1e-10 * max(box))
    st = eng.stats()
    assert st["segments"] == orc.n_segments == strict.n_segments
    assert st["tracks"] == orc.n_tracks and st["lost"] == 0 and orc.n_lost == 0
    return eng, orc


def test_config_c2_full_size_oracle_parity():
    """BASELINE configs[1]: 998,250 tets, 10 M particles, element for element against the oracle."""
    eng, _ = _full_size_oracle_parity("c2", CONFIGS["c2"]["particles"])
    assert eng.get_option("variant") in (8, 24)


def test_config_c4_full_size_oracle_parity():
    """BASELINE configs[3]: 1 M collimated tracks of ~200 segments on the 1.0 M-tet pin-cell mesh."""
    _full_size_oracle_parity("c4", CONFIGS["c4"]["particles"])


def test_config_c5_per_gpu_share_full_size_oracle_parity():
    """BASELINE configs[4], one GPU's share: 12.5 M particles on the 9.86 M-tet mesh (binned kernel)."""
    eng, _ = _full_size_oracle_parity("c5", CONFIGS["c5"]["particles"] // CONFIGS["c5"]["gpus"])
    assert eng.get_option("variant") == 16


def test_config_c3_ten_million_particle_slice_oracle_parity():
    """BASELINE configs[2] (contention: 48,000 tets), a 10 M-particle slice of its 100 M."""
    _full_size_oracle_parity("c3", 10_000_000)


@pytest.mark.parametrize("variant", [0, 8, 16] + _X)
def test_walks_cut_short_by_the_crossing_limit_are_reported_and_recoverable(variant):
    """Reference: "ERROR: Not all particles are found. May need more loops in search" and execution
    continues (PumiTallyImpl.cpp:455-458).  Here a walk that runs into the limit is counted as lost and
    stops where it is: its stored position lies in its stored element, nothing is tallied twice, and the
    next move relocates it like any other particle."""
    coords, t2v, wl = box_case((8, 8, 8), 20_000, mean_length=6.0)
    eng = gpu_engine(variant)(coords, t2v, wl.n)
    orc = OraclePumiTally(coords, t2v, wl.n)
    init = wl.initial_positions().reshape(-1)
    for e in (eng, orc):
        e.CopyInitialPosition(init.copy())
    eng.set_option("max_iters", 5)
    o, d, f, w = wl.next_step()
    eng.MoveToNextLocation(o.reshape(-1).copy(), d.reshape(-1).copy(), f.copy(), w.copy())
    st = eng.stats()
    assert st["lost"] > 100
    elem, pos = eng.elem_ids, eng.positions
    v = coords[t2v[elem]]
    T = np.transpose(v[:, 1:] - v[:, :1], (0, 2, 1))
    lam = np.linalg.solve(T, (pos - v[:, 0])[..., None])[..., 0]
    assert min(lam.min(), (1.0 - lam.sum(1)).min()) > -1e-9
    fly = f == 1
    full = float((np.linalg.norm(np.clip(d[fly], 0, 8) - o[fly], axis=1) * w[fly]).sum())
    assert 0.0 < eng.flux.sum() < full
    # back to the normal limit: the oracle continues from the engine's state
    eng.set_option("max_iters", 0)
    eng.reset_tally()
    orc2 = OraclePumiTally(coords, t2v, wl.n)
    orc2.CopyInitialPosition(pos.reshape(-1).copy())  # (stopped particles sit on a face: either tet is theirs)
    o, d, f, w = wl.next_step()
    for e in (eng, orc2):
        e.MoveToNextLocation(o.reshape(-1).copy(), d.reshape(-1).copy(), f.copy(), w.copy())
    assert eng.stats()["lost"] == 0
    assert_flux_close(eng.flux, orc2.flux, "after recovery")
    moved = f == 1  # particles that did not fly still sit on their face
    np.testing.assert_array_equal(eng.elem_ids[moved], orc2.elem_ids[moved])


def test_autotuner_switches_kernels_without_changing_results():
    """Default engine (variant chosen automatically): moves 1-4 alternate the streaming and the packed/sorted
    kernel, later moves use the faster one.  Whatever it picks, every move must match the oracle."""
    coords, t2v, wl = box_case((8, 8, 40), 30_000, mean_length=60.0, mu_min=0.99)
    eng = PumiTally.from_arrays(coords, t2v, wl.n)
    assert eng.get_option("autotune") == 1
    orc = OraclePumiTally(coords, t2v, wl.n)
    run_workload(eng, orc, wl, steps=8, label="autotune")
    assert eng.get_option("variant") in (8, 24)
    assert eng.get_option("launches") >= 8 + 1 + 2 * 5  # 8 moves + localisation + two packed exploration moves
    assert eng.stats()["segments"] == orc.n_segments
    pinned = PumiTally.from_arrays(coords, t2v, wl.n)
    pinned.set_option("autotune", 0)
    wl2 = SyntheticWorkload(box=(8.0, 8.0, 40.0), num_particles=wl.n, mean_length=60.0, mu_min=0.99)
    run_workload(pinned, OraclePumiTally(coords, t2v, wl.n), wl2, steps=6, label="autotune off")
    assert pinned.get_option("variant") == 8 and pinned.get_option("launches") == 6 + 1


@pytest.mark.parametrize("variant", [0, 8, 16, 24] + _X)
def test_degenerate_starts_and_tracks_conserve_length(variant):
    """Particles on mesh vertices, edges and faces, tracks along edges, inside face planes (the hull
    surface included) and through vertices: which of the touching tets gets a piece is a tie-break,
    but no particle may be lost or stopped early, the total tally must equal the total track length
    and every particle must end in a tet that contains its final position."""
    coords, t2v = kuhn_box(3, 3, 3)
    special = np.array([[0, 0, 0], [1, 1, 1], [2, 1, 0], [1.5, 1.5, 1.5], [1.5, 1.0, 1.0], [0.5, 0.5, 1.0],
                        [1.0, 2.0, 1.0], [2.5, 2.5, 2.5], [1.0, 1.0, 0.5], [3, 3, 3], [0.25, 0.25, 0.25],
                        [2.0, 0.5, 1.5], [1.25, 1.25, 2.0]], dtype=float)
    rng = np.random.default_rng(5)
    pairs = [(a, b) for a in range(len(special)) for b in range(len(special)) if a != b]
    n = len(pairs)
    start = np.array([special[a] for a, _ in pairs])
    dest = np.array([special[b] for _, b in pairs])
    w = rng.uniform(0.5, 1.0, n)
    eng = gpu_engine(variant)(coords, t2v, n)
    eng.CopyInitialPosition(start.reshape(-1).copy())
    assert not eng.flux.any()
    eng.MoveToNextLocation(start.reshape(-1).copy(), dest.reshape(-1).copy(), np.ones(n, dtype=np.int8), w.copy())
    assert eng.stats()["lost"] == 0
    np.testing.assert_allclose(eng.flux.sum(), (np.linalg.norm(dest - start, axis=1) * w).sum(), rtol=1e-12)
    np.testing.assert_array_equal(eng.positions, dest)  # hull corner (3,3,3) included: hull planes err outwards
    v = coords[t2v[eng.elem_ids]]
    T = np.transpose(v[:, 1:] - v[:, :1], (0, 2, 1))
    lam = np.linalg.solve(T, (eng.positions - v[:, 0])[..., None])[..., 0]
    assert min(lam.min(), (1.0 - lam.sum(1)).min()) > -1e-12
    back = rng.uniform(0.1, 2.9, size=(n, 3))
    eng.MoveToNextLocation(dest.reshape(-1).copy(), back.reshape(-1).copy(), np.ones(n, dtype=np.int8), w.copy())
    assert eng.stats()["lost"] == 0
    np.testing.assert_array_equal(eng.positions, back)
    orc = OraclePumiTally(coords, t2v, n)
    orc.CopyInitialPosition(back.reshape(-1).copy())
    np.testing.assert_array_equal(eng.elem_ids, orc.elem_ids)


@pytest.mark.parametrize("variant", [0, 8, 16, 24] + _X)
def test_non_finite_inputs_do_not_poison_tally_or_state(variant):
    non_finite_input_scenario(gpu_engine(variant))


@pytest.mark.parametrize("variant", [-1, 0, 16, 24])
def test_zero_and_one_particle(variant):
    coords, t2v = kuhn_box(2, 2, 2)
    e = PumiTally.from_arrays(coords, t2v, 0)
    e.set_option("variant", variant)
    e.CopyInitialPosition(np.empty(0))
    for _ in range(3):
        e.MoveToNextLocation(np.empty(0), np.empty(0), np.empty(0, dtype=np.int8), np.empty(0))
    assert not e.flux.any() and e.stats()["tracks"] == 0
    e1, o1 = PumiTally.from_arrays(coords, t2v, 1), OraclePumiTally(coords, t2v, 1)
    e1.set_option("variant", variant)
    p0, p1, p2 = np.array([0.3, 0.2, 0.1]), np.array([1.7, 1.2, 0.4]), np.array([0.6, 1.1, 1.9])
    for x in (e1, o1):
        x.CopyInitialPosition(p0.copy())
        x.MoveToNextLocation(p0.copy(), p1.copy(), np.ones(1, dtype=np.int8), np.ones(1))
        x.MoveToNextLocation(p1.copy(), p2.copy(), np.ones(1, dtype=np.int8), np.full(1, 2.0))
    assert_flux_close(e1.flux, o1.flux, "one particle")
    np.testing.assert_array_equal(e1.elem_ids, o1.elem_ids)


@pytest.mark.parametrize("variant", [-1, 8, 16, 24] + _X)
def test_randomised_meshes_and_tracks_parity(variant):
    """Seeded sweep through the C ABI: random Delaunay / jittered / anisotropic Kuhn meshes, random particle
    counts, track lengths and collimation -- five moves each against the oracle."""
    for seed in range(10):
        rng = np.random.default_rng(seed)
        kind = seed % 3
        if kind == 0:
            c, t = delaunay_box(int(rng.integers(30, 400)), seed=seed)
            box = (1.0, 1.0, 1.0)
        elif kind == 1:
            dims = tuple(int(x) for x in rng.integers(1, 7, 3))
            c, t = jitter_interior(*kuhn_box(*dims), amplitude=float(rng.uniform(0, 0.3)), seed=seed)
            box = tuple(float(d) for d in dims)
        else:
            dims = tuple(int(x) for x in rng.integers(1, 9, 3))
            box = tuple(float(x) for x in rng.uniform(0.3, 5, 3))
            c, t = kuhn_box(*dims, *box)
        n = int(rng.integers(1, 3000))
        wl = SyntheticWorkload(box=box, num_particles=n, mean_length=float(rng.uniform(0.05, 3.0)) * min(box), seed=seed,
                               mu_min=float(rng.choice([-1.0, 0.5, 0.99])))
        eng = PumiTally.from_arrays(c, t, n)
        eng.set_option("variant", variant)
        run_workload(eng, OraclePumiTally(c, t, n), wl, steps=5, label=f"seed {seed} v{variant}")
        assert eng.stats()["lost"] == 0


@pytest.mark.parametrize("variant", [0, 8, 16, 24] + _X)
def test_lattice_tracks_on_hull_faces_edges_and_vertices(variant):
    lattice_track_scenario(gpu_engine(variant), range(8))


@pytest.mark.parametrize("variant", [0, 8, 16, 24] + _X)
def test_tracks_through_vertices_and_along_edges_of_unstructured_meshes(variant):
    unstructured_special_point_scenario(gpu_engine(variant), range(6))


@pytest.mark.skipif(not EXPERIMENTS, reason="needs libpumitally_exp.so (PUMITALLY_LIB)")
@pytest.mark.parametrize("variant", [9, 27, 28, 29, 30, 31, 32])
def test_round2_experiment_kernels_match_oracle(variant):
    """The round-2 experiments (64-register build, two rays per lane, aggregated tally, lean step with
    prefetch) through the same parity scenarios as the product kernels."""
    golden_scenario(gpu_engine(variant))
    edge_case_scenario(gpu_engine(variant))
    coords, t2v, wl = box_case((6, 6, 5), 30_000)
    eng, orc = gpu_engine(variant)(coords, t2v, wl.n), OraclePumiTally(coords, t2v, wl.n)
    run_workload(eng, orc, wl, steps=3, label=f"experiment v{variant}")
    assert eng.stats()["segments"] == orc.n_segments and eng.stats()["lost"] == 0
