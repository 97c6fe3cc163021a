"""The whole library on the CPU: tests/emul/build/libmdgpu_emul.so is libmdgpu's own sources (plan.cu, every kernel file) compiled by g++ —
kernel launches turned into emul_launch, CUDA runtime calls served by tests/emul/fake_cudart.cpp — so the C ABI, the plan's host logic
(batching, slots, scratch sizing, result folds) and the kernels run together without a GPU. Here: the tests of the device paths written after
the GPU budget was spent (tests/test_zz_gpu_new_ops.py, all of them) and a few of the GPU-validated parity tests as a check of the emulation.
The complete GPU suite passes this way too (28 tests, ~25 min): `python tests/emul/run_under_emulation.py tests/test_gpu_parity.py -m gpu`.

This is evidence about source logic, not a substitute for the GPU run: launch limits, memory spaces and timing are not modelled."""
import os
import sys

import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emul"))


@pytest.fixture(scope="module")
def emulated_library():
    import build_emul
    import viamd_b200.api as api
    saved = (api.LIB_PATH, api._lib)
    api.LIB_PATH = build_emul.build_library(); api._lib = None
    yield api
    api.LIB_PATH, api._lib = saved


def _run_all(mod, names):
    for n in names:
        getattr(mod, n)()


def test_new_device_paths_through_the_c_abi(emulated_library):
    """rmsd, distance_pair + aggregates, com, plane, count(within()), their error paths: every test of tests/test_zz_gpu_new_ops.py."""
    import test_zz_gpu_new_ops as P
    import inspect
    names = [n for n in dir(P) if n.startswith("test_") and not inspect.signature(getattr(P, n)).parameters]   # the shim test (tmp_path) drives a binary linked to the real library
    for slow in ("test_within_min_max_form", "test_static_selection_and_within"):   # ~40 s each under emulation; they pass (run_under_emulation.py) and
        names.remove(slow)                                                              # their forms are in the shim test of this suite, against the reference itself
    assert len(names) >= 7
    _run_all(P, names)


def test_validated_paths_agree_under_emulation(emulated_library):
    """A slice of tests/test_gpu_parity.py (all of which have passed on a B200): rdf per-frame bins incl. batching and stream slots,
    centre-of-mass references, density + every temporal, error paths."""
    import test_gpu_parity as G
    _run_all(G, ["test_golden_water_rdf_per_frame_bitexact", "test_golden_water_rdf_com_references_bitexact", "test_golden_water_density_and_temporals",
                 "test_empty_and_error_paths"])


def _shard_worker(rank, world, port, q):
    """one rank of the frame-sharded evaluation: global plan, its shard at global frame offsets, the one exchange step over gloo"""
    import ctypes
    import numpy as np
    import torch
    import torch.distributed as dist
    here = os.path.dirname(os.path.abspath(__file__))
    for p in (os.path.dirname(here), here, os.path.join(here, "emul")):
        sys.path.insert(0, p)
    import build_emul
    import viamd_b200.api as api
    api.LIB_PATH = build_emul.build_library(); api._lib = None
    import viamd_b200 as vb
    from viamd_b200 import dist as vdist
    from helpers import load_golden, golden_system, vb_system, vb_cell
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    g = load_golden("water6.npz"); s = golden_system(g); F = g["frames"].shape[0]
    props = vb.compile_script("r = rdf(element('O'), element('O'), 6.0); d = distance(1,10); dp = distance_pair(atom(1:5), atom(20:30)); cw = count(within(4.0, residue(1)));", vb_system(s))
    plan = vb.Plan(vb_system(s), props, F)
    cells = [vb_cell(g["cells"][f], g["cell_flags"][f]) for f in range(F)]
    plan.set_initial_frame(*g["frames"][0], cells[0])
    beg, end = vdist.frame_shard(F, world, rank)
    plan.eval_host_frames(g["frames"][beg:end], cells[beg:end], beg)

    def host_view(ptr, n, typestr):   # the emulated library's "device" memory is host memory: wrap it in place
        dt = np.dtype(typestr); buf = (ctypes.c_char * (n * dt.itemsize)).from_address(ptr)
        return torch.from_numpy(np.frombuffer(buf, dtype=dt))
    vdist.allreduce_plan(plan, F, view=host_view)
    out = {k: plan.property_data(k).values.copy() for k in ("r", "d", "dp", "cw")}
    out["dp_mean"] = plan.aggregate("dp")["mean"]; out["d_minmax"] = np.array([plan.property_data("d").min_value, plan.property_data("d").max_value], np.float32)
    out["mask"] = plan.frame_mask()
    plan.close()
    q.put((rank, out))
    dist.destroy_process_group()


def test_two_rank_frame_shards_merge_through_the_exchange_step():
    """SURVEY 8(e) with world_size 2 over gloo, on the emulated library: every rank holds a plan over the GLOBAL frame range, evaluates its
    contiguous shard, and viamd_b200.dist.allreduce_plan — the function bench.py calls over NCCL — merges integer bins and the disjoint float
    rows of the temporals. Both ranks end with the reference's 4-frame results: rdf mean, distance, the distance_pair matrix with its
    per-frame aggregates, count(within()), min/max over all frames, a full frame mask."""
    import numpy as np
    import torch.multiprocessing as mp
    from helpers import load_golden
    ctx = mp.get_context("spawn"); q = ctx.Queue(); port = 29700 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_shard_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs: p.start()
    res = dict(q.get(timeout=600) for _ in procs)
    for p in procs: p.join(120)
    g = load_golden("water6.npz"); pz = load_golden("pairs6.npz")
    for r in (0, 1):
        o = res[r]
        np.testing.assert_allclose(o["r"][:1024], g["r__full"][:1024], rtol=1e-5, atol=1e-6)
        assert np.array_equal(o["d"], g["d__full"]) and np.array_equal(o["dp"], pz["w_dp__full"]) and np.array_equal(o["cw"], g["cw__full"])
        assert np.array_equal(o["dp_mean"], pz["w_dp__mean"]) and o["d_minmax"][0] == g["d__meta"][0] and o["d_minmax"][1] == g["d__meta"][1]
        assert o["mask"].all()
    assert np.array_equal(res[0]["r"], res[1]["r"])


# ---------------------------------------------------------------------------------------------------------------------------------------------
# Round-2 host logic: compact ingest, concurrent callers, per-batch publication into bound storage, several devices in one process.
# ---------------------------------------------------------------------------------------------------------------------------------------------
SCRIPT_MIX = ("r = rdf(element('O'), element('O'), 6.0); v = sdf(residue(1:20), element('O'), 5.0); dz = density_z(element('O')); "
              "d = distance(1,10); dp = distance_pair(atom(1:5), atom(20:30)); rm = rmsd(residue(1:10)); a = angle(1,2,3) in residue(1:10); "
              "dfar = distance(200, 401); cfar = com(500);")   # single atoms beyond the dense part of the compact space


def _mix_results(plan):
    import numpy as np
    out = {k: plan.counts(k) for k in ("r", "v", "dz")}
    for k in ("d", "dp", "rm", "a", "dfar", "cfar"): out[k] = plan.property_data(k).values.copy()
    out["r_w"] = plan.property_data("r").weights.copy(); out["mask"] = plan.frame_mask()
    out["dp_mean"] = plan.aggregate("dp")["mean"].copy()
    out["minmax"] = np.array([[plan.property_data(k).min_value, plan.property_data(k).max_value] for k in ("r", "dz", "d", "dp")], np.float32)
    return out


def _golden_mix(api):
    import viamd_b200 as vb
    from helpers import load_golden, golden_system, vb_system, vb_cell
    g = load_golden("water6.npz"); s = golden_system(g); sysm = vb_system(s); F = g["frames"].shape[0]
    cells = [vb_cell(g["cells"][f], g["cell_flags"][f]) for f in range(F)]
    return vb, g, sysm, F, cells


def _same(a, b):
    import numpy as np
    assert a.keys() == b.keys()
    for k in a: assert np.array_equal(a[k], b[k]), k


def test_compact_ingest_copies_only_the_atoms_the_properties_read(emulated_library):
    """Host ingest gathers the atoms the properties read (here the O atoms + the first residues: 224 of 648) into the staging buffers and the
    kernels run on index lists remapped into that compact space: results identical to whole-frame ingest (ingest_mode=1), for host frames
    and for the md_trajectory_i frame source, pageable memory."""
    vb, g, sysm, F, cells = _golden_mix(emulated_library)
    res = {}
    for mode in (0, 1):
        for src in ("host", "traj"):
            plan = vb.Plan(sysm, vb.compile_script(SCRIPT_MIX, sysm), F, batch_frames=3, ingest_mode=mode)
            na, nt = plan.ingest_info()
            assert (60 < na < 300 and nt >= 1) if mode == 0 else (na == 648)
            plan.set_initial_frame(*g["frames"][0], cells[0])
            if src == "host": plan.eval_host_frames(g["frames"], cells, 0)
            else: assert plan.eval_frame_range(vb.ArrayTrajectory(g["frames"], cells), 0, F, loader_threads=2)
            res[(mode, src)] = _mix_results(plan); plan.close()
    for k in ((0, "traj"), (1, "host"), (1, "traj")): _same(res[(0, "host")], res[k])
    assert res[(0, "host")]["r"].sum() > 0 and res[(0, "host")]["v"].sum() > 0


def test_concurrent_disjoint_ranges_on_one_plan(emulated_library):
    """md_script_eval_frame_range is re-entrant on one eval from many threads with disjoint ranges (VIAMD's enkiTS range task,
    src/task_system.cpp:73-87; mdlib/unittest/test_script.c:1352-1417 `parallel_evaluation` demands exact equality): four threads, one frame
    each, one plan, two stream slots -> the results of a single call over the whole range."""
    import threading
    vb, g, sysm, F, cells = _golden_mix(emulated_library)
    traj = vb.ArrayTrajectory(g["frames"], cells); traj._as_c()
    ref = vb.Plan(sysm, vb.compile_script(SCRIPT_MIX, sysm), F); ref.eval_frame_range(traj, 0, F); want = _mix_results(ref); ref.close()
    for rep in range(3):
        plan = vb.Plan(sysm, vb.compile_script(SCRIPT_MIX, sysm), F, batch_frames=1, num_streams=2)
        plan.set_initial_frame(*g["frames"][0], cells[0])
        ok = [False] * F
        def work(f): ok[f] = plan.eval_frame_range(traj, f, f + 1, loader_threads=1) and (plan.sync() is None)
        th = [threading.Thread(target=work, args=(f,)) for f in range(F)]
        for t in th: t.start()
        for t in th: t.join()
        assert all(ok)
        _same(want, _mix_results(plan)); plan.close()


def test_progress_callback_publishes_batches_into_bound_storage(emulated_library):
    """The md_script shim's contract: values are written into caller-owned arrays (md_script_property_data_t::values), and after every
    completed batch the callback fires with that batch's frames while their temporal rows are already in place (src/main.cpp:1513-1524 reads
    them while the evaluation runs)."""
    import numpy as np
    vb, g, sysm, F, cells = _golden_mix(emulated_library)
    plan = vb.Plan(sysm, vb.compile_script(SCRIPT_MIX, sysm), F, batch_frames=1)
    plan.set_initial_frame(*g["frames"][0], cells[0])
    d_vals = np.full(F, -1.0, np.float32); dp_vals = np.zeros(F * 55, np.float32); r_vals = np.zeros(2048, np.float32)
    dp_mean = np.zeros(F, np.float32); dp_var = np.zeros(F, np.float32); dp_ext = np.zeros(2 * F, np.float32)
    plan.bind_property_storage("d", d_vals); plan.bind_property_storage("dp", dp_vals, dp_mean, dp_var, dp_ext); plan.bind_property_storage("r", r_vals)
    seen = []
    def on_batch(beg, cnt):
        seen.append((beg, cnt, d_vals[beg:beg + cnt].copy(), dp_mean[beg:beg + cnt].copy()))
    plan.set_progress_callback(on_batch)
    plan.eval_host_frames(g["frames"], cells, 0); plan.sync()
    assert sorted(b for b, _, _, _ in seen) == list(range(F)) and all(c == 1 for _, c, _, _ in seen)
    pz = __import__("helpers").load_golden("pairs6.npz")
    for beg, cnt, dv, dm in seen:
        assert dv[0] == g["d__full"][beg] and dm[0] == pz["w_dp__mean"][beg]        # the row was in place when the callback ran
    assert np.array_equal(d_vals, g["d__full"]) and np.array_equal(dp_vals, pz["w_dp__full"]) and np.array_equal(dp_mean, pz["w_dp__mean"])
    np.testing.assert_allclose(r_vals[:1024], g["r__full"][:1024], rtol=1e-5, atol=1e-6)
    plan.close()


def test_several_devices_in_one_process_merge_at_sync(emulated_library, monkeypatch):
    """mdgpu_plan_options_t.num_devices = 2 (SURVEY 8(e) inside the C++ library, for the one-process VIAMD): contiguous frame blocks per device,
    every accumulator reduced onto devices[0] by the exchange step at sync (NCCL bound at run time; here tests/emul/fake_nccl.cpp on the
    emulated runtime's shared heap). Results, frame mask, weights and min/max equal the single-device evaluation; a second sync changes nothing;
    evaluating the second half later merges exactly once."""
    import build_emul
    monkeypatch.setenv("MDGPU_EMUL_DEVICES", "2"); monkeypatch.setenv("MDGPU_NCCL_LIB", build_emul.build_fake_nccl())
    vb, g, sysm, F, cells = _golden_mix(emulated_library)
    one = vb.Plan(sysm, vb.compile_script(SCRIPT_MIX, sysm), F, keep_frame_results=True); one.set_initial_frame(*g["frames"][0], cells[0])
    one.eval_host_frames(g["frames"], cells, 0); want = _mix_results(one); one.close()
    for src in ("host", "traj"):
        plan = vb.Plan(sysm, vb.compile_script(SCRIPT_MIX, sysm), F, keep_frame_results=True, devices=[0, 1])
        plan.set_initial_frame(*g["frames"][0], cells[0])
        if src == "host": plan.eval_host_frames(g["frames"], cells, 0)
        else: assert plan.eval_frame_range(vb.ArrayTrajectory(g["frames"], cells), 0, F, loader_threads=2)
        _same(want, _mix_results(plan)); plan.sync(); _same(want, _mix_results(plan))
        assert plan.exchange_stats()[1] == 1
        bins, tot = plan.frame_counts("r", F - 1); assert tot == int(bins.sum()) > 0       # a frame the second device evaluated
        plan.clear()
        plan.eval_host_frames(g["frames"][:2], cells[:2], 0); plan.sync(); plan.eval_host_frames(g["frames"][2:], cells[2:], 2)
        _same(want, _mix_results(plan))
        plan.close()


def test_rdf_kernel_variants_under_emulation(emulated_library):
    """rdf_variant 2 (3 CTAs / SM, longer hit queue; the default has 4) and 4 (TMA-staged reference chunks; the bulk copy + mbarrier helpers are emulated by a
    memcpy and a phase counter) give the reference's per-frame bins, orthorhombic goldens."""
    import numpy as np
    import test_gpu_parity as G
    from helpers import load_golden, golden_system
    g = load_golden("water6.npz"); s = golden_system(g)
    for variant in (2, 4):
        plan, cells = G._water_plan(g, s, "r = rdf(element('O'), element('O'), 6.0); rh = rdf(element('O'), element('H'), 1.5:6.0);", rdf_variant=variant)
        plan.eval_host_frames(g["frames"], cells, 0)
        for key in ("r", "rh"):
            for f in range(g["frames"].shape[0]):
                bins, tot = plan.frame_counts(key, f)
                assert np.array_equal(bins.astype(np.float32), g[f"{key}__pf"][f, :1024]) and tot == int(bins.sum()), (variant, key, f)
        plan.close()


PROBE_FORMS = [   # statement forms compared with the UNMODIFIED reference's results (tests/golden/forms45.npz): the sweep that found the silently
    # flattened rdf target, the missing triclinic min-image of dihedral and the context-relative selections
    "p01 = rdf(residue(1:30), element('O'), 1.0:7.0);", "p02 = rdf(atom(1), atom(2:648), 8.0);", "p03 = rdf(element('H'), element('H'), 5.5);",
    "p04 = sdf(residue(1:30), within(5.0, residue(1:3)), 4.0);", "p05 = density_x(element('O'));", "p06 = density_y(within(6.0, residue(1:5)));",
    "p07 = rdf(within(3.0:6.0, residue(1)), element('H'), 4.0);", "p08 = rdf(element('O') and within(5.0, residue(2)), element('H') and within(6.0, residue(3)), 5.0);",
    "p09 = count(within(2.0, atom(1)));", "p10 = contact_count(residue(1:5), residue(10:40), 4.0);", "p11 = distance(within(4.0, residue(1)), 200);",
    "p12 = com(within(4.0, residue(1)));", "p13 = dihedral(1, 100, 300, 500);", "p14 = angle(1, 200, 400);", "p15 = distance(1, 600);",
    "p16 = distance(residue(1), residue(100));", "p17 = distance_min(residue(1:3), residue(100:120));", "p18 = rmsd(residue(1:50));", "p19 = com(element('O'));",
    "p20 = plane(atom(1:200));", "p21 = distance_pair(atom(1:3), atom(400:402));", "p22 = count(within(6.0, atom(1:3)));",
    "p23 = rdf(atom(1:100), atom(50:150), 6.0);", "p24 = rdf(atom(1:3), atom(2:2), 8.0);", "p25 = sdf(residue(1:4), atom(1:200), 5.0);",
    "p26 = rdf(residue(1:20), residue(10:30), 5.0);", "p27 = rdf(element('O'), all, 4.0);", "p28 = sdf(residue(1:10), residue(20:40), 5.0);",
    "p29 = density_z(residue(1:10));", "p30 = rdf(element('O') and residue(1:50), element('H') or atom(1:3), 5.0);", "p31 = rdf(not element('H'), all, 3.0);",
    "p32 = distance(element('O'), element('H')) in residue(1:10);", "p33 = angle(atom(2), element('O'), 3) in residue(1:5);",
    "p34 = dihedral(1, element('O'), atom(2:3), 3) in residue(:);", "p35 = angle(com(element('H')), 1, 2) in residue(3:40);",
    "p36 = distance_min(residue(1), residue(2:9));", "p37 = distance_max(residue(3:5), element('O'));", "p38 = coord_x(residue(1:5));", "p39 = plane(residue(1:10));",
    "p40 = angle(residue(1:2), residue(5:7), 30);", "p41 = com(residue(1:6));", "p42 = distance(com(residue(1:4)), residue(50:52));",
    "p43 = rdf(element('O'), element('O'), 12.0);", "p44 = sdf(residue(1:10), element('O'), 12.0);", "p45 = distance_pair(residue(1), residue(2:5));",
]


@pytest.mark.parametrize("golden,seed", [("water6.npz", "77"), ("tric6.npz", "91")])
def test_statement_forms_against_the_reference_itself(emulated_library, golden, seed):
    """45 statement forms in ONE script: the unmodified reference's evaluation of 2 frames of the golden box (tests/golden/forms45.npz, made by
    tests/golden/make_golden.py) against the library (emulated build) evaluating the Python mirror's lowering of the same statements; distributions
    and volumes must agree count for count, temporals within 1e-5 (bit-equal for distances). Orthorhombic and changing triclinic cell."""
    run_statement_forms(golden, seed)


def run_statement_forms(golden, seed):
    """(also called by tests/test_zz_gpu_new_ops.py with the real library on the device)"""
    import numpy as np
    import refio
    import viamd_b200 as vb
    from helpers import load_golden, golden_system, vb_system, vb_cell, dense_from_sparse
    g = load_golden(golden); sysm = vb_system(golden_system(g)); F = 2; script = " ".join(PROBE_FORMS)
    ref = load_golden("forms45.npz"); tag = golden[0]   # w(ater6) / t(ric6)
    assert str(ref["script"]) == script and int(ref[f"{tag}_seed"]) == int(seed), "forms45.npz is stale: regenerate it with make_golden.py forms45"
    props = vb.compile_script(script, sysm)
    plan = vb.Plan(sysm, props, F, keep_frame_results=True); cells = [vb_cell(g["cells"][f], g["cell_flags"][f]) for f in range(F)]
    plan.set_initial_frame(*g["frames"][0], cells[0]); plan.eval_host_frames(g["frames"][:F], cells, 0)
    for p in props:
        k = f"{tag}_{p.name}"; flags = int(ref[k + "__flags"]); d = plan.property_data(p.name)
        if flags & refio.FLAG_VOLUME:
            want = sum(dense_from_sparse(ref[f"{k}__pf{f}_idx"], ref[f"{k}__pf{f}_val"]) for f in range(F))
            assert np.array_equal(plan.counts(p.name).astype(np.float32), want), p.name
        elif flags & refio.FLAG_TEMPORAL:
            a, b = np.asarray(d.values).ravel(), ref[k + "__full"].ravel()
            assert a.shape == b.shape and np.allclose(a, b, rtol=1e-5, atol=1e-6), (p.name, a[:4], b[:4])
        elif p.op == vb.OP_RDF:
            for f in range(F): assert np.array_equal(plan.frame_counts(p.name, f)[0].astype(np.float32), ref[k + "__pf"][f, :1024]), (p.name, f)
        else:
            assert np.allclose(d.values[:1024], ref[k + "__full"][:1024], rtol=1e-5, atol=1e-3), p.name
    plan.close()
