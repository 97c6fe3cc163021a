"""Parity tests proper: the CUDA path (through the libmdgpu C ABI) against the golden vectors of the unmodified reference
and against the plain-C oracle on seeded inputs. Integer work is asserted bit-exact; float temporals within 1e-5 relative
(BASELINE.json north_star tolerance; acosf/atan2f differ in the last ulp between glibc and CUDA)."""
import os

import numpy as np
import pytest

import oracle_lib as O
from helpers import load_golden, cell_from_row, dense_from_mask, dense_from_sparse, golden_system, sel_element, vb_system, vb_cell

pytestmark = pytest.mark.gpu
RTOL = 1e-5   # north_star: "within 1e-5 relative for float densities"


def _vb():
    import viamd_b200 as vb
    return vb


def _water_plan(g, s, props_src, **kw):
    vb = _vb()
    sysm = vb_system(s)
    props = vb.compile_script(props_src, sysm)
    F = g["frames"].shape[0]
    plan = vb.Plan(sysm, props, F, keep_frame_results=True, **kw)
    cells = [vb_cell(g["cells"][f], g["cell_flags"][f]) for f in range(F)]
    plan.set_initial_frame(*g["frames"][0], cells[0])
    return plan, cells


def test_golden_water_rdf_per_frame_bitexact():
    g = load_golden("water6.npz"); s = golden_system(g); vb = _vb()
    plan, cells = _water_plan(g, s, "r = rdf(element('O'), element('O'), 6.0); rh = rdf(element('O'), element('H'), 1.5:6.0);")
    F = g["frames"].shape[0]
    plan.eval_host_frames(g["frames"], cells, 0)
    for key in ("r", "rh"):
        acc = np.zeros(1024, np.float64)
        for f in range(F):
            bins, tot = plan.frame_counts(key, f)
            ref = g[f"{key}__pf"][f, :1024]
            assert np.array_equal(bins.astype(np.float32), ref), f"{key} frame {f}"
            assert tot == int(ref.sum())
            acc += ref
        assert np.array_equal(plan.counts(key).astype(np.float64), acc)
        d = plan.property_data(key)
        assert d.dim == (1, 2, 1024, 0) and d.frames_accumulated == F
        # averaged bins: exact mean vs the reference's float cumulative moving average
        np.testing.assert_allclose(d.values[:1024], g[f"{key}__full"][:1024], rtol=RTOL, atol=1e-6)
        np.testing.assert_allclose(d.values[:1024], (acc / F).astype(np.float32), rtol=0, atol=0)
        # weights are those of the last frame (bit-exact: same double arithmetic)
        assert np.array_equal(d.weights, g[f"{key}__pf"][F - 1, 1024:])
        mn, mx, r0, r1 = g[f"{key}__meta"]
        assert d.min_value == mn and d.max_value == mx and d.min_range[0] == r0 and d.max_range[0] == r1
    assert plan.frame_mask().all()
    plan.close()


def test_golden_water_rdf_com_references_bitexact():
    """rdf(residue(1:20), element('O'), 5.0): array-of-selections reference -> centres of mass + exclusion masks (compute_rdf :5274)."""
    g = load_golden("water6.npz"); s = golden_system(g)
    plan, cells = _water_plan(g, s, "rc = rdf(residue(1:20), element('O'), 5.0);", batch_frames=3)
    F = g["frames"].shape[0]
    plan.eval_host_frames(g["frames"], cells, 0)
    for f in range(F):
        bins, tot = plan.frame_counts("rc", f)
        assert np.array_equal(bins.astype(np.float32), g["rc__pf"][f, :1024]) and tot == int(g["rc__pf"][f, :1024].sum()) > 0
    d = plan.property_data("rc")
    assert np.array_equal(d.weights, g["rc__pf"][F - 1, 1024:])
    np.testing.assert_allclose(d.values[:1024], g["rc__full"][:1024], rtol=RTOL, atol=1e-6)
    plan.close()


def test_oracle_rdf_com_references_larger():
    """400 water molecules as centre-of-mass references against all oxygens of a 1536-atom box, device-resident frames, vs the oracle."""
    vb = _vb()
    n, seed, F = 8, 4242, 5
    base, L = vb.synth_water_base(n, seed)
    frames = vb.synth_water_frames_host(n, seed, base, 0, F)
    sysm = vb.water_system(n)
    groups = [np.arange(3 * r, 3 * r + 3, dtype=np.int32) for r in range(50, 450)]
    trg = np.arange(0, 3 * n ** 3, 3, dtype=np.int32)
    plan = vb.Plan(sysm, [vb.rdf_com("rc", groups, trg, 9.0, 0.5)], F, keep_frame_results=True, batch_frames=2)
    cell = vb.UnitCell.from_basis(L, L, L); oc = O.UnitCell.ortho(L, L, L)
    plan.eval_host_frames(frames, cell, 0)
    for f in range(F):
        pos, off, idx = O.group_com(*frames[f], sysm.mass, groups)
        ob, ow, ot = O.rdf_frame(*frames[f], None, trg, oc, 0.5, 9.0, ref_pos=pos, excl_off=off, excl_idx=idx)
        bins, tot = plan.frame_counts("rc", f)
        assert tot == ot > 0 and np.array_equal(bins.astype(np.float32), ob), f"frame {f}"
    assert np.array_equal(plan.property_data("rc").weights, ow)
    plan.close()


def test_golden_triclinic_rdf_bitexact():
    """Reference-generated golden in a triclinic cell that changes every frame: plain, min:max and centre-of-mass reference rdf()."""
    g = load_golden("tric6.npz"); s = golden_system(g)
    plan, cells = _water_plan(g, s, str(g["script"]), batch_frames=3)
    F = g["frames"].shape[0]
    total = np.zeros(128 ** 3, np.float64)
    for f in range(F):   # sdf() in a triclinic cell, per-frame raw voxels (incl. the reference's fractional-coordinate callback quirk)
        plan.clear(); plan.eval_host_frames(g["frames"][f:f + 1], [cells[f]], f)
        ref = dense_from_sparse(g[f"vt__pf{f}_idx"], g[f"vt__pf{f}_val"]); got = plan.counts("vt")
        assert int(got.sum()) == int(ref.sum()) > 0 and np.array_equal(got.astype(np.float32), ref), f"vt frame {f}"
        total += ref
    plan.clear()
    plan.eval_host_frames(g["frames"], cells, 0)
    assert np.array_equal(plan.counts("vt").astype(np.float64), total)
    for key in ("dmt", "dmxt"):   # distance_min / distance_max with the 27-image triclinic minimum
        assert np.array_equal(plan.property_data(key).values, g[f"{key}__full"]), key
    for key in ("rt", "rth", "rtc"):
        for f in range(F):
            bins, tot = plan.frame_counts(key, f)
            assert np.array_equal(bins.astype(np.float32), g[f"{key}__pf"][f, :1024]) and tot == int(g[f"{key}__pf"][f, :1024].sum()) > 0, (key, f)
        d = plan.property_data(key)
        assert np.array_equal(d.weights, g[f"{key}__pf"][F - 1, 1024:])
        np.testing.assert_allclose(d.values[:1024], g[f"{key}__full"][:1024], rtol=RTOL, atol=1e-6)
    plan.close()


def test_golden_water_sdf_per_frame_bitexact():
    g = load_golden("water6.npz"); s = golden_system(g)
    plan, cells = _water_plan(g, s, "v = sdf(residue(1:20), element('O'), 5.0);")
    F = g["frames"].shape[0]
    total = np.zeros(128 ** 3, np.float64)
    for f in range(F):   # per-frame raw voxels: evaluate one frame into cleared accumulators
        plan.clear()
        plan.eval_host_frames(g["frames"][f:f + 1], [cells[f]], f)
        ref = dense_from_sparse(g[f"v__pf{f}_idx"], g[f"v__pf{f}_val"])
        got = plan.counts("v")
        assert int(got.sum()) == int(ref.sum()) > 0
        assert np.array_equal(got.astype(np.float32), ref), f"frame {f}: {(got.astype(np.float32) != ref).sum()} voxels differ"
        total += ref
    plan.clear()
    plan.eval_host_frames(g["frames"], cells, 0)
    assert np.array_equal(plan.counts("v").astype(np.float64), total)
    d = plan.property_data("v")
    assert d.dim == (1, 128, 128, 128)
    ref_full = dense_from_sparse(g["v__full_idx"], g["v__full_val"])
    np.testing.assert_allclose(d.values, ref_full, rtol=RTOL, atol=1e-7)
    assert d.min_value == np.float32(3.4028234663852886e+38) and d.max_value == -np.float32(3.4028234663852886e+38)   # never updated for volumes
    plan.close()


def test_golden_water_density_and_temporals():
    g = load_golden("water6.npz"); s = golden_system(g)
    plan, cells = _water_plan(g, s, "dz = density_z(element('O')); dx = density_x(element('O')); d = distance(1,10); a = angle(1,2,3); t = dihedral(1,4,7,10); "
                            "dc = distance(residue(1), residue(5)); ac = angle(residue(1), residue(2), residue(3)); "
                            "tc = dihedral(residue(1), residue(2), residue(3), residue(4)); dg = distance(atom(1:30), atom(100:151)); dm = distance(atom(1:30), 200); "
                            "dmn = distance_min(residue(1), atom(100:648)); dmx = distance_max(atom(1:30), atom(100:151)); dmh = distance_min(element('H'), atom(300:400));")
    F = g["frames"].shape[0]
    plan.eval_host_frames(g["frames"], cells, 0)
    for key in ("dmn", "dmx", "dmh"):   # brute-force pair minimum (distance_max evaluates the minimum in the reference too)
        assert np.array_equal(plan.property_data(key).values, g[f"{key}__full"]), key
    # arguments that are selections: periodic centre of mass (md_util_com_compute), lane-by-lane restatement of the AVX2 reference
    for key in ("dc", "dg", "dm"):
        assert np.array_equal(plan.property_data(key).values, g[f"{key}__full"]), key      # distances: every operation is IEEE on both sides
    np.testing.assert_allclose(plan.property_data("ac").values, g["ac__full"], rtol=RTOL)
    np.testing.assert_allclose(plan.property_data("tc").values, g["tc__full"], rtol=RTOL)
    for key in ("dz", "dx"):
        d = plan.property_data(key)
        np.testing.assert_allclose(d.values[:1024], g[f"{key}__full"][:1024], rtol=RTOL, atol=1e-3)
        assert np.all(d.weights == 1.0)
        mn, mx, r0, r1 = g[f"{key}__meta"]
        assert d.min_value == mn and abs(d.max_value - mx) <= RTOL * mx and d.min_range[0] == r0 and d.max_range[0] == r1
    d = plan.property_data("d")
    assert d.dim[:2] == (F, 1)
    assert np.array_equal(d.values, g["d__full"])                                  # sqrt is correctly rounded on both sides
    np.testing.assert_allclose(plan.property_data("a").values, g["a__full"], rtol=RTOL)
    np.testing.assert_allclose(plan.property_data("t").values, g["t__full"], rtol=RTOL)
    mn, mx, r0, r1 = g["d__meta"]
    assert d.min_value == mn and d.max_value == mx and d.min_range[0] == r0 and d.max_range[0] == r1
    plan.close()


def test_golden_config1_1ala_distance_and_friends():
    """BASELINE config 1 (datasets/1ALA-500.pdb, d = distance(1,10)) on the first 50 frames + rdf/density/angle/dihedral."""
    g = load_golden("ala50.npz"); s = golden_system(g); vb = _vb()
    sysm = vb_system(s)
    script = ";".join(st for st in str(g["script"]).split(";") if "rmsd(" not in st)   # rmsd: pinned in the oracle only, outside the GPU scope so far
    props = vb.compile_script(script, sysm)
    F = g["frames"].shape[0]
    plan = vb.Plan(sysm, props, F, keep_frame_results=True, batch_frames=16)
    cells = [vb_cell(g["cells"][f], g["cell_flags"][f]) for f in range(F)]
    traj = vb.ArrayTrajectory(g["frames"], cells)
    assert plan.eval_frame_range(traj, 0, F)          # md_script_eval_frame_range path (frame source interface)
    d = plan.property_data("d")
    assert np.array_equal(d.values, g["d__full"]) and abs(float(d.values[0]) - 2.770258) < 1e-6
    np.testing.assert_allclose(plan.property_data("a").values, g["a__full"], rtol=RTOL)
    np.testing.assert_allclose(plan.property_data("t").values, g["t__full"], rtol=RTOL, atol=1e-6)
    assert np.array_equal(plan.property_data("dr").values, g["dr__full"])      # distance between residue centres of mass (periodic, trigonometric)
    np.testing.assert_allclose(plan.property_data("ar").values, g["ar__full"], rtol=RTOL)
    np.testing.assert_allclose(plan.property_data("tr").values, g["tr__full"], rtol=RTOL, atol=1e-6)
    for f in range(F):
        for key in ("rc", "rr"):   # rr: centre-of-mass references of three residues of different sizes, own atoms excluded
            bins, tot = plan.frame_counts(key, f)
            assert np.array_equal(bins.astype(np.float32), g[f"{key}__pf"][f, :1024]) and tot == int(g[f"{key}__pf"][f, :1024].sum()), f"{key} frame {f}"
    assert np.array_equal(plan.property_data("rr").weights, g["rr__pf"][F - 1, 1024:])
    np.testing.assert_allclose(plan.property_data("dz").values[:1024], g["dz__full"][:1024], rtol=RTOL, atol=1e-3)
    assert plan.frame_mask().all()
    plan.close()


@pytest.mark.parametrize("n,cutoff,ref_el,trg_el", [(8, 10.0, 8, 8), (8, 5.0, 8, 1), (10, 12.0, 1, 8), (5, 4.0, 8, 8)])
def test_oracle_water_rdf_bitexact(n, cutoff, ref_el, trg_el):
    """Seeded synthetic water of several sizes / cutoffs (cdim from 1 to 3, duplicated periodic images when the cutoff
    exceeds half the box, see SURVEY.md §7) against the oracle, through device-generated frames."""
    vb = _vb()
    seed, F = 1000 + n, 6
    base, L = vb.synth_water_base(n, seed)
    frames = vb.synth_water_frames_host(n, seed, base, 0, F)
    sysm = vb.water_system(n)
    el = np.tile(np.array([8, 1, 1]), n ** 3)
    ref = np.nonzero(el == ref_el)[0].astype(np.int32); trg = np.nonzero(el == trg_el)[0].astype(np.int32)
    plan = vb.Plan(sysm, [vb.rdf("r", ref, trg, cutoff)], F, keep_frame_results=True, batch_frames=4)
    cell = vb.UnitCell.from_basis(L, L, L)
    # device-resident frames generated on the GPU must equal the host generator bit for bit
    na = 3 * n ** 3
    d_base = vb.device_alloc(0, base.nbytes); vb.memcpy_h2d(0, d_base, base.ctypes.data, base.nbytes)
    d_fr = vb.device_alloc(0, frames.nbytes)
    vb.synth_water_frames_device(0, n, seed, d_base, 0, F, d_fr, 3 * na, na)
    back = np.empty_like(frames); vb.memcpy_d2h(0, back.ctypes.data, d_fr, frames.nbytes)
    assert np.array_equal(back, frames)
    plan.eval_device_frames(d_fr, 3 * na, na, cell, 0, F)
    ocell = O.UnitCell.ortho(L, L, L)
    for f in range(F):
        bins, tot = plan.frame_counts("r", f)
        obins, ow, otot = O.rdf_frame(frames[f, 0], frames[f, 1], frames[f, 2], ref, trg, ocell, 0.0, cutoff)
        assert tot == otot
        assert np.array_equal(bins.astype(np.float32), obins), f"frame {f}"
    assert np.array_equal(plan.property_data("r").weights, ow)
    vb.device_free(0, d_base); vb.device_free(0, d_fr)
    plan.close()


def test_oracle_random_boxes_rdf_bitexact():
    """Random points in anisotropic / partially periodic / non-periodic cells (edge cases of md_spatial_acc_init:
    AABB-fitted origin, skipped non-periodic wraps), ragged sizes, empty-ish cells."""
    vb = _vb(); rng = np.random.default_rng(11)
    cases = [
        (dict(x=31.0, y=47.5, z=23.25), 4 | 8 | 16 | 1, 500, 7.5),
        (dict(x=40.0, y=40.0, z=40.0), 4 | 8 | 1, 300, 9.0),        # z not periodic
        (dict(x=0.0, y=0.0, z=0.0), 0, 257, 6.0),                   # no cell at all
        (dict(x=25.0, y=25.0, z=60.0), 4 | 8 | 16 | 1, 33, 12.0),   # cutoff ~ half box: cdim 2
        (dict(x=18.0, y=18.0, z=18.0), 4 | 8 | 16 | 1, 64, 17.0),   # cutoff > half box: periodic images counted per offset
    ]
    for cellp, flags, N, cutoff in cases:
        ext = np.array([cellp["x"] or 50.0, cellp["y"] or 50.0, cellp["z"] or 50.0])
        F = 3
        frames = (rng.random((F, 3, N)) * ext[None, :, None] * 1.2 - 0.1 * ext[None, :, None]).astype(np.float32)   # some atoms outside the cell
        ref = np.sort(rng.choice(N, N // 2, replace=False)).astype(np.int32); trg = np.sort(rng.choice(N, (2 * N) // 3, replace=False)).astype(np.int32)
        sysm = vb.System(N, np.ones(N, np.float32))
        plan = vb.Plan(sysm, [vb.rdf("r", ref, trg, cutoff)], F, keep_frame_results=True, batch_frames=2)
        cell = vb.UnitCell(cellp["x"], 0, 0, cellp["y"], 0, cellp["z"], flags)
        plan.eval_host_frames(frames, cell, 0)
        ocell = O.UnitCell.from_params(cellp["x"], 0, 0, cellp["y"], 0, cellp["z"], flags)
        for f in range(F):
            bins, tot = plan.frame_counts("r", f)
            obins, ow, otot = O.rdf_frame(frames[f, 0], frames[f, 1], frames[f, 2], ref, trg, ocell, 0.0, cutoff)
            assert tot == otot, (cellp, flags, f, tot, otot)
            assert np.array_equal(bins.astype(np.float32), obins), (cellp, flags, f)
        plan.close()


def test_oracle_triclinic_rdf_bitexact():
    vb = _vb(); rng = np.random.default_rng(5)
    N, F, cutoff = 400, 3, 7.0
    cellp = (30.0, 4.0, -3.0, 28.0, 5.0, 26.0)   # x, xy, xz, y, yz, z
    flags = 2 | 4 | 8 | 16
    # points inside the cell: fractional coords in [0,1) mapped through A
    s = rng.random((F, 3, N))
    A = np.array([[cellp[0], cellp[1], cellp[2]], [0, cellp[3], cellp[4]], [0, 0, cellp[5]]])
    frames = np.einsum("ij,fjn->fin", A, s).astype(np.float32)
    idx = np.arange(N, dtype=np.int32)
    plan = vb.Plan(vb.System(N, np.ones(N, np.float32)), [vb.rdf("r", idx[::2], idx, cutoff)], F, keep_frame_results=True)
    plan.eval_host_frames(frames, vb.UnitCell(cellp[0], cellp[1], cellp[2], cellp[3], cellp[4], cellp[5], flags), 0)
    ocell = O.UnitCell.from_params(*cellp, flags)
    for f in range(F):
        bins, tot = plan.frame_counts("r", f)
        obins, ow, otot = O.rdf_frame(frames[f, 0], frames[f, 1], frames[f, 2], idx[::2], idx, ocell, 0.0, cutoff)
        assert tot == otot and np.array_equal(bins.astype(np.float32), obins)
    plan.close()


def test_oracle_water_sdf_bitexact_and_batching():
    """sdf() on seeded water vs the oracle, bit-exact voxels; result independent of batch size / stream count."""
    vb = _vb()
    n, seed, F = 8, 4242, 5
    base, L = vb.synth_water_base(n, seed); frames = vb.synth_water_frames_host(n, seed, base, 0, F)
    sysm = vb.water_system(n)
    o = np.arange(0, 3 * n ** 3, 3, dtype=np.int32)
    structs = np.arange(3 * 100, dtype=np.int32).reshape(100, 3)
    cell = vb.UnitCell.from_basis(L, L, L); ocell = O.UnitCell.ortho(L, L, L)
    ref = np.zeros(128 ** 3, np.float32)
    for f in range(F):
        O.sdf_frame(frames[f, 0], frames[f, 1], frames[f, 2], frames[0], sysm.mass, structs, o, sysm.conn_offset, sysm.conn_idx, ocell, 6.0, vol=ref)
    results = []
    for bf, ns in ((1, 1), (3, 2), (0, 0)):
        plan = vb.Plan(sysm, [vb.sdf("v", structs, o, 6.0)], F, batch_frames=bf, num_streams=ns)
        plan.set_initial_frame(*frames[0], cell)
        plan.eval_host_frames(frames, cell, 0)
        results.append(plan.counts("v")); plan.close()
    assert int(results[0].sum()) == int(ref.sum()) > 0
    assert np.array_equal(results[0].astype(np.float32), ref)
    assert np.array_equal(results[0], results[1]) and np.array_equal(results[0], results[2])
    # non-contiguous structures (O + second H of each molecule): exercises the general exclusion-mask path
    st2 = np.stack([np.arange(60) * 3, np.arange(60) * 3 + 2], axis=1).astype(np.int32)
    ref2 = np.zeros(128 ** 3, np.float32)
    for f in range(F):
        O.sdf_frame(frames[f, 0], frames[f, 1], frames[f, 2], frames[0], sysm.mass, st2, o, sysm.conn_offset, sysm.conn_idx, ocell, 7.5, vol=ref2)
    plan = vb.Plan(sysm, [vb.sdf("v", st2, o, 7.5)], F)
    plan.set_initial_frame(*frames[0], cell); plan.eval_host_frames(frames, cell, 0)
    assert np.array_equal(plan.counts("v").astype(np.float32), ref2) and ref2.sum() > 0
    plan.close()


def test_empty_and_error_paths():
    vb = _vb()
    s = vb.water_system(3)
    o = np.arange(0, 81, 3, dtype=np.int32)
    with pytest.raises(vb.MdgpuError, match="empty reference"):
        vb.Plan(s, [vb.rdf("r", np.zeros(0, np.int32), o, 5.0)], 2)
    with pytest.raises(vb.MdgpuError, match="Invalid cutoff"):
        vb.Plan(s, [vb.rdf("r", o, o, 5.0, cutoff_min=6.0)], 2)
    with pytest.raises(vb.MdgpuError, match="out of range"):
        vb.Plan(s, [vb.rdf("r", np.array([1000], np.int32), o, 5.0)], 2)
    base, L = vb.synth_water_base(3, 1); frames = vb.synth_water_frames_host(3, 1, base, 0, 2)
    plan = vb.Plan(s, [vb.rdf("r", o, o, 5.0)], 2)
    with pytest.raises(vb.MdgpuError, match="Invalid frame range"):
        plan.eval_host_frames(frames, vb.UnitCell.from_basis(L, L, L), 1)
    # zero frames evaluated: property data stays cleared (weights 1, min/max +-FLT_MAX)
    d = plan.property_data("r")
    assert d.frames_accumulated == 0 and np.all(d.values[:1024] == 0) and np.all(d.weights == 1.0)
    # cutoff too large for the cell grid (2*ncell+1 > 5): the reference logs an error and yields no pairs
    plan2 = vb.Plan(s, [vb.rdf("r", o, o, 30.0)], 2, keep_frame_results=True)
    plan2.eval_host_frames(frames, vb.UnitCell.from_basis(L, L, L), 0)
    assert plan2.frame_counts("r", 0)[1] == 0
    ob, ow, ot = O.rdf_frame(frames[0, 0], frames[0, 1], frames[0, 2], o, o, O.UnitCell.ortho(L, L, L), 0.0, 30.0)
    assert ot == 0
    plan.close(); plan2.close()


def test_full_size_properties_config2_config3():
    """BASELINE config 2/3 shape (98 304 atoms): size-independent properties.
       - sum of RDF bins == pair total reported per frame; accumulated counts == sum of per-frame counts;
       - evaluating frames in two halves (or in reverse batch order) gives identical integer accumulators;
       - rdf(O,O) pair total equals the oracle's on one frame (the oracle finishes one frame in < 1 s)."""
    vb = _vb()
    n, seed, F = 32, 1234, 8
    base, L = vb.synth_water_base(n, seed); na = base.shape[1]
    d_base = vb.device_alloc(0, base.nbytes); vb.memcpy_h2d(0, d_base, base.ctypes.data, base.nbytes)
    d_fr = vb.device_alloc(0, F * 3 * na * 4)
    vb.synth_water_frames_device(0, n, seed, d_base, 0, F, d_fr, 3 * na, na)
    sysm = vb.water_system(n)
    o = np.arange(0, na, 3, dtype=np.int32)
    structs = np.arange(3000, dtype=np.int32).reshape(1000, 3)
    cell = vb.UnitCell.from_basis(L, L, L)
    props = [vb.rdf("r", o, o, 10.0), vb.sdf("v", structs, o, 10.0)]
    f0 = vb.synth_water_frames_host(n, seed, base, 0, 1)
    plan = vb.Plan(sysm, props, F, keep_frame_results=True)
    plan.set_initial_frame(*f0[0], cell)
    plan.eval_device_frames(d_fr, 3 * na, na, cell, 0, F)
    acc = plan.counts("r"); vol = plan.counts("v")
    per = [plan.frame_counts("r", f) for f in range(F)]
    assert all(int(b.sum()) == t for b, t in per)
    assert np.array_equal(acc, np.sum([b.astype(np.uint64) for b, _ in per], axis=0))
    ob, ow, ot = O.rdf_frame(f0[0, 0], f0[0, 1], f0[0, 2], o, o, O.UnitCell.ortho(L, L, L), 0.0, 10.0)
    assert per[0][1] == ot and np.array_equal(per[0][0].astype(np.float32), ob)
    # split evaluation, second half first
    plan.clear()
    plan.eval_device_frames(d_fr + 4 * 3 * na * 4, 3 * na, na, cell, 4, 4)
    plan.eval_device_frames(d_fr, 3 * na, na, cell, 0, 4)
    assert np.array_equal(plan.counts("r"), acc) and np.array_equal(plan.counts("v"), vol)
    assert 2.5e5 * F < int(vol.sum()) < 3.5e5 * F
    vb.device_free(0, d_base); vb.device_free(0, d_fr); plan.close()


def test_full_size_config2_config3_vs_reference_golden_voxel_for_voxel():
    """BASELINE configs 2 + 3 at FULL size (98 304 atoms; rdf(O,O,10) and sdf(residue(1:1000), O, 10), 1000 reference structures) against the
    strict reference's per-frame results (tests/golden/water32_full.npz): rdf bins + weights bit-exact, sdf voxels voxel for voxel, and the
    2-frame mean of both within 1e-5 of the reference's cumulative moving average."""
    import hashlib
    vb = _vb(); g = load_golden("water32_full.npz"); n, seed, F = int(g["n"]), int(g["seed"]), 2
    base, L = vb.synth_water_base(n, seed); frames = vb.synth_water_frames_host(n, seed, base, 0, F)
    for f in range(F): assert hashlib.sha256(np.ascontiguousarray(frames[f]).tobytes()).hexdigest() == str(g["frames_sha256"][f])
    sysm = vb.water_system(n)
    props = vb.compile_script(str(g["script"]), sysm)
    cell = vb_cell(g["cells"][0], g["cell_flags"][0])
    plan = vb.Plan(sysm, props, F, keep_frame_results=True)
    plan.set_initial_frame(*frames[0], cell)
    for f in range(F):      # one frame at a time: the volume accumulator then holds that frame's raw voxels
        plan.clear(); plan.eval_host_frames(frames[f:f + 1], cell, f)
        bins, tot = plan.frame_counts("r", f)
        assert np.array_equal(bins.astype(np.float32), g["r__pf"][f, :1024]) and tot == int(g["r__pf"][f, :1024].sum())
        assert np.array_equal(plan.property_data("r").weights, g["r__pf"][f, 1024:])
        ref = dense_from_mask(g[f"v__pf{f}_mask"], g[f"v__pf{f}_val"])
        vox = plan.counts("v")
        assert int(vox.sum()) == int(ref.sum()) > 2.5e5 and np.array_equal(vox.astype(np.float32), ref), f"sdf frame {f}"
    plan.clear(); plan.eval_host_frames(frames, cell, 0)
    np.testing.assert_allclose(plan.property_data("r").values[:1024], g["r__full"][:1024], rtol=RTOL, atol=0)
    np.testing.assert_allclose(plan.property_data("v").values, dense_from_mask(g["v__full_mask"], g["v__full_val"]), rtol=RTOL, atol=0)
    plan.close()


def test_long_run_average_4096_frames_vs_reference_cma():
    """4096-frame averaged rdf bins, sdf voxels and density_z profile (water n=12, frames generated on the device) against the reference's
    single-thread run (tests/golden/water12_avg.npz). The product returns the exact mean of the integer per-frame results; the reference keeps a
    float cumulative moving average (md_script.c:5909-5955) that by itself sits 1.1e-5 / 2.9e-5 / 1.8e-5 (rdf / sdf / density) from that exact
    mean after 4096 frames (tests/test_oracle_golden.py::test_long_run_average_oracle_exact_mean_vs_reference_cma measures it with the oracle).
    Asserted: within 5e-5 of the reference everywhere (its own rounding noise), the deviation printed; non-zero pattern identical."""
    vb = _vb(); g = load_golden("water12_avg.npz"); n, seed, F = int(g["n"]), int(g["seed"]), int(g["num_frames"])
    base, L = vb.synth_water_base(n, seed); na = base.shape[1]
    d_base = vb.device_alloc(0, base.nbytes); vb.memcpy_h2d(0, d_base, base.ctypes.data, base.nbytes)
    d_fr = vb.device_alloc(0, F * 3 * na * 4)
    vb.synth_water_frames_device(0, n, seed, d_base, 0, F, d_fr, 3 * na, na)
    f0 = vb.synth_water_frames_host(n, seed, base, 0, 1)
    sysm = vb.water_system(n); cell = vb.UnitCell.from_basis(L, L, L)
    plan = vb.Plan(sysm, vb.compile_script(str(g["script"]), sysm), F)
    plan.set_initial_frame(*f0[0], cell)
    plan.eval_device_frames(d_fr, 3 * na, na, cell, 0, F)
    rel = lambda a, b: float(np.max(np.abs(a.astype(np.float64) - b.astype(np.float64)) / np.abs(b.astype(np.float64))))
    r = plan.property_data("r"); r_ref = g["r__full"]; nz = r_ref[:1024] > 0
    assert np.array_equal(r.values[:1024] > 0, nz) and np.array_equal(r.weights, r_ref[1024:])
    d_r = rel(r.values[:1024][nz], r_ref[:1024][nz])
    v = plan.property_data("v").values; vs = g["v__sample_idx"]
    assert int(np.count_nonzero(v)) == int(g["v__nnz"])
    d_v = rel(v[vs], g["v__sample_val"]); d_vs = abs(float(v.astype(np.float64).sum()) - float(g["v__sum"])) / float(g["v__sum"])
    dz = plan.property_data("dz"); dz_ref = g["dz__full"][:1024]; nzd = dz_ref > 0
    d_d = rel(dz.values[:1024][nzd], dz_ref[nzd])
    print(f"GPU exact mean vs reference CMA after {F} frames: rdf {d_r:.2e}, sdf {d_v:.2e} (sum {d_vs:.2e}), density_z {d_d:.2e}")
    assert d_r <= 5e-5 and d_v <= 5e-5 and d_vs <= 1e-5 and d_d <= 5e-5
    m = g["r__meta"]; assert r.min_value == m[0] and r.max_value == m[1]           # per-frame min / max of the bins folded over all frames
    assert plan.frame_mask().all()
    vb.device_free(0, d_base); vb.device_free(0, d_fr); plan.close()


def test_fast_sqrt_matches_ieee():
    """The branch-free sqrt used when binning RDF hits equals the correctly rounded sqrt for every float in [2^-100, 2^100]
    (d2 values that reach it lie in [1e-6, cutoff^2])."""
    from viamd_b200.api import debug_sqrt_sweep
    import struct
    bits = lambda x: struct.unpack("<I", struct.pack("<f", x))[0]
    assert debug_sqrt_sweep(bits(2.0 ** -100), bits(2.0 ** 100)) == 0


def test_golden_membrane_config4_shape():
    """BASELINE config 4 at reduced size against the reference's goldens: lipid-tail rdf (symmetric same-selection path, non-cubic cell),
    density profiles of a subset and of all atoms."""
    g = load_golden("membrane6.npz"); s = golden_system(g); vb = _vb()
    names = np.array(s["names"]); c2 = np.nonzero(np.char.startswith(names, "C2"))[0].astype(np.int32); allat = np.arange(len(names), dtype=np.int32)
    sysm = vb.System(len(names), s["mass"])
    props = [vb.rdf("rt", c2, c2, 12.0), vb.density("dz", 2, c2), vb.density("dall", 2, allat), vb.density("dxall", 0, allat)]
    F = g["frames"].shape[0]
    plan = vb.Plan(sysm, props, F, keep_frame_results=True)
    cells = [vb_cell(g["cells"][f], g["cell_flags"][f]) for f in range(F)]
    plan.set_initial_frame(*g["frames"][0], cells[0])
    plan.eval_host_frames(g["frames"], cells, 0)
    for f in range(F):
        bins, tot = plan.frame_counts("rt", f)
        assert np.array_equal(bins.astype(np.float32), g["rt__pf"][f, :1024]) and tot == int(g["rt__pf"][f, :1024].sum())
    assert np.array_equal(plan.property_data("rt").weights, g["rt__pf"][F - 1, 1024:])
    for key in ("dz", "dall", "dxall"):
        d = plan.property_data(key)
        np.testing.assert_allclose(d.values[:1024], g[f"{key}__full"][:1024], rtol=RTOL, atol=1e-3)
    plan.close()


def test_full_size_config4_membrane_1M_atoms():
    """BASELINE config 4 at full size (994 656 atoms): frames generated on the device, lipid-tail rdf + density_z over all atoms.
    Size-independent properties: bins sum to the pair total, accumulators independent of evaluation order, total mass conserved in
    every frame's density profile, frame 0 equal to the oracle."""
    vb = _vb()
    nl, nwxy, nwz, seed, F = 38, 100, 48, 4321, 6
    base, whole, mol, L3 = vb.synth_membrane_base(nl, nwxy, nwz, seed); na = base.shape[1]
    assert na == 994656
    sysm = vb.membrane_system(nl, nwxy, nwz)
    props = vb.compile_script("rt = rdf(name('C2*'), name('C2*'), 12.0); dz = density_z(all);", sysm)
    d_base = vb.device_alloc(0, base.nbytes); vb.memcpy_h2d(0, d_base, base.ctypes.data, base.nbytes)
    d_mol = vb.device_alloc(0, mol.nbytes); vb.memcpy_h2d(0, d_mol, mol.ctypes.data, mol.nbytes)
    d_fr = vb.device_alloc(0, F * 3 * na * 4)
    vb.synth_membrane_frames_device(0, nl, nwxy, nwz, seed, d_base, d_mol, 0, F, d_fr, 3 * na, na)
    f0 = vb.synth_membrane_frames_host(nl, nwxy, nwz, seed, base, mol, 0, 1)
    back = np.empty((3, na), np.float32); vb.memcpy_d2h(0, back.ctypes.data, d_fr, back.nbytes)
    assert np.array_equal(back, f0[0])                       # device generator == host generator
    cell = vb.UnitCell.from_basis(*L3)
    plan = vb.Plan(sysm, props, F, keep_frame_results=True, batch_frames=4)
    plan.set_initial_frame(*f0[0], cell)
    plan.eval_device_frames(d_fr, 3 * na, na, cell, 0, F)
    acc = plan.counts("rt"); dacc = plan.counts("dz")
    per = [plan.frame_counts("rt", f) for f in range(F)]
    assert all(int(b.sum()) == t > 0 for b, t in per)
    assert np.array_equal(acc, np.sum([b.astype(np.uint64) for b, _ in per], axis=0))
    # every atom lands in exactly one bin: fixed-point mass sum is exact
    assert int(dacc.sum()) == F * int(np.round(sysm.mass.astype(np.float64) * 2 ** 24).sum())
    c2 = props[0].idx[0]; oc = O.UnitCell.ortho(*L3)
    ob, ow, ot = O.rdf_frame(*f0[0], c2, c2, oc, 0.0, 12.0)
    assert per[0][1] == ot and np.array_equal(per[0][0].astype(np.float32), ob)
    db, _ = O.density_frame(*f0[0], sysm.mass, np.arange(na, dtype=np.int32), oc, 2)
    plan.clear()
    plan.eval_device_frames(d_fr + 3 * 3 * na * 4, 3 * na, na, cell, 3, 3)
    plan.eval_device_frames(d_fr, 3 * na, na, cell, 0, 3)
    assert np.array_equal(plan.counts("rt"), acc) and np.array_equal(plan.counts("dz"), dacc)
    plan.clear(); plan.eval_device_frames(d_fr, 3 * na, na, cell, 0, 1)
    np.testing.assert_allclose(plan.property_data("dz").values[:1024], db, rtol=3e-5, atol=1e-3)   # float sequential sum of ~1000 masses per bin in the reference
    for p in (d_base, d_mol, d_fr): vb.device_free(0, p)
    plan.close()


XTC_CASES = ("water6", "lowprec", "tric6", "water16", "small5", "wide12", "huge12")


@pytest.mark.parametrize("case", XTC_CASES)
def test_xtc_device_decode_bitexact(case):
    """XTC streams from the reference's writer expanded on the device vs the reference reader's decode (tests/golden/xtc_cases.npz):
    coordinates bit for bit, unit cell + flags, step, time. wide12 / huge12: the reference mis-decodes them, the written data is the truth."""
    import hashlib
    vb = _vb(); g = load_golden("xtc_cases.npz"); blob = g[case + "__xtc"]; na = int(g[case + "__na"])
    offs, na2 = vb.xtc_frame_offsets(blob); F = len(g[case + "__cells"])
    assert na2 == na and len(offs) == F + 1 and int(offs[-1]) == blob.size
    xyz, cells, steps, times = vb.xtc_decode_frames(blob, offs, na)
    assert list(steps) == list(range(F)) and list(times) == [float(f) for f in range(F)]
    for f in range(F):
        if case in ("wide12", "huge12"): assert np.abs(xyz[f] - g[case + "__orig"][f]).max() <= 0.02
        elif case + "__frames" in g: assert np.array_equal(xyz[f], g[case + "__frames"][f]), (case, f)
        else: assert hashlib.sha256(xyz[f].tobytes()).hexdigest() == str(g[case + "__sha"][f])
        c = cells[f]
        assert [c.x, c.xy, c.xz, c.y, c.yz, c.z] == list(g[case + "__cells"][f]) and c.flags == int(g[case + "__flags"][f])
    o_ok, o_xyz, _, _, _ = O.xtc_decode_frame(blob, offs[0], offs[1], na)
    assert o_ok and np.array_equal(o_xyz, xyz[0])               # oracle == device on every case


def test_xtc_input_gives_the_results_of_the_decoded_frames():
    """md_script evaluation fed with XTC bytes (decode on the device) == evaluation of the frames the reference reader decodes."""
    vb = _vb(); g = load_golden("xtc_cases.npz"); w = load_golden("water6.npz"); s = golden_system(w)
    blob = g["water6__xtc"]; offs, na = vb.xtc_frame_offsets(blob); F = len(offs) - 1
    sysm = vb_system(s)
    src = "r = rdf(element('O'), element('O'), 6.0); v = sdf(residue(1:20), element('O'), 5.0); dz = density_z(element('O')); d = distance(1,10);"
    props = vb.compile_script(src, sysm)
    frames = g["water6__frames"]; cells = [vb_cell(g["water6__cells"][f], g["water6__flags"][f]) for f in range(F)]
    res = []
    for mode in ("xtc", "host"):
        plan = vb.Plan(sysm, vb.compile_script(src, sysm), F, keep_frame_results=True, batch_frames=3)
        plan.set_initial_frame(*frames[0], cells[0])
        if mode == "xtc": plan.eval_xtc_frames(blob, offs, 0)
        else: plan.eval_host_frames(frames, cells, 0)
        res.append((plan.counts("r"), plan.counts("v"), plan.counts("dz"), plan.property_data("d").values.copy(), plan.frame_mask().copy()))
        plan.close()
    for a, b in zip(*res): assert np.array_equal(a, b)
    assert res[0][0].sum() > 0 and res[0][1].sum() > 0


def test_xtc_file_input(tmp_path):
    """mdgpu_eval_xtc_file: the bytes of an .xtc file on disk -> results; frame 0 becomes the initial configuration when none was set."""
    vb = _vb(); g = load_golden("xtc_cases.npz"); w = load_golden("water6.npz"); s = golden_system(w)
    path = str(tmp_path / "w6.xtc"); g["water6__xtc"].tofile(path)
    sysm = vb_system(s); F = len(g["water6__cells"])
    src = "r = rdf(element('O'), element('O'), 6.0); v = sdf(residue(1:20), element('O'), 5.0); d = distance(1,10);"
    frames = g["water6__frames"]; cells = [vb_cell(g["water6__cells"][f], g["water6__flags"][f]) for f in range(F)]
    a = vb.Plan(sysm, vb.compile_script(src, sysm), F, batch_frames=3); a.eval_xtc_file(path, 0, F)
    b = vb.Plan(sysm, vb.compile_script(src, sysm), F, batch_frames=3); b.set_initial_frame(*frames[0], cells[0]); b.eval_host_frames(frames, cells, 0)
    for key in ("r", "v"): assert np.array_equal(a.counts(key), b.counts(key)) and a.counts(key).sum() > 0
    assert np.array_equal(a.property_data("d").values, b.property_data("d").values) and a.frame_mask().all()
    with pytest.raises(vb.MdgpuError): a.eval_xtc_file(str(tmp_path / "missing.xtc"), 0, 1)
    a.close(); b.close()


@pytest.mark.parametrize("variant", [1, 2, 4])
def test_rdf_kernel_variants_are_bit_identical(variant):
    """mdgpu_plan_options_t.rdf_variant: 1 = scalar kernel without candidate lists, 2 = 3 CTAs / SM (default: 4), 4 = reference chunks staged by the TMA unit
    (cp.async.bulk + mbarrier). Every variant must produce the default kernel's per-frame bins: reference goldens (ortho + triclinic) and a
    24 576-atom box against the default variant."""
    vb = _vb()
    for gname, keys, src in (("water6.npz", ("r", "rh"), "r = rdf(element('O'), element('O'), 6.0); rh = rdf(element('O'), element('H'), 1.5:6.0);"),
                             ("tric6.npz", ("rt", "rth"), "rt = rdf(element('O'), element('O'), 6.0); rth = rdf(element('O'), element('H'), 2.0:7.0);")):
        g = load_golden(gname); s = golden_system(g)
        plan, cells = _water_plan(g, s, src, rdf_variant=variant)
        plan.eval_host_frames(g["frames"], cells, 0)
        for key in keys:
            for f in range(g["frames"].shape[0]):
                bins, tot = plan.frame_counts(key, f)
                assert np.array_equal(bins.astype(np.float32), g[f"{key}__pf"][f, :1024]) and tot == int(bins.sum()), (gname, key, f)
        plan.close()
    n, seed, F = 20, 99, 6
    base, L = vb.synth_water_base(n, seed); frames = vb.synth_water_frames_host(n, seed, base, 0, F)
    sysm = vb.water_system(n); o = np.arange(0, 3 * n ** 3, 3, dtype=np.int32); cell = vb.UnitCell.from_basis(L, L, L)
    out = []
    for v in (0, variant):
        plan = vb.Plan(sysm, [vb.rdf("r", o, o, 10.0)], F, keep_frame_results=True, rdf_variant=v)
        plan.eval_host_frames(frames, cell, 0)
        out.append([plan.frame_counts("r", f) for f in range(F)]); plan.close()
    for (b0, t0), (b1, t1) in zip(*out): assert t0 == t1 > 0 and np.array_equal(b0, b1)


def test_rdf_triclinic_unwrapped_coordinates_overflow_pass():
    """ADVICE r1 (high): a triclinic trajectory whose atoms are not wrapped into the unit cell (20 % shifted by a lattice vector) populates home
    cells outside the cell grid — the reference serves them through its single wrap — so the candidate lists outgrow `neighbours x |targets|`.
    The home cells that do not fit are evaluated by the overflow pass (k_rdf_pairs<.., OVF>) instead of failing with MDGPU_ERR_CAPACITY:
    per-frame bins equal the oracle's and the list-free scalar kernel's, for different and for identical selections."""
    vb = _vb(); rng = np.random.default_rng(5)
    n, seed, F = 8, 321, 3
    base, L = vb.synth_water_base(n, seed); fr = vb.synth_water_frames_host(n, seed, base, 0, F).astype(np.float64); na = 3 * n ** 3
    xy, xz, yz = 0.21 * L, -0.13 * L, 0.17 * L
    X, Y, Z = fr[:, 0].copy(), fr[:, 1].copy(), fr[:, 2].copy()
    fr[:, 0] = X + (xy / L) * Y + (xz / L) * Z; fr[:, 1] = Y + (yz / L) * Z
    mol = rng.random(n ** 3) < 0.2; sh = np.repeat(mol, 3)                      # whole molecules moved by +a / -b: still the same periodic system
    fr[:, 0, sh] += L; half = sh & (np.arange(na) % 2 == 0); fr[:, 0, half] -= xy; fr[:, 1, half] -= L
    fr = fr.astype(np.float32)
    cell = vb.UnitCell.from_basis(L, L, L, xy, xz, yz); ocell = O.UnitCell.from_params(L, xy, xz, L, yz, L, O.TRICLINIC | O.PBC_ALL)
    sysm = vb.water_system(n); o = np.arange(0, na, 3, dtype=np.int32); h = np.setdiff1d(np.arange(na, dtype=np.int32), o)
    for ref, trg, cut in ((o, h, 7.0), (o, o, 7.5)):
        res = []
        for variant in (0, 1):
            plan = vb.Plan(sysm, [vb.rdf("r", ref, trg, cut)], F, keep_frame_results=True, rdf_variant=variant)
            plan.eval_host_frames(fr, cell, 0)
            res.append([plan.frame_counts("r", f) for f in range(F)]); plan.close()
        for f in range(F):
            ob, ow, ot = O.rdf_frame(*fr[f], ref, trg, ocell, 0.0, cut)
            for bins, tot in (res[0][f], res[1][f]):
                assert tot == ot > 0 and np.array_equal(bins.astype(np.float32), ob), (len(trg), f)


def test_two_device_plans_of_one_process_on_one_gpu_through_a_loopback_exchange(monkeypatch):
    """SURVEY 8(e) inside the library (mdgpu_plan_options_t.num_devices = 2) on the hardware a one-GPU box offers: both "devices" are GPU 0
    (MDGPU_ALLOW_DUPLICATE_DEVICES) and the exchange step's NCCL entry points are the loopback of tests/emul/fake_nccl.cpp (device buffers
    staged through the host) — real NCCL refuses two ranks on one device. What runs on the device is everything else: the peer plan and its
    stream slots, one host thread per device block, the reduce onto devices[0] with peers zeroed, frame masks merged, the fold. Results equal
    the single-device plan's; a second sync changes nothing; evaluating the halves separately merges once."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emul"))
    import build_emul
    from test_emulated_library import SCRIPT_MIX, _mix_results
    import viamd_b200.api as api
    emulated = "emul" in os.path.basename(api.LIB_PATH)   # (this file's tests also run on the CPU emulation of the library: host-memory exchange there)
    monkeypatch.setenv("MDGPU_ALLOW_DUPLICATE_DEVICES", "1"); monkeypatch.setenv("MDGPU_NCCL_LIB", build_emul.build_fake_nccl() if emulated else build_emul.build_loopback_nccl())
    vb = _vb(); g = load_golden("water6.npz"); sysm = vb_system(golden_system(g)); F = g["frames"].shape[0]
    cells = [vb_cell(g["cells"][f], g["cell_flags"][f]) for f in range(F)]
    def same(a, b):
        assert a.keys() == b.keys()
        for k in a: assert np.array_equal(a[k], b[k]), k
    one = vb.Plan(sysm, vb.compile_script(SCRIPT_MIX, sysm), F, keep_frame_results=True); one.set_initial_frame(*g["frames"][0], cells[0])
    one.eval_host_frames(g["frames"], cells, 0); want = _mix_results(one); one.close()
    for src in ("host", "traj"):
        plan = vb.Plan(sysm, vb.compile_script(SCRIPT_MIX, sysm), F, keep_frame_results=True, devices=[0, 0])
        plan.set_initial_frame(*g["frames"][0], cells[0])
        if src == "host": plan.eval_host_frames(g["frames"], cells, 0)
        else: assert plan.eval_frame_range(vb.ArrayTrajectory(g["frames"], cells), 0, F, loader_threads=2)
        same(want, _mix_results(plan)); plan.sync(); same(want, _mix_results(plan))
        assert plan.exchange_stats()[1] == 1
        bins, tot = plan.frame_counts("r", F - 1); assert tot == int(bins.sum()) > 0       # a frame the second plan evaluated
        plan.clear()
        plan.eval_host_frames(g["frames"][:2], cells[:2], 0); plan.sync(); plan.eval_host_frames(g["frames"][2:], cells[2:], 2)
        same(want, _mix_results(plan))
        plan.close()
