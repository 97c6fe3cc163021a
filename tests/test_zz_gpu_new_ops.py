"""GPU tests of the device paths written after this round's GPU budget was spent: rmsd, distance_pair + the multi-valued temporal container,
com, plane, count(within()). They first ran on a B200 in the round's last GPU call (profiles/r03a_newops_gpu_tests.log, 16 passed); they were written against the CPU execution of the same
sources: every test here passes through the C ABI against tests/emul's emulated build of the whole library (tests/test_emulated_library.py;
the complete, GPU-validated tests/test_gpu_parity.py passes under that emulation too), also with AddressSanitizer watching the "device"
buffers. The file sorts last on purpose: with `pytest -x` every test that has already passed on the GPU runs before these.
"""
import os

import numpy as np
import pytest

import oracle_lib as O
from helpers import load_golden, cell_from_row, dense_from_sparse, golden_system, sel_element, vb_system, vb_cell

pytestmark = pytest.mark.gpu


def _same(a, b):
    """Floats that go through a fit (svd3) or a double sin / cos / atan2: bit-equal when the library's sources run on the CPU (tests/emul: the
    reference's own libm), within the north-star float tolerance on the device (CUDA's double libm may differ in the last bit)."""
    import viamd_b200.api as api
    a = np.asarray(a, np.float32); b = np.asarray(b, np.float32)
    if "emul" in os.path.basename(api.LIB_PATH): return bool(np.array_equal(a, b))
    return bool(np.allclose(a, b, rtol=1e-5, atol=1e-6))


def _vb():
    import viamd_b200 as vb
    return vb


def _plan(g, s, src, **kw):
    import viamd_b200 as vb
    sysm = vb_system(s); props = vb.compile_script(src, sysm); F = g["frames"].shape[0]
    plan = vb.Plan(sysm, props, F, **kw)
    cells = [vb_cell(g["cells"][f], g["cell_flags"][f]) for f in range(F)]
    plan.set_initial_frame(*g["frames"][0], cells[0])
    return plan, cells


def test_rmsd_goldens_bitexact():
    """rmsd(selection) (k_rmsd, sdf.cu) against the reference's values: water (ortho), 1ALA (ortho, 153 atoms, through the frame-source
    interface) and the triclinic cell that changes every frame. Every operation is IEEE on both sides (sqrt, division, no libm)."""
    g = load_golden("water6.npz"); s = golden_system(g)
    plan, cells = _plan(g, s, "rm = rmsd(residue(1:10)); d = distance(1,10);")
    plan.eval_host_frames(g["frames"], cells, 0)
    d = plan.property_data("rm")
    assert _same(d.values, g["rm__full"]), (d.values, g["rm__full"])
    mn, mx, r0, r1 = g["rm__meta"]
    assert _same([d.min_value, d.max_value, d.min_range[0], d.max_range[0]], [mn, mx, r0, r1])
    assert np.array_equal(plan.property_data("d").values, g["d__full"])
    plan.close()

    import viamd_b200 as vb
    g = load_golden("ala50.npz"); s = golden_system(g)
    plan, cells = _plan(g, s, "rma = rmsd(residue(1:15));", batch_frames=16)
    assert plan.eval_frame_range(vb.ArrayTrajectory(g["frames"], cells), 0, g["frames"].shape[0])
    assert _same(plan.property_data("rma").values, g["rma__full"])
    plan.close()

    g = load_golden("tric6.npz"); s = golden_system(g); r = load_golden("tric6_rmsd.npz")
    plan, cells = _plan(g, s, str(r["script"]))
    plan.eval_host_frames(g["frames"], cells, 0)
    for key in ("rmt", "rma", "rmo"):
        assert _same(plan.property_data(key).values, r[f"{key}__full"]), key
    plan.close()


def test_rmsd_oracle_larger_and_batched():
    """A 3 000-atom selection over 40 frames in batches of 7 (ragged last batch), two stream slots: oracle vs device, value by value."""
    import viamd_b200 as vb
    n = 10; sysm = vb.water_system(n); base, L = vb.synth_water_base(n, 5)
    F = 40; frames = vb.synth_water_frames_host(n, 5, base, 0, F)
    cell = vb.UnitCell.from_basis(L, L, L); ocell = cell_from_row([L, 0, 0, L, 0, L], 29)
    idx = np.arange(0, 3000, dtype=np.int32)
    plan = vb.Plan(sysm, [vb.rmsd("rm", idx)], F, batch_frames=7, num_streams=2)
    plan.set_initial_frame(*frames[0], cell)
    plan.eval_host_frames(frames, [cell] * F, 0)
    got = plan.property_data("rm").values
    mass = np.asarray(sysm.mass, np.float32)
    for f in range(F):
        want = O.rmsd_frame(*frames[f], frames[0], mass, idx, np.asarray(sysm.conn_offset, np.uint32), np.asarray(sysm.conn_idx, np.int32), ocell)
        assert _same(got[f], want), (f, got[f], want)
    plan.close()


def test_rmsd_empty_selection_and_missing_initial_frame():
    import viamd_b200 as vb
    sysm = vb.water_system(4); base, L = vb.synth_water_base(4, 1); frames = vb.synth_water_frames_host(4, 1, base, 0, 3)
    cell = vb.UnitCell.from_basis(L, L, L)
    plan = vb.Plan(sysm, [vb.rmsd("e", np.zeros(0, np.int32))], 3)
    plan.set_initial_frame(*frames[0], cell); plan.eval_host_frames(frames, [cell] * 3, 0)
    assert np.array_equal(plan.property_data("e").values, np.zeros(3, np.float32))   # _rmsd :4311: nothing written for an empty selection
    plan.close()
    plan = vb.Plan(sysm, [vb.rmsd("r", np.arange(9, dtype=np.int32))], 3)
    with pytest.raises(vb.MdgpuError):
        plan.eval_host_frames(frames, [cell] * 3, 0)
    plan.close()


def test_distance_pair_goldens_and_aggregates():
    """distance_pair(a, b) (k_distance_pair, props.cu) -> [F, |a|*|b|] with the per-frame aggregates of a multi-valued temporal, against the
    reference (pairs6.npz), orthorhombic and triclinic; through the script lowering."""
    p = load_golden("pairs6.npz")
    for tag, name in (("w", "water6.npz"), ("t", "tric6.npz")):
        g = load_golden(name); s = golden_system(g); F = g["frames"].shape[0]
        plan, cells = _plan(g, s, str(p["script"]), batch_frames=3)
        plan.eval_host_frames(g["frames"], cells, 0)
        for key in ("dp", "dpo"):
            k = f"{tag}_{key}"; d = plan.property_data(key)
            assert tuple(d.dim[:2]) == tuple(p[k + "__dim"][:2])
            assert np.array_equal(d.values, p[k + "__full"]), k
            mn, mx, r0, r1 = p[k + "__meta"]
            assert d.min_value == mn and d.max_value == mx and d.min_range[0] == r0 and d.max_range[0] == r1
            agg = plan.aggregate(key)
            assert np.array_equal(agg["mean"], p[k + "__mean"]) and np.array_equal(agg["var"], p[k + "__var"]) and np.array_equal(agg["ext"], p[k + "__ext"]), k
        plan.close()


def test_distance_pair_between_arrays_of_selections():
    """distance_pair whose arguments are arrays of selections (k_group_com -> k_distance_pair on positions): the residue contact map,
    groups x groups and groups x atoms, against the reference (pairs6.npz), ortho + triclinic."""
    p = load_golden("pairs6.npz")
    for tag, name in (("w", "water6.npz"), ("t", "tric6.npz")):
        g = load_golden(name); s = golden_system(g)
        plan, cells = _plan(g, s, "dpg = distance_pair(residue(1:4), residue(10:15)); dpm = distance_pair(residue(2:5), atom(100:103));", batch_frames=3)
        plan.eval_host_frames(g["frames"], cells, 0)
        for key in ("dpg", "dpm"):
            k = f"{tag}_{key}"; d = plan.property_data(key)
            assert tuple(d.dim[:2]) == tuple(p[k + "__dim"][:2]) and np.array_equal(d.values, p[k + "__full"]), k
            agg = plan.aggregate(key)
            assert np.array_equal(agg["mean"], p[k + "__mean"]) and np.array_equal(agg["var"], p[k + "__var"])
        plan.close()


def test_distance_pair_limits():
    import viamd_b200 as vb
    sysm = vb.water_system(8)
    with pytest.raises(vb.MdgpuError):   # 1 536 x 1 536 pairs > 1 000 000 values per frame (md_script_functions.inl:4056)
        vb.Plan(sysm, [vb.distance_pair("big", np.arange(1536), np.arange(1536))], 2)
    with pytest.raises(vb.MdgpuError):
        vb.Plan(sysm, [vb.distance_pair("e", np.zeros(0, np.int32), np.arange(3))], 2)
    plan = vb.Plan(sysm, [vb.distance("d", 0, 1)], 2)
    with pytest.raises(vb.MdgpuError):   # one value per frame: no aggregate
        plan.aggregate("d")
    plan.close()


def test_com_and_plane_goldens():
    """com(x) -> [F, 3] (k_arg_com + k_com_rows) and plane(selection) -> [F, 4] (k_plane), with aggregates, against pairs6.npz."""
    p = load_golden("pairs6.npz")
    for tag, name in (("w", "water6.npz"), ("t", "tric6.npz")):
        g = load_golden(name); s = golden_system(g)
        plan, cells = _plan(g, s, "c = com(residue(1)); ca = com(atom(1:30)); ci = com(5); pl = plane(atom(1:30)); plo = plane(element('O'));", batch_frames=3)
        plan.eval_host_frames(g["frames"], cells, 0)
        for key in ("c", "ca", "ci", "pl", "plo"):
            k = f"{tag}_{key}"; d = plan.property_data(key)
            assert tuple(d.dim[:2]) == tuple(p[k + "__dim"][:2])
            assert _same(d.values, p[k + "__full"]), (k, d.values[:8], p[k + "__full"][:8])
            mn, mx, r0, r1 = p[k + "__meta"]
            assert _same([d.min_value, d.max_value, d.min_range[0], d.max_range[0]], [mn, mx, r0, r1])
            agg = plan.aggregate(key)
            assert _same(agg["mean"], p[k + "__mean"]) and _same(agg["var"], p[k + "__var"]) and _same(agg["ext"], p[k + "__ext"]), k
        plan.close()
    import viamd_b200 as vb
    with pytest.raises(vb.MdgpuError):   # "need at least 3 to compute a plane" (:4815)
        vb.Plan(vb.water_system(4), [vb.plane("p", np.arange(2))], 2)


def test_count_within_goldens_and_oracle():
    """count(within(radius, selection)) (cells.cu cell lists over all atoms + k_within_mark / k_within_count): the reference's counts on the
    water goldens, the oracle in the triclinic cell and with a non-periodic axis; together with an rdf in the same plan (shared slots)."""
    g = load_golden("water6.npz"); s = golden_system(g)
    plan, cells = _plan(g, s, "cw = count(within(4.0, residue(1))); cw2 = count(within(7.5, atom(10:12))); r = rdf(element('O'), element('O'), 6.0);", batch_frames=3)
    plan.eval_host_frames(g["frames"], cells, 0)
    assert np.array_equal(plan.property_data("cw").values, g["cw__full"]) and np.array_equal(plan.property_data("cw2").values, g["cw2__full"])
    assert np.array_equal(plan.property_data("r").values[:1024], g["r__full"][:1024]) or np.allclose(plan.property_data("r").values[:1024], g["r__full"][:1024], rtol=1e-5, atol=1e-6)
    plan.close()
    import viamd_b200 as vb
    for name, flags, sel, radius in (("tric6.npz", None, np.arange(0, 30), 5.0), ("water6.npz", 1 | 4 | 8, np.arange(0, 12), 6.5)):
        g = load_golden(name); s = golden_system(g); F = g["frames"].shape[0]
        fl = g["cell_flags"] if flags is None else np.full(F, flags, np.uint32)
        plan = vb.Plan(vb_system(s), [vb.count_within("c", radius, sel)], F)
        cells = [vb_cell(g["cells"][f], fl[f]) for f in range(F)]
        plan.eval_host_frames(g["frames"], cells, 0)
        got = plan.property_data("c").values
        for f in range(F):
            assert got[f] == len(O.within(*g["frames"][f], np.asarray(sel, np.int32), radius, cell_from_row(g["cells"][f], fl[f]))), (name, f)
        plan.close()
    with pytest.raises(vb.MdgpuError):
        vb.Plan(vb.water_system(4), [vb.count_within("c", 0.0, np.arange(3))], 2)


def test_rdf_candidate_lists_follow_a_cell_whose_neighbour_reach_grows():
    """Regression (found by tests/golden/fuzz_gpu.py --emulated): a sheared cell can take the pair query from 27 to 45+ neighbour offsets in a
    later frame; the candidate lists were sized from the first frame's cell and the evaluation failed with MDGPU_ERR_CAPACITY. They now grow
    with the batch's cells. Frame 0: shear 0.05 L (reach 1,1,1); frames 1-3: shear 0.25 L (reach 2,1,1). Bins against the oracle."""
    import viamd_b200 as vb
    n = 6; sysm = vb.water_system(n); base, L = vb.synth_water_base(n, 9725); F = 4
    fr = vb.synth_water_frames_host(n, 9725, base, 0, F).astype(np.float64); o = np.arange(0, 3 * n ** 3, 3, dtype=np.int32)
    cells, ocells = [], []
    for f in range(F):
        sh = (0.05 if f == 0 else 0.25) * L; xy, xz, yz = sh, -sh, sh
        X, Y, Z = fr[f].copy(); fr[f, 0] = X + (xy / L) * Y + (xz / L) * Z; fr[f, 1] = Y + (yz / L) * Z
        cells.append(vb.UnitCell(L, xy, xz, L, yz, L, vb.CELL_TRICLINIC | vb.CELL_PBC_ALL)); ocells.append(O.UnitCell.from_params(L, xy, xz, L, yz, L, vb.CELL_TRICLINIC | vb.CELL_PBC_ALL))
    fr = fr.astype(np.float32)
    for bf in (1, 4):   # growth between batches and inside one batch
        plan = vb.Plan(sysm, [vb.rdf("r", o, o, 3.59)], F, keep_frame_results=True, batch_frames=bf)
        plan.eval_host_frames(fr, cells, 0)
        for f in range(F):
            want, _, tot_w = O.rdf_frame(*fr[f], o, o, ocells[f], 0.0, 3.59); bins, tot = plan.frame_counts("r", f)
            assert np.array_equal(bins.astype(np.float32), want) and tot == tot_w, (bf, f)
        plan.close()


def test_expressions_in_contexts():
    """`expr in contexts` for distance / angle / dihedral with integer arguments (k_temporal_ctx): [F, n_contexts] rows and aggregates against
    the reference (pairs6.npz), ortho + triclinic; distances equal, angles / dihedrals within the libm tolerance."""
    p = load_golden("pairs6.npz")
    for tag, name in (("w", "water6.npz"), ("t", "tric6.npz")):
        g = load_golden(name); s = golden_system(g)
        plan, cells = _plan(g, s, "anc = angle(2,1,3) in residue(1:10); ddc = distance(1,3) in residue(:); dhc = dihedral(1,2,3,1) in residue(3:4);", batch_frames=3)
        plan.eval_host_frames(g["frames"], cells, 0)
        d = plan.property_data("ddc")
        assert tuple(d.dim[:2]) == tuple(p[f"{tag}_ddc__dim"][:2]) and np.array_equal(d.values, p[f"{tag}_ddc__full"])
        agg = plan.aggregate("ddc")
        assert np.array_equal(agg["mean"], p[f"{tag}_ddc__mean"]) and np.array_equal(agg["var"], p[f"{tag}_ddc__var"]) and np.array_equal(agg["ext"], p[f"{tag}_ddc__ext"])
        mn, mx, r0, r1 = p[f"{tag}_ddc__meta"]
        assert d.min_value == mn and d.max_value == mx and d.min_range[0] == r0 and d.max_range[0] == r1
        np.testing.assert_allclose(plan.property_data("anc").values, p[f"{tag}_anc__full"], rtol=1e-5)
        np.testing.assert_allclose(plan.property_data("dhc").values, p[f"{tag}_dhc__full"], rtol=1e-5, atol=1e-6)
        plan.close()


def test_shape_weights_of_structures():
    """Shape weights per structure and frame (k_shape_weights) against the reference's functions (shapes.npz): 1ALA residues mass-weighted
    through the frame-source interface, water with unit weights, the triclinic cell. The double atan2 of the periodic centre is libm on the
    reference side and CUDA's on the device: 1e-5 relative (equal under the CPU emulation)."""
    import viamd_b200 as vb
    W = load_golden("shapes.npz")
    for tag, name in (("a", "ala50.npz"), ("w", "water6.npz"), ("t", "tric6.npz")):
        g = load_golden(name); s = golden_system(g); co = s["comp_off"]; w = W[tag + "__weights"]; F, n = w.shape[:2]
        groups = [np.arange(co[r], co[r + 1], dtype=np.int32) for r in range(n)]
        plan = vb.Plan(vb_system(s), [vb.shape_weights("sw", groups, use_mass=bool(int(W[tag + "__mass"])))], F, batch_frames=7)
        cells = [vb_cell(g["cells"][f], g["cell_flags"][f]) for f in range(F)]
        assert plan.eval_frame_range(vb.ArrayTrajectory(g["frames"], cells), 0, F)
        d = plan.property_data("sw")
        assert tuple(d.dim[:2]) == (F, 3 * n)
        # weights live in [0, 1]; the third one of a planar structure is rounding noise (~1e-6) that a last-bit difference in the centre moves freely
        np.testing.assert_allclose(d.values.reshape(F, n, 3), w, rtol=1e-5, atol=1e-5)
        plan.close()
    with pytest.raises(vb.MdgpuError):
        vb.Plan(vb.water_system(4), [vb.Property("x", vb.OP_SHAPE_WEIGHTS, [np.zeros(0, np.int32)])], 2)


def test_coord_rows():
    """coord_x / coord_y / coord_z (k_coord_rows): the atoms' coordinates as [F, n] temporals with aggregates, against the reference (pairs6.npz)."""
    p = load_golden("pairs6.npz")
    for tag, name in (("w", "water6.npz"), ("t", "tric6.npz")):
        g = load_golden(name); s = golden_system(g)
        plan, cells = _plan(g, s, "cx = coord_x(residue(1)); cz = coord_z(atom(5:40)); cyi = coord_y(7);", batch_frames=3)
        plan.eval_host_frames(g["frames"], cells, 0)
        for key in ("cx", "cz", "cyi"):
            k = f"{tag}_{key}"; d = plan.property_data(key)
            assert tuple(d.dim[:2]) == tuple(p[k + "__dim"][:2]) and np.array_equal(d.values, p[k + "__full"]), k
            mn, mx, r0, r1 = p[k + "__meta"]
            assert d.min_value == mn and d.max_value == mx and d.min_range[0] == r0 and d.max_range[0] == r1
        agg = plan.aggregate("cz")
        assert np.array_equal(agg["mean"], p[f"{tag}_cz__mean"]) and np.array_equal(agg["var"], p[f"{tag}_cz__var"]) and np.array_equal(agg["ext"], p[f"{tag}_cz__ext"])
        plan.close()


def test_within_min_max_form():
    """within(min:max, selection) (_within_expl_frng :2609): as the argument of count() against the reference (pairs6.npz, ortho + triclinic) and
    as the reference set of an rdf against the oracle."""
    import viamd_b200 as vb
    p = load_golden("pairs6.npz")
    for tag, name in (("w", "water6.npz"), ("t", "tric6.npz")):
        g = load_golden(name); s = golden_system(g); F = g["frames"].shape[0]; o = sel_element(s, 8)
        plan, cells = _plan(g, s, "cwr = count(within(2.5:5.0, residue(1))); cwr2 = count(within(3.0:8.0, atom(10:40))); rwr = rdf(within(3.0:6.0, residue(2)), element('O'), 1.0:6.5);", keep_frame_results=True)
        plan.eval_host_frames(g["frames"], cells, 0)
        assert np.array_equal(plan.property_data("cwr").values, p[f"{tag}_cwr__full"]) and np.array_equal(plan.property_data("cwr2").values, p[f"{tag}_cwr2__full"])
        for f in range(F):
            x, y, z = g["frames"][f]; cell = cell_from_row(g["cells"][f], g["cell_flags"][f])
            ref = O.within(x, y, z, np.arange(3, 6, dtype=np.int32), 6.0, cell, rmin=3.0)
            want, _, tot_w = O.rdf_frame(x, y, z, ref, o, cell, 1.0, 6.5)
            bins, tot = plan.frame_counts("rwr", f)
            assert np.array_equal(bins.astype(np.float32), want) and tot == tot_w, (tag, f)
        plan.close()
    with pytest.raises(vb.MdgpuError):
        vb.Plan(vb.water_system(4), [vb.count_within("c", 3.0, np.arange(3), radius_min=4.0)], 2)


def test_static_selection_and_within():
    """`selection and within(...)` (_and :1975) — e.g. the oxygens in the first shell of a residue: the static side masks the per-frame set.
    Counts against the reference (pairs6.npz, either operand order, min:max form), the masked set as an rdf reference against the oracle."""
    p = load_golden("pairs6.npz")
    for tag, name in (("w", "water6.npz"), ("t", "tric6.npz")):
        g = load_golden(name); s = golden_system(g); F = g["frames"].shape[0]; o = sel_element(s, 8); h = sel_element(s, 1)
        plan, cells = _plan(g, s, "cwo = count(element('O') and within(4.0, residue(1))); cwh = count(within(2.5:5.0, residue(1)) and element('H')); "
                                  "rwo = rdf(element('H') and within(5.0, residue(2)), element('O'), 6.0);", keep_frame_results=True)
        plan.eval_host_frames(g["frames"], cells, 0)
        assert np.array_equal(plan.property_data("cwo").values, p[f"{tag}_cwo__full"]) and np.array_equal(plan.property_data("cwh").values, p[f"{tag}_cwh__full"])
        for f in range(F):
            x, y, z = g["frames"][f]; cell = cell_from_row(g["cells"][f], g["cell_flags"][f])
            ref = np.intersect1d(O.within(x, y, z, np.arange(3, 6, dtype=np.int32), 5.0, cell), h).astype(np.int32)
            want, _, tot_w = O.rdf_frame(x, y, z, ref, o, cell, 0.0, 6.0)
            bins, tot = plan.frame_counts("rwo", f)
            assert np.array_equal(bins.astype(np.float32), want) and tot == tot_w, (tag, f)
        plan.close()


def test_rdf_with_a_dynamic_within_reference_set():
    """rdf(within(radius, selection), targets, cutoff): the reference atoms change every frame (marks -> per-frame index list -> home-grid cell
    list -> the usual cull + pair kernels). Per-frame bins, weights and the mean against the reference (golden rw); a second property in
    the same plan shares the target cell list; triclinic + a larger radius against the oracle."""
    g = load_golden("water6.npz"); s = golden_system(g); F = g["frames"].shape[0]
    plan, cells = _plan(g, s, "rw = rdf(within(4.0, residue(1)), element('O'), 6.0); r = rdf(element('O'), element('O'), 6.0);", keep_frame_results=True, batch_frames=3)
    plan.eval_host_frames(g["frames"], cells, 0)
    for f in range(F):
        for key in ("rw", "r"):
            bins, tot = plan.frame_counts(key, f)
            assert np.array_equal(bins.astype(np.float32), g[f"{key}__pf"][f, :1024]) and tot == int(g[f"{key}__pf"][f, :1024].sum()), (key, f)
    d = plan.property_data("rw")
    assert np.array_equal(d.weights, g["rw__pf"][F - 1, 1024:])
    np.testing.assert_allclose(d.values[:1024], g["rw__full"][:1024], rtol=1e-5, atol=1e-6)
    plan.close()
    import viamd_b200 as vb
    g = load_golden("tric6.npz"); s = golden_system(g); F = g["frames"].shape[0]; o = sel_element(s, 8); sel = np.arange(30, 39, dtype=np.int32)
    plan = vb.Plan(vb_system(s), [vb.rdf_within("rw", 6.5, sel, o, 7.0, 1.0)], F, keep_frame_results=True)
    cells = [vb_cell(g["cells"][f], g["cell_flags"][f]) for f in range(F)]
    plan.eval_host_frames(g["frames"], cells, 0)
    for f in range(F):
        x, y, z = g["frames"][f]; cell = cell_from_row(g["cells"][f], g["cell_flags"][f])
        ref = O.within(x, y, z, sel, 6.5, cell)
        want, _, tot_w = O.rdf_frame(x, y, z, ref, o, cell, 1.0, 7.0)
        bins, tot = plan.frame_counts("rw", f)
        assert np.array_equal(bins.astype(np.float32), want) and tot == tot_w, f
    plan.close()


def test_new_ops_through_the_md_script_shim(tmp_path):
    """md_script_eval_frame_range (reference CPU path) vs md_script_gpu_eval_frame_range on a script made of the new ops, through the
    reference's own md_script.c + integration/md_script_mdgpu.inl (oracle/_ref/shim_harness)."""
    import json, os, subprocess
    import test_integration_shim as T
    T._need()
    gro = str(tmp_path / "w6.gro")
    subprocess.check_call([T.TOOL, "water-gro", "6", "1008", gro])
    p = subprocess.run([T.SHIM, "eval", "--sys", gro, "--traj", "synthwater:6:1008:9", "--script", "r = rdf(element('O'), element('O'), 6.0); " + T.SCRIPT_NEW], capture_output=True, text=True)
    line = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert line, p.stdout + p.stderr
    res = json.loads(line[-1])
    assert p.returncode == 0 and res["parity"] is True, res
    assert all(q["out_of_tol"] == 0 and q["frame_mask_equal"] for q in res["properties"])



def test_backbone_angles_of_every_segment_per_frame():
    """VIAMD's "Backbone Operations" pass (src/viamd.cpp:488-520 -> md_util_backbone_angles_compute md_util.c:2572-2620) as ONE op: (phi, psi) of
    all backbone segments of 1ALA for 50 frames against the reference's own values (tests/golden/backbone.npz); chain ends stay 0 as in the
    reference. atan2f on the device vs glibc: 1e-5."""
    vb = _vb(); g = load_golden("backbone.npz"); a = load_golden("ala50.npz"); s = golden_system(a)
    F, ns = g["angles"].shape[:2]
    plan = vb.Plan(vb_system(s), [vb.backbone_angles("bb", g["five"])], F)
    cells = [vb_cell(a["cells"][f], a["cell_flags"][f]) for f in range(F)]
    plan.eval_host_frames(a["frames"], cells, 0)
    d = plan.property_data("bb"); assert d.dim[:2] == (F, 2 * ns)
    got = d.values.reshape(F, ns, 2)
    np.testing.assert_allclose(got, g["angles"], rtol=1e-5, atol=2e-6)
    assert np.all(got[:, 0] == 0) and np.all(got[:, -1] == 0) and np.all(np.abs(got[:, 1:-1]) > 0)
    agg = plan.aggregate("bb"); assert agg["mean"].shape == (F,)
    plan.close()


def test_temporal_histogram_on_the_device():
    """compute_histogram_masked (src/main.cpp:172-226), VIAMD's per-property display histogram, with the [F, dim] values left on the device:
    per-column and aggregated forms, out-of-range values skipped, only evaluated frames counted, scale 1 / (bin width x samples)."""
    vb = _vb(); g = load_golden("water6.npz"); pz = load_golden("pairs6.npz"); s = golden_system(g); F = g["frames"].shape[0]
    plan = vb.Plan(vb_system(s), vb.compile_script("dp = distance_pair(atom(1:5), atom(20:30)); d = distance(1,10);", vb_system(s)), F)
    cells = [vb_cell(g["cells"][f], g["cell_flags"][f]) for f in range(F)]
    plan.eval_host_frames(g["frames"][:3], cells[:3], 0)                         # frame 3 stays unevaluated: it must not be counted
    vals = pz["w_dp__full"].reshape(F, 55)[:3]

    def ref_hist(v, nb, lo, hi, aggregate):                                       # the reference's loop, float for float
        dim = v.shape[1]; rows = 1 if aggregate else dim
        bins = np.zeros((rows, nb), np.float32); cnt = np.zeros(rows, np.int64)
        ext = np.float32(hi) - np.float32(lo); inv = np.float32(1.0) / ext if ext > 0 else np.float32(0)
        for f in range(v.shape[0]):
            for i in range(dim):
                x = np.float32(v[f, i])
                if x < np.float32(lo) or np.float32(hi) < x: continue
                b = min(max(int(np.float32(np.float32(x - np.float32(lo)) * inv) * np.float32(nb)), 0), nb - 1)
                bins[0 if aggregate else i, b] += 1; cnt[0 if aggregate else i] += 1
        width = ext / np.float32(nb)
        for i in range(rows): bins[i] *= np.float32(1.0) / (width * np.float32(cnt[i]))
        return bins
    for nb, lo, hi, agg in ((32, 0.0, float(vals.max()), True), (16, 2.0, 9.0, False), (1024, 0.0, 20.0, True)):
        got, (mn, mx) = plan.histogram("dp", nb, lo, hi, aggregate=agg)
        want = ref_hist(vals, nb, lo, hi, agg)
        assert got.shape == want.shape and np.array_equal(got, want) and mn == want.min() and mx == want.max(), (nb, agg)
    got, _ = plan.histogram("d", 8, 8.0, 10.0)
    assert got.shape == (1, 8) and np.array_equal(got, ref_hist(g["d__full"][:3].reshape(3, 1), 8, 8.0, 10.0, False))
    with pytest.raises(vb.MdgpuError, match="not a temporal"):
        vb.Plan(vb_system(s), vb.compile_script("r = rdf(element('O'), element('O'), 5.0);", vb_system(s)), F).histogram("r", 8, 0.0, 1.0)
    plan.close()


def _dyn_plan(tag):
    vb = _vb(); g = load_golden("dyn6.npz"); src = load_golden("water6.npz" if tag == "w" else "tric6.npz"); s = golden_system(src)
    sysm = vb_system(s); F = src["frames"].shape[0]
    plan = vb.Plan(sysm, vb.compile_script(str(g["script"]), sysm), F, keep_frame_results=True, batch_frames=3)
    cells = [vb_cell(src["cells"][f], src["cell_flags"][f]) for f in range(F)]
    plan.set_initial_frame(*src["frames"][0], cells[0])
    plan.eval_host_frames(src["frames"], cells, 0)
    return plan, g, F


@pytest.mark.parametrize("tag", ["w", "t"])
def test_dynamic_selections_as_arguments_of_every_lowered_consumer(tag):
    """SURVEY 8(f)2: within([min:]max, sel) [and static] as rdf reference AND target, sdf target, density_z argument, centre-of-mass argument
    of distance / angle / com, distance_min argument — each against the reference's values on the orthorhombic (w) and the changing
    triclinic (t) frames (tests/golden/dyn6.npz): integer bins / voxels bit-exact, floats as the static forms of the same procedures."""
    plan, g, F = _dyn_plan(tag)
    for key in ("rwt", "rww", "rwo"):
        for f in range(F):
            bins, tot = plan.frame_counts(key, f); ref = g[f"{tag}_{key}__pf"][f, :1024]
            assert np.array_equal(bins.astype(np.float32), ref) and tot == int(ref.sum()), (key, f)
        assert np.array_equal(plan.property_data(key).weights, g[f"{tag}_{key}__pf"][F - 1, 1024:]), key
    vol = np.zeros(128 ** 3, np.float32)
    for f in range(F): vol += dense_from_sparse(g[f"{tag}_vw__pf{f}_idx"], g[f"{tag}_vw__pf{f}_val"])
    assert np.array_equal(plan.counts("vw").astype(np.float32), vol) and vol.sum() > 0
    np.testing.assert_allclose(plan.property_data("dzw").values[:1024], g[f"{tag}_dzw__full"][:1024], rtol=1e-5, atol=1e-3)
    for key in ("dw", "dmw"): assert _same(plan.property_data(key).values, g[f"{tag}_{key}__full"]), key
    assert _same(plan.property_data("cmw").values, g[f"{tag}_cmw__full"])
    np.testing.assert_allclose(plan.property_data("aw").values, g[f"{tag}_aw__full"], rtol=1e-5, atol=1e-6)
    plan.close()


def test_rdf_with_an_array_of_selections_as_target():
    """tests/golden/rdftrg6.npz: rdf whose target (and in two cases also the reference) is an array of selections — the targets are the selections'
    centres of mass, binned from an AoS stream; exclusion by the target's ordinal as the reference has it. Per-frame bins, pair totals and the
    last frame's weights equal the reference's, orthorhombic and changing triclinic cell."""
    vb = _vb(); g = load_golden("rdftrg6.npz")
    for tag, name in (("w", "water6.npz"), ("t", "tric6.npz")):
        src = load_golden(name); sysm = vb_system(golden_system(src)); F = src["frames"].shape[0]
        props = vb.compile_script(str(g["script"]), sysm)
        assert [p.structure_offsets_b is not None for p in props] == [True] * 4 and [p.num_structures for p in props] == [20, 0, 40, 0]
        plan = vb.Plan(sysm, props, F, keep_frame_results=True, batch_frames=3)
        plan.eval_host_frames(src["frames"], [vb_cell(src["cells"][f], src["cell_flags"][f]) for f in range(F)], 0)
        for key in ("ra", "rb", "rc", "rd"):
            for f in range(F):
                bins, tot = plan.frame_counts(key, f); ref = g[f"{tag}_{key}__pf"][f, :1024]
                assert np.array_equal(bins.astype(np.float32), ref) and tot == int(ref.sum()) > 0, (tag, key, f)
            assert np.array_equal(plan.property_data(key).weights, g[f"{tag}_{key}__pf"][F - 1, 1024:]), (tag, key)
        plan.close()


def test_cutoffs_beyond_half_the_box():
    """tests/golden/bigcut6.npz: rdf (12, 17, 11 A; plain and centre-of-mass references) and sdf (12 A) in the 18.6 A boxes — neighbour reach of 2 - 3
    cells, pairs met through several periodic images — bins and voxels equal to the reference's, orthorhombic and changing triclinic cell."""
    vb = _vb(); g = load_golden("bigcut6.npz")
    for tag, name in (("w", "water6.npz"), ("t", "tric6.npz")):
        src = load_golden(name); sysm = vb_system(golden_system(src)); F = 2
        plan = vb.Plan(sysm, vb.compile_script(str(g["script"]), sysm), F, keep_frame_results=True)
        cells = [vb_cell(src["cells"][f], src["cell_flags"][f]) for f in range(F)]
        plan.set_initial_frame(*src["frames"][0], cells[0]); plan.eval_host_frames(src["frames"][:F], cells, 0)
        for key in ("r1", "r2", "r4"):
            for f in range(F):
                bins, tot = plan.frame_counts(key, f); ref = g[f"{tag}_{key}__pf"][f, :1024]
                assert np.array_equal(bins.astype(np.float32), ref) and tot == int(ref.sum()) > 0, (tag, key, f)
        vol = np.zeros(128 ** 3, np.float32)
        for f in range(F): vol += dense_from_sparse(g[f"{tag}_v__pf{f}_idx"], g[f"{tag}_v__pf{f}_val"])
        assert np.array_equal(plan.counts("v").astype(np.float32), vol) and vol.sum() > 0, tag
        plan.close()


def test_array_of_selections_as_one_position_argument():
    """angle / dihedral / com with an ARRAY of selections as one argument (residue(a:b) over several residues): the centre of the selections'
    centres — md_util_com_compute per selection, then md_util_com_compute_vec4 (coordinate_extract_com md_script_functions.inl:1826-1842) —
    while distance() is FLAG_FLATTEN and takes the union, com(...) inside it included. Against the reference (tests/golden/arrargs.npz),
    orthorhombic and changing triclinic cell (whose vec4 centre goes through the scaled inverse twice, as written)."""
    vb = _vb(); g = load_golden("arrargs.npz")
    for tag, name in (("w", "water6.npz"), ("t", "tric6.npz")):
        src = load_golden(name); sysm = vb_system(golden_system(src)); F = src["frames"].shape[0]
        props = vb.compile_script(str(g["script"]), sysm)
        assert {p.name: sorted(p.arg_offsets) for p in props} == {"da": [], "db": [], "dc": [], "aa": [0, 1], "ha": [0, 1, 2, 3], "ca": [0], "cb": [0], "dd": [],
                                                                    "dmg": [], "dmh": [], "dxg": [], "cxg": [], "czg": [], "plg": [], "plh": [],
                                                                    "dctx": [0, 1], "actx": [0, 1], "ectx": [0, 1], "hctx": [1, 2]}
        assert [(p.num_structures, p.structure_offsets_b is not None) for p in props[-11:-4]] == [(4, True), (0, True), (3, False), (5, False), (31, False), (10, False), (181, False)]
        assert [p.num_structures for p in props[-4:]] == [10, 5, 4, 216]   # contexts
        plan = vb.Plan(sysm, props, F, batch_frames=3)
        plan.eval_host_frames(src["frames"], [vb_cell(src["cells"][f], src["cell_flags"][f]) for f in range(F)], 0)
        for key in ("da", "db", "dc", "dd", "ca", "cb"): assert _same(plan.property_data(key).values, g[f"{tag}_{key}__full"]), (tag, key)
        for key in ("dmg", "dmh", "dxg", "cxg", "czg"):   # one centre of mass per selection: distance_min / _max over them, coord_* of them
            assert np.array_equal(plan.property_data(key).values, g[f"{tag}_{key}__full"]), (tag, key)
        for key in ("plg", "plh"): assert _same(plan.property_data(key).values, g[f"{tag}_{key}__full"]), (tag, key)   # the plane through the selections' centres of mass
        for key in ("dctx", "ectx"): assert _same(plan.property_data(key).values, g[f"{tag}_{key}__full"]), (tag, key)   # selections inside `in` contexts
        for key in ("actx", "hctx"): np.testing.assert_allclose(plan.property_data(key).values, g[f"{tag}_{key}__full"], rtol=1e-5, atol=1e-6, err_msg=f"{tag} {key}")
        for key in ("aa", "ha"): np.testing.assert_allclose(plan.property_data(key).values, g[f"{tag}_{key}__full"], rtol=1e-5, atol=1e-6, err_msg=f"{tag} {key}")
        plan.close()
    with pytest.raises(vb.MdgpuError):   # offsets that do not cover the list
        p = vb.angle("x", [np.arange(0, 3), np.arange(3, 6)], 10, 20); p.arg_offsets[0] = np.array([0, 3, 5], np.uint32)
        vb.Plan(sysm, [p], 2)


@pytest.mark.parametrize("tag", ["w", "t"])
def test_contact_count_running_totals(tag):
    """contact_count(A[], B, cutoff) (md_script_functions.inl:2756-2866) with disjoint sets — the reference's exclusion mask is then empty and its
    result deterministic: per frame the RUNNING total over the sets (the reference never resets its counter), equal to the reference's floats."""
    plan, g, F = _dyn_plan(tag)
    for key in ("cc", "cc2"):
        d = plan.property_data(key); ref = g[f"{tag}_{key}__full"]
        assert d.values.shape == ref.shape and np.array_equal(d.values, ref), key
        row = d.values.reshape(F, -1); assert np.all(np.diff(row, axis=1) >= 0) and row[:, -1].min() > 0
    plan.close()


def test_contact_count_exclusion_lists_and_errors():
    """overlapping sets: b atoms within `path_length` bonds of A_i & B are excluded (md_util_mask_grow_by_bonds, intended breadth-first semantics —
    the reference walks an unzeroed depth array there, md_util.c:5560, so this case is pinned against a brute-force count, not the reference)."""
    vb = _vb(); g = load_golden("water6.npz"); s = golden_system(g); sysm = vb_system(s); F = g["frames"].shape[0]
    A = [np.arange(0, 9, dtype=np.int32), np.arange(30, 36, dtype=np.int32)]; Bsel = np.arange(0, 120, dtype=np.int32)
    plan = vb.Plan(sysm, [vb.contact_count("c", A, Bsel, 3.5, sysm, 1)], F)
    cells = [vb_cell(g["cells"][f], g["cell_flags"][f]) for f in range(F)]
    plan.eval_host_frames(g["frames"], cells, 0)
    got = plan.property_data("c").values.reshape(F, 2)
    for f in range(F):
        x, y, z = g["frames"][f]; cell = cell_from_row(g["cells"][f], g["cell_flags"][f]); run = 0; want = []
        for a_set in A:
            excl = set(vb.api.grow_by_bonds(np.intersect1d(a_set, Bsel), sysm.conn_offset, sysm.conn_idx, 1).tolist())
            trg = np.array([b for b in Bsel if b not in excl], np.int32)
            run += O.count_pairs(x, y, z, a_set, trg, cell, 3.5, 3.5); want.append(run)
        assert list(got[f]) == [float(w) for w in want], f
    with pytest.raises(vb.MdgpuError, match="cutoff distance must be positive"):
        vb.Plan(sysm, [vb.contact_count("c", A, Bsel, 0.0, sysm)], F)
    plan.close()


def test_array_and_context_forms_with_empty_or_single_atom_groups():
    """Degenerate groups in the array / context forms: an empty selection inside an array (its centre is (0, 0, 0), md_util_com_compute's count == 0
    answer, md_util.c:8168), an empty (selection AND context), single-atom selections, 216 parts in one argument — no fault, finite values, and the
    non-degenerate entries equal the same quantity computed without the degenerate neighbours."""
    vb = _vb(); g = load_golden("water6.npz"); sysm = vb_system(golden_system(g)); F = 2
    cells = [vb_cell(g["cells"][f], g["cell_flags"][f]) for f in range(F)]; E = np.zeros(0, np.int32)
    props = [vb.in_contexts("c_empty", vb.OP_DISTANCE, [[np.array([0], np.int32), E, np.array([6], np.int32)], 1], [0, 3, 6]),
             vb.in_contexts("c_full", vb.OP_DISTANCE, [[np.array([0], np.int32), np.array([6], np.int32)], 1], [0, 6]),
             vb.angle("a_emptypart", [np.arange(0, 3), E, np.arange(6, 9)], 10, 20),
             vb.com("c_single", [np.array([5], np.int32), np.array([7], np.int32)]),
             vb.distance_min("dm_g", [np.arange(0, 3), E], [np.arange(30, 33), np.arange(60, 63)]),
             vb.coord("cx_g", 0, [np.arange(0, 3), E, np.arange(3, 4)]), vb.coord("cx_a", 0, [np.arange(0, 3), np.arange(3, 4)]),
             vb.rdf("rt_g", np.arange(0, 60, 3), [np.arange(3 * k, 3 * k + 3) for k in range(40, 44)] + [E], 6.0),
             vb.com("c_many", [np.arange(3 * k, 3 * k + 3) for k in range(216)])]
    plan = vb.Plan(sysm, props, F, keep_frame_results=True); plan.set_initial_frame(*g["frames"][0], cells[0]); plan.eval_host_frames(g["frames"][:F], cells, 0)
    val = {p.name: np.asarray(plan.property_data(p.name).values).copy() for p in props}
    assert all(np.all(np.isfinite(v)) for v in val.values())
    assert np.array_equal(val["c_empty"].reshape(F, 3)[:, [0, 2]], val["c_full"].reshape(F, 2))
    assert np.array_equal(val["cx_g"].reshape(F, 3)[:, [0, 2]], val["cx_a"].reshape(F, 2)) and np.all(val["cx_g"].reshape(F, 3)[:, 1] == 0)
    plan.close()


@pytest.mark.parametrize("golden,seed", [("water6.npz", "77"), ("tric6.npz", "91")])
def test_statement_forms_against_the_reference_itself(golden, seed):
    """The 45-form sweep of tests/test_emulated_library.py with libmdgpu itself on the device: the library evaluates the lowered statements on the
    GPU, against the reference's results stored in tests/golden/forms45.npz."""
    from test_emulated_library import run_statement_forms
    run_statement_forms(golden, seed)
