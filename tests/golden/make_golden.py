"""Generate the golden fixtures in tests/golden/ from the UNMODIFIED reference (oracle/_ref/ref_harness_strict).

Run here (needs /root/reference + `make -C oracle ref oracle`):   python tests/golden/make_golden.py
The fixtures are small .npz files; each stores the inputs (coordinates, cells, system statics) together with the
reference's outputs, so the tests need neither the reference nor the harness on the GPU box.

  water6.npz : synthetic water n=6 (648 atoms, L=18.624), 4 frames:
               r  = rdf(element('O'), element('O'), 6.0)            per-frame raw bins + weights + 4-frame mean
               rh = rdf(element('O'), element('H'), 1.5:6.0)         (min:max form)
               v  = sdf(residue(1:20), element('O'), 5.0)            per-frame raw voxels (sparse)
               dz/dx = density_z / density_x (element('O'))          per-frame bins
               d, a, t = distance(1,10), angle(1,2,3), dihedral(1,4,7,10)
               rc = rdf(residue(1:20), element('O'), 5.0)            centre-of-mass references + exclusion masks (array-of-bitfields form)
               dc, ac, tc, dg, dm                                     distance/angle/dihedral whose arguments are selections (periodic centre of mass)
  membrane6.npz : synthetic coarse-grained membrane (BASELINE config 4 shape at 1728 atoms: 72 lipids x 12 beads + 864 solvent beads,
               cell 48 x 48 x 75), 4 frames: rt = rdf(name('C2*'), name('C2*'), 12.0), dz = density_z(name('C2*')), dall/dxall = density over all atoms
  tric6.npz  : water n=6 sheared into a TRICLINIC cell that changes every frame, 4 frames: rt, rth (min:max), rtc (centre-of-mass references)
  tric6_rmsd.npz : the tric6 frames again: rmt = rmsd(residue(1:10)), rma = rmsd(atom(100:160)), rmo = rmsd(element('O')) — the triclinic wrap
               A * fract(I * r) of md_util_pbc_vec4, the triclinic bond-walk unwrap, non-contiguous selections
  pairs6.npz : multi-valued temporals on the water6 and the tric6 frames, each with its per-frame aggregates: distance_pair() matrices
               (5 x 11 and 3 x 216 per frame), com() of a residue / 30 atoms / one atom, plane() of 30 atoms / all oxygens; count(within(min:max, sel)); angle / distance / dihedral evaluated `in` residue contexts
  shapes.npz : shape weights (linear, planar, isotropic) per structure and frame through the reference's md_util functions, as VIAMD's shape-space
               component calls them: 1ALA residues (mass-weighted), water6 residues (unit weights), tric6 residues
  xtc_cases.npz : XTC byte streams from the reference's writer + the reference reader's decode of them (see xtc_cases below)
  ala50.npz  : first 50 frames of datasets/1ALA-500.pdb (153 atoms, ortho cell 46.645 x 96.666 x 48.362), config 1:
               d = distance(1,10) (BASELINE config 1), rc = rdf(element('C'), element('O'), 10.0), dz = density_z(element('C')),
               a = angle(1,5,9), t = dihedral(5,7,9,15), rr = rdf(residue(1:3), element('H'), 8.0) (COM references, groups of different sizes)
"""
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import refio  # noqa: E402

HARNESS = os.path.join(ROOT, "oracle", "_ref", "ref_harness_strict")
SHIM = os.path.join(ROOT, "oracle", "_ref", "shim_harness")
SYNTH = os.path.join(ROOT, "oracle", "build", "synth_tool")


def run(*a):
    subprocess.check_call(list(a), stdout=subprocess.DEVNULL)


def sparse(v):
    nz = np.nonzero(v)[0].astype(np.uint32)
    return nz, v[nz].astype(np.float32)


def sysdict(s):
    return dict(mass=s["mass"], z=s["z"].astype(np.uint8), names=np.array(s["names"]), comp_off=s["comp_off"],
                conn_off=s["conn_off"], conn_idx=s["conn_idx"])


def pack(out, props, frames):
    for name, p in props.items():
        out[f"{name}__flags"] = np.int32(p.flags); out[f"{name}__dim"] = np.array(p.dim, np.int32)
        if p.flags & refio.FLAG_VOLUME:
            for f in frames:
                i, v = sparse(p.perframe[f]); out[f"{name}__pf{f}_idx"] = i; out[f"{name}__pf{f}_val"] = v
            i, v = sparse(p.full); out[f"{name}__full_idx"] = i; out[f"{name}__full_val"] = v
        elif p.flags & refio.FLAG_TEMPORAL:
            out[f"{name}__full"] = p.full
        else:
            out[f"{name}__pf"] = np.stack([p.perframe[f] for f in frames]); out[f"{name}__full"] = p.full
        m = p.meta[(1, frames[0])]
        out[f"{name}__meta"] = np.array([m["min_value"], m["max_value"], m["min_range"][0], m["max_range"][0]], np.float32)


def water6(tmp):
    n, seed, F = 6, 77, 4
    gro, raw = os.path.join(tmp, "w.gro"), os.path.join(tmp, "w.raw")
    run(SYNTH, "water-gro", str(n), str(seed), gro); run(SYNTH, "water-raw", str(n), str(seed), str(F), raw)
    script = ("r = rdf(element('O'), element('O'), 6.0); rh = rdf(element('O'), element('H'), 1.5:6.0); "
              "v = sdf(residue(1:20), element('O'), 5.0); dz = density_z(element('O')); dx = density_x(element('O')); "
              "d = distance(1,10); a = angle(1,2,3); t = dihedral(1,4,7,10); "
              "rc = rdf(residue(1:20), element('O'), 5.0); "
              "dc = distance(residue(1), residue(5)); ac = angle(residue(1), residue(2), residue(3)); "
              "tc = dihedral(residue(1), residue(2), residue(3), residue(4)); dg = distance(atom(1:30), atom(100:151)); dm = distance(atom(1:30), 200); "
              "dmn = distance_min(residue(1), atom(100:648)); dmx = distance_max(atom(1:30), atom(100:151)); dmh = distance_min(element('H'), atom(300:400)); rm = rmsd(residue(1:10)); "
              "cw = count(within(4.0, residue(1))); cw2 = count(within(7.5, atom(10:12))); rw = rdf(within(4.0, residue(1)), element('O'), 6.0);")
    o = os.path.join(tmp, "w.out"); si = os.path.join(tmp, "w.sys")
    run(HARNESS, "eval", "--sys", gro, "--traj", f"raw:{raw}", "--script", script, "--out", o, "--perframe", f"0:{F}", "--full", f"0:{F}")
    run(HARNESS, "sysinfo", "--sys", gro, "--out", si)
    frames, cells, flags = refio.read_raw_traj(raw)
    out = dict(script=np.array(script), n=np.int32(n), seed=np.int32(seed), frames=frames, cells=cells, cell_flags=flags, **sysdict(refio.read_sysinfo(si)))
    pack(out, refio.read_refout(o), list(range(F)))
    np.savez_compressed(os.path.join(HERE, "water6.npz"), **out)


def ala50(tmp):
    pdb = "/root/reference/datasets/1ALA-500.pdb"; F = 50
    raw = os.path.join(tmp, "a.raw"); o = os.path.join(tmp, "a.out"); si = os.path.join(tmp, "a.sys")
    run(HARNESS, "dumptraj", "--sys", pdb, "--traj", "sys", "--frames", f"0:{F}", "--out", raw)
    script = ("d = distance(1,10); rc = rdf(element('C'), element('O'), 10.0); dz = density_z(element('C')); "
              "a = angle(1,5,9); t = dihedral(5,7,9,15); rr = rdf(residue(1:3), element('H'), 8.0); "
              "dr = distance(residue(1), residue(15)); ar = angle(residue(1), residue(7), residue(15)); tr = dihedral(residue(1), residue(5), 100, residue(15)); rma = rmsd(residue(1:15));")
    # evaluate on the dumped frames so that frame 0 (initial configuration) is identical
    run(HARNESS, "eval", "--sys", pdb, "--traj", f"raw:{raw}", "--script", script, "--out", o, "--perframe", f"0:{F}", "--full", f"0:{F}")
    run(HARNESS, "sysinfo", "--sys", pdb, "--out", si)
    frames, cells, flags = refio.read_raw_traj(raw)
    out = dict(script=np.array(script), frames=frames, cells=cells, cell_flags=flags, **sysdict(refio.read_sysinfo(si)))
    pack(out, refio.read_refout(o), list(range(F)))
    # the published-by-probe numbers of BASELINE config 1 (SURVEY.md §8d): values[0]=2.770258, sum over 500 frames=1493.846763
    o2 = os.path.join(tmp, "a2.out")
    run(HARNESS, "eval", "--sys", pdb, "--traj", "sys", "--script", "d = distance(1,10);", "--out", o2, "--full", "0:500")
    out["d500__full"] = refio.read_refout(o2)["d"].full
    np.savez_compressed(os.path.join(HERE, "ala50.npz"), **out)


def membrane6(tmp):
    nl, nwxy, nwz, seed, F = 6, 12, 3, 4321, 4
    gro, raw = os.path.join(tmp, "m.gro"), os.path.join(tmp, "m.raw")
    run(SYNTH, "membrane-gro", str(nl), str(nwxy), str(nwz), str(seed), gro)
    run(SYNTH, "membrane-raw", str(nl), str(nwxy), str(nwz), str(seed), str(F), raw)
    script = "rt = rdf(name('C2*'), name('C2*'), 12.0); dz = density_z(name('C2*')); dall = density_z(all); dxall = density_x(all);"
    o = os.path.join(tmp, "m.out"); si = os.path.join(tmp, "m.sys")
    run(HARNESS, "eval", "--sys", gro, "--traj", f"raw:{raw}", "--script", script, "--out", o, "--perframe", f"0:{F}", "--full", f"0:{F}")
    run(HARNESS, "sysinfo", "--sys", gro, "--out", si)
    frames, cells, flags = refio.read_raw_traj(raw)
    out = dict(script=np.array(script), params=np.array([nl, nwxy, nwz, seed], np.int32), frames=frames, cells=cells, cell_flags=flags,
               **sysdict(refio.read_sysinfo(si)))
    pack(out, refio.read_refout(o), list(range(F)))
    np.savez_compressed(os.path.join(HERE, "membrane6.npz"), **out)


def tric6(tmp):
    """water n=6 sheared into a triclinic cell (a = (L,0,0), b = (xy,L,0), c = (xz,yz,L)), the cell changing from frame to frame:
    pins the triclinic branch of the pair query (md_spatial_acc.c:1498-1647) and the triclinic cell-list build."""
    n, seed, F = 6, 91, 4
    gro, raw0, raw = os.path.join(tmp, "t.gro"), os.path.join(tmp, "t0.raw"), os.path.join(tmp, "t.raw")
    run(SYNTH, "water-gro", str(n), str(seed), gro); run(SYNTH, "water-raw", str(n), str(seed), str(F), raw0)
    fr, cells, _ = refio.read_raw_traj(raw0)
    out_fr = np.empty_like(fr); out_cells = np.empty_like(cells); flags = np.full(F, 2 | 4 | 8 | 16, np.uint32)
    for f in range(F):
        L = cells[f][0]; xy, xz, yz = 3.1 + 0.2 * f, -2.2 - 0.1 * f, 4.3 - 0.15 * f
        x, y, z = fr[f].astype(np.float64)
        out_fr[f, 0] = (x + (xy / L) * y + (xz / L) * z).astype(np.float32)
        out_fr[f, 1] = (y + (yz / L) * z).astype(np.float32); out_fr[f, 2] = z.astype(np.float32)
        out_cells[f] = [L, xy, xz, L, yz, L]
    refio.write_raw_traj(raw, out_fr, out_cells, flags)
    script = "rt = rdf(element('O'), element('O'), 6.0); rth = rdf(element('O'), element('H'), 2.0:7.0); rtc = rdf(residue(1:30), element('H'), 5.0); vt = sdf(residue(1:20), element('O'), 5.0); dmt = distance_min(atom(1:30), atom(100:151)); dmxt = distance_max(element('O'), atom(7:9));"
    o = os.path.join(tmp, "t.out"); si = os.path.join(tmp, "t.sys")
    run(HARNESS, "eval", "--sys", gro, "--traj", f"raw:{raw}", "--script", script, "--out", o, "--perframe", f"0:{F}", "--full", f"0:{F}")
    run(HARNESS, "sysinfo", "--sys", gro, "--out", si)
    out = dict(script=np.array(script), frames=out_fr, cells=out_cells, cell_flags=flags, **sysdict(refio.read_sysinfo(si)))
    pack(out, refio.read_refout(o), list(range(F)))
    np.savez_compressed(os.path.join(HERE, "tric6.npz"), **out)


def tric6_rmsd(tmp):
    """rmsd() in the changing triclinic cell of tric6 (its frames are reused): md_util_pbc_vec4's triclinic wrap + unwrap + Kabsch."""
    g = np.load(os.path.join(HERE, "tric6.npz")); F = g["frames"].shape[0]
    gro, raw = os.path.join(tmp, "tr.gro"), os.path.join(tmp, "tr.raw")
    run(SYNTH, "water-gro", "6", "91", gro); refio.write_raw_traj(raw, g["frames"], g["cells"], g["cell_flags"])
    script = "rmt = rmsd(residue(1:10)); rma = rmsd(atom(100:160)); rmo = rmsd(element('O'));"
    o = os.path.join(tmp, "tr.out")
    run(HARNESS, "eval", "--sys", gro, "--traj", f"raw:{raw}", "--script", script, "--out", o, "--full", f"0:{F}")
    out = dict(script=np.array(script))
    pack(out, refio.read_refout(o), list(range(F)))
    np.savez_compressed(os.path.join(HERE, "tric6_rmsd.npz"), **out)


def pairs6(tmp):
    """Multi-valued temporals: distance_pair() matrices with their per-frame aggregates (mean / variance / extent, md_script.c:5646-5677),
    on the water6 frames (orthorhombic) and the tric6 frames (triclinic cell changing every frame)."""
    out = {}
    script = ("dp = distance_pair(atom(1:5), atom(20:30)); dpo = distance_pair(residue(1), element('O')); "
              "c = com(residue(1)); ca = com(atom(1:30)); ci = com(5); pl = plane(atom(1:30)); plo = plane(element('O')); "
              "cwr = count(within(2.5:5.0, residue(1))); cwr2 = count(within(3.0:8.0, atom(10:40))); "
              "anc = angle(2,1,3) in residue(1:10); ddc = distance(1,3) in residue(:); dhc = dihedral(1,2,3,1) in residue(3:4); "
              "cx = coord_x(residue(1)); cz = coord_z(atom(5:40)); cyi = coord_y(7); "
              "cwo = count(element('O') and within(4.0, residue(1))); cwh = count(within(2.5:5.0, residue(1)) and element('H')); "
              "cwg = count(within(6.0, residue(1:5))); cwg2 = count(within(2.0:4.5, residue(10:40))); "
              "dpg = distance_pair(residue(1:4), residue(10:15)); dpm = distance_pair(residue(2:5), atom(100:103));")
    w = np.load(os.path.join(HERE, "water6.npz")); t = np.load(os.path.join(HERE, "tric6.npz"))
    for tag, g, seed in (("w", w, "77"), ("t", t, "91")):
        gro, raw, o = os.path.join(tmp, tag + "p.gro"), os.path.join(tmp, tag + "p.raw"), os.path.join(tmp, tag + "p.out")
        F = g["frames"].shape[0]
        run(SYNTH, "water-gro", "6", seed, gro); refio.write_raw_traj(raw, g["frames"], g["cells"], g["cell_flags"])
        run(HARNESS, "eval", "--sys", gro, "--traj", f"raw:{raw}", "--script", script, "--out", o, "--full", f"0:{F}")
        for name, p in refio.read_refout(o).items():
            k = f"{tag}_{name}"
            out[k + "__dim"] = np.array(p.dim, np.int32); out[k + "__full"] = p.full
            m = p.meta[(1, 0)]; out[k + "__meta"] = np.array([m["min_value"], m["max_value"], m["min_range"][0], m["max_range"][0]], np.float32)
            if p.aggregate is not None: out[k + "__mean"] = p.aggregate["mean"]; out[k + "__var"] = p.aggregate["var"]; out[k + "__ext"] = p.aggregate["ext"]
    out["script"] = np.array(script)
    np.savez_compressed(os.path.join(HERE, "pairs6.npz"), **out)


ARR_SCRIPT = ("da = distance(residue(1:4), residue(10)); db = distance(residue(2:9), residue(20:31)); dc = distance(residue(1:3), 40); "
              "aa = angle(residue(1:2), residue(5:7), 30); ha = dihedral(residue(1:2), residue(3:4), residue(5:6), residue(7:9)); "
              "ca = com(residue(1:6)); cb = com(residue(100:140)); dd = distance(com(residue(1:4)), residue(50:52)); "
              # one position (centre of mass, extract_com) per selection of an array: distance_min / _max, coord_*
              "dmg = distance_min(residue(1:4), residue(10:30)); dmh = distance_min(residue(1), residue(2:9)); dxg = distance_max(residue(3:5), element('O')); "
              "cxg = coord_x(residue(1:5)); czg = coord_z(residue(10:40)); plg = plane(residue(1:10)); plh = plane(residue(20:200)); "
              # selections inside `in` contexts: per context the centre of mass of (selection AND context); atom(a:b) relative to the context
              "dctx = distance(element('O'), element('H')) in residue(1:10); actx = angle(atom(2), element('O'), 3) in residue(1:5); "
              "ectx = distance(element('O'), atom(2:3)) in residue(2:5); hctx = dihedral(1, element('O'), atom(2:3), 3) in residue(:);")


def arrargs(tmp):
    """An ARRAY of selections as ONE position argument of distance / angle / dihedral / com: the centre of the selections' centres
    (coordinate_extract_com md_script_functions.inl:1826-1842 -> md_util_com_compute per selection, then md_util_com_compute_vec4, whose triclinic
    branch is the one 'as written'), on the water6 frames (orthorhombic) and the tric6 frames (triclinic cell changing every frame)."""
    out = {"script": np.array(ARR_SCRIPT)}
    w = np.load(os.path.join(HERE, "water6.npz")); t = np.load(os.path.join(HERE, "tric6.npz"))
    for tag, g, seed in (("w", w, "77"), ("t", t, "91")):
        gro, raw, o = os.path.join(tmp, tag + "a.gro"), os.path.join(tmp, tag + "a.raw"), os.path.join(tmp, tag + "a.out")
        F = g["frames"].shape[0]
        run(SYNTH, "water-gro", "6", seed, gro); refio.write_raw_traj(raw, g["frames"], g["cells"], g["cell_flags"])
        run(HARNESS, "eval", "--sys", gro, "--traj", f"raw:{raw}", "--script", ARR_SCRIPT, "--out", o, "--full", f"0:{F}")
        for name, pr in refio.read_refout(o).items():
            out[f"{tag}_{name}__dim"] = np.array(pr.dim, np.int32); out[f"{tag}_{name}__full"] = pr.full
    np.savez_compressed(os.path.join(HERE, "arrargs.npz"), **out)


BIGCUT_SCRIPT = "r1 = rdf(element('O'), element('O'), 12.0); r2 = rdf(element('O'), element('H'), 17.0); v = sdf(residue(1:10), element('O'), 12.0); r4 = rdf(residue(1:20), element('H'), 11.0);"


def bigcut6(tmp):
    """Cutoffs beyond half the box (12, 17 and 11 A in the 18.6 A water6 / tric6 boxes): the neighbour reach grows to 2 - 3 cells per axis, a pair is
    met through several periodic images and the reference's single wrap decides which of them count (md_spatial_acc.c:1724-1755). (Beyond the box
    length the reference itself crashes: rdf(..., 25.0) segfaults there, so that regime has no parity to pin.)"""
    out = {"script": np.array(BIGCUT_SCRIPT)}
    w = np.load(os.path.join(HERE, "water6.npz")); t = np.load(os.path.join(HERE, "tric6.npz")); F = 2
    for tag, g, seed in (("w", w, "77"), ("t", t, "91")):
        gro, raw, o = os.path.join(tmp, tag + "b.gro"), os.path.join(tmp, tag + "b.raw"), os.path.join(tmp, tag + "b.out")
        run(SYNTH, "water-gro", "6", seed, gro); refio.write_raw_traj(raw, g["frames"][:F], g["cells"][:F], g["cell_flags"][:F])
        run(HARNESS, "eval", "--sys", gro, "--traj", f"raw:{raw}", "--script", BIGCUT_SCRIPT, "--out", o, "--perframe", f"0:{F}", "--full", f"0:{F}")
        sub = {}; pack(sub, refio.read_refout(o), list(range(F)))
        for k, v in sub.items(): out[f"{tag}_{k}"] = v
    np.savez_compressed(os.path.join(HERE, "bigcut6.npz"), **out)


RDFTRG_SCRIPT = ("ra = rdf(residue(1:20), residue(10:30), 5.0); rb = rdf(element('O'), residue(10:60), 6.0); rc = rdf(residue(1:40), residue(1:40), 2.0:8.0); "
                 "rd = rdf(atom(1:60), residue(1:20), 4.0);")


def rdftrg6(tmp):
    """An ARRAY of selections as rdf TARGET: one centre of mass per selection is the target point (coordinate_extract md_script_functions.inl:1503 ->
    extract_com :857, compute_rdf :5293-5302). With an array as reference too, the exclusion test reads bit j of reference group i's mask with j the
    target's ORDINAL (rdf_cb_excl_mask :5252) — reproduced as written. water6 (orthorhombic) and tric6 (triclinic, cell changing every frame)."""
    out = {"script": np.array(RDFTRG_SCRIPT)}
    w = np.load(os.path.join(HERE, "water6.npz")); t = np.load(os.path.join(HERE, "tric6.npz"))
    for tag, g, seed in (("w", w, "77"), ("t", t, "91")):
        gro, raw, o = os.path.join(tmp, tag + "g.gro"), os.path.join(tmp, tag + "g.raw"), os.path.join(tmp, tag + "g.out")
        F = g["frames"].shape[0]
        run(SYNTH, "water-gro", "6", seed, gro); refio.write_raw_traj(raw, g["frames"], g["cells"], g["cell_flags"])
        run(HARNESS, "eval", "--sys", gro, "--traj", f"raw:{raw}", "--script", RDFTRG_SCRIPT, "--out", o, "--perframe", f"0:{F}", "--full", f"0:{F}")
        sub = {}; pack(sub, refio.read_refout(o), list(range(F)))
        for k, v in sub.items(): out[f"{tag}_{k}"] = v
    np.savez_compressed(os.path.join(HERE, "rdftrg6.npz"), **out)


def shapes(tmp):
    """Shape weights per structure and frame from the reference's own functions (harness mode `shapespace`: the loop body of VIAMD's shape-space
    component): 1ALA residues (15 structures of 9-12 atoms, orthorhombic, mass-weighted), water6 residues with unit weights, tric6 residues."""
    out = {}
    a = np.load(os.path.join(HERE, "ala50.npz")); w = np.load(os.path.join(HERE, "water6.npz")); t = np.load(os.path.join(HERE, "tric6.npz"))
    for tag, g, sysarg, res, mass in (("a", a, "/root/reference/datasets/1ALA-500.pdb", "0:15", "1"), ("w", w, None, "0:40", "0"), ("t", t, None, "0:40", "1")):
        raw, o = os.path.join(tmp, tag + "s.raw"), os.path.join(tmp, tag + "s.bin")
        if sysarg is None:
            sysarg = os.path.join(tmp, tag + "s.gro"); run(SYNTH, "water-gro", "6", "77" if tag == "w" else "91", sysarg)
        refio.write_raw_traj(raw, g["frames"], g["cells"], g["cell_flags"])
        run(HARNESS, "shapespace", "--sys", sysarg, "--traj", f"raw:{raw}", "--res", res, "--mass", mass, "--out", o)
        b = open(o, "rb").read(); assert b[:8] == b"MDSHAPES"
        F, n = np.frombuffer(b, np.uint64, 2, 8)
        out[tag + "__weights"] = np.frombuffer(b, np.float32, -1, 24).reshape(int(F), int(n), 3).copy(); out[tag + "__res"] = np.array(res); out[tag + "__mass"] = np.int32(int(mass))
    np.savez_compressed(os.path.join(HERE, "shapes.npz"), **out)


def water32_full(tmp):
    """BASELINE configs 2 + 3 at FULL size from the strict reference: water n=32 (98 304 atoms), seed 1234, frames 0..1:
    r = rdf(element('O'), element('O'), 10.0) per-frame raw bins + weights, v = sdf(residue(1:1000), element('O'), 10.0) per-frame raw
    voxels (sparse: ~3e5 of 2 097 152 per frame). Coordinates are not stored — the tests regenerate them with the same generator
    (viamd_b200/csrc/synth.h) and check the sha256 kept here."""
    import hashlib
    n, seed, F = 32, 1234, 2
    gro, raw = os.path.join(tmp, "w32.gro"), os.path.join(tmp, "w32.raw")
    run(SYNTH, "water-gro", str(n), str(seed), gro); run(SYNTH, "water-raw", str(n), str(seed), str(F), raw)
    script = "r = rdf(element('O'), element('O'), 10.0); v = sdf(residue(1:1000), element('O'), 10.0);"
    o = os.path.join(tmp, "w32.out")
    run(HARNESS, "eval", "--sys", gro, "--traj", f"raw:{raw}", "--script", script, "--out", o, "--perframe", f"0:{F}", "--full", f"0:{F}")
    frames, cells, flags = refio.read_raw_traj(raw)
    out = dict(script=np.array(script), n=np.int32(n), seed=np.int32(seed), cells=cells, cell_flags=flags,
               frames_sha256=np.array([hashlib.sha256(np.ascontiguousarray(f).tobytes()).hexdigest() for f in frames]))
    pack(out, refio.read_refout(o), list(range(F)))
    for k in [k for k in out if k.startswith("v__") and k.endswith("_idx")]:   # voxel index lists -> bit mask of the non-zero voxels: half the size
        mask = np.zeros(128 ** 3, bool); mask[out.pop(k)] = True; out[k[:-4] + "_mask"] = np.packbits(mask)   # compressed (helpers.dense_from_mask)
    np.savez_compressed(os.path.join(HERE, "water32_full.npz"), **out)


def water12_avg(tmp):
    """Long-run AVERAGED results (the reference's float cumulative moving average, md_script.c:5909-5955, one thread = frame order):
    water n=12 (5184 atoms), seed 4242, 4096 frames: rdf bins + weights, density_z bins, sdf voxels (every 16th non-zero voxel + the sum
    over all voxels, to keep the fixture small). Pins the 1e-5 bar of averaged values at the frame counts BASELINE's configs use."""
    n, seed, F = 12, 4242, 4096
    gro, raw = os.path.join(tmp, "w12.gro"), os.path.join(tmp, "w12.raw")
    run(SYNTH, "water-gro", str(n), str(seed), gro); run(SYNTH, "water-raw", str(n), str(seed), str(F), raw)
    script = "r = rdf(element('O'), element('O'), 8.0); v = sdf(residue(1:100), element('O'), 6.0); dz = density_z(element('O'));"
    o = os.path.join(tmp, "w12.out")
    run(HARNESS, "eval", "--sys", gro, "--traj", f"raw:{raw}", "--script", script, "--out", o, "--full", f"0:{F}", "--threads", "1")
    props = refio.read_refout(o)
    out = dict(script=np.array(script), n=np.int32(n), seed=np.int32(seed), num_frames=np.int32(F))
    for name in ("r", "dz"):
        out[f"{name}__full"] = props[name].full
        m = props[name].meta[(1, 0)]; out[f"{name}__meta"] = np.array([m["min_value"], m["max_value"], m["min_range"][0], m["max_range"][0]], np.float32)
    v = props["v"].full; nz = np.nonzero(v)[0].astype(np.uint32)
    out["v__nnz"] = np.int64(len(nz)); out["v__sum"] = np.float64(v.astype(np.float64).sum())
    out["v__sample_idx"] = nz[::16]; out["v__sample_val"] = v[nz[::16]]
    np.savez_compressed(os.path.join(HERE, "water12_avg.npz"), **out)


DYN_SCRIPT = ("rwt = rdf(element('O'), within(4.0, residue(1)), 6.0); rww = rdf(within(4.0, residue(1)), within(5.0, residue(2)), 6.0); "
              "vw = sdf(residue(1:20), within(6.0, residue(1:5)), 5.0); dzw = density_z(within(5.0, residue(1))); dw = distance(within(4.0, residue(1)), 200); "
              "cmw = com(within(4.0, residue(1))); dmw = distance_min(within(3.5, residue(1)), residue(30)); "
              "rwo = rdf(element('O') and within(5.0, residue(2)), element('H') and within(6.0, residue(3)), 5.0); aw = angle(within(2.5:5.0, residue(4)), 10, residue(7)); "
              "cc = contact_count(residue(1:5), residue(10:40), 4.0); cc2 = contact_count(residue(3:20), element('O') and residue(50:216), 3.5);")


def dyn6(tmp):
    """Dynamic selections (within([min:]max, sel) [and static]) as arguments of every consumer the device path lowers, and contact_count with
    disjoint sets (its exclusion mask is then empty and the reference deterministic, md_util.c:5537-5560), on the water6 and tric6 frames."""
    out = {"script": np.array(DYN_SCRIPT)}
    w = np.load(os.path.join(HERE, "water6.npz")); t = np.load(os.path.join(HERE, "tric6.npz"))
    for tag, g, seed in (("w", w, "77"), ("t", t, "91")):
        gro, raw, o = os.path.join(tmp, tag + "d.gro"), os.path.join(tmp, tag + "d.raw"), os.path.join(tmp, tag + "d.out")
        F = g["frames"].shape[0]
        run(SYNTH, "water-gro", "6", seed, gro); refio.write_raw_traj(raw, g["frames"], g["cells"], g["cell_flags"])
        run(HARNESS, "eval", "--sys", gro, "--traj", f"raw:{raw}", "--script", DYN_SCRIPT, "--out", o, "--perframe", f"0:{F}", "--full", f"0:{F}")
        sub = {}; pack(sub, refio.read_refout(o), list(range(F)))
        for k, v in sub.items(): out[f"{tag}_{k}"] = v
    np.savez_compressed(os.path.join(HERE, "dyn6.npz"), **out)


def forms45(tmp):
    """The 45 statement forms of tests/test_emulated_library.py (PROBE_FORMS, one script) on the first 2 frames of water6 (w) and tric6 (t), each
    box's topology from the generator seed stored with it: per-frame bins / voxels and full values of every property, as pack() stores them."""
    from test_emulated_library import PROBE_FORMS
    script = " ".join(PROBE_FORMS); out = {"script": np.array(script)}; F = 2
    for tag, name, seed in (("w", "water6.npz", 77), ("t", "tric6.npz", 91)):
        g = np.load(os.path.join(HERE, name))
        gro, raw, o = os.path.join(tmp, tag + "f.gro"), os.path.join(tmp, tag + "f.raw"), os.path.join(tmp, tag + "f.out")
        run(SYNTH, "water-gro", "6", str(seed), gro); refio.write_raw_traj(raw, g["frames"][:F], g["cells"][:F], g["cell_flags"][:F])
        run(HARNESS, "eval", "--sys", gro, "--traj", f"raw:{raw}", "--script", script, "--out", o, "--perframe", f"0:{F}", "--full", f"0:{F}")
        sub = {}; pack(sub, refio.read_refout(o), list(range(F)))
        out.update({f"{tag}_{k}": v for k, v in sub.items()}); out[f"{tag}_seed"] = np.int32(seed)
    np.savez_compressed(os.path.join(HERE, "forms45.npz"), **out)


def shim_lowered(tmp):
    """integration/md_script_mdgpu.inl's lowering of a compiled md_script IR (oracle/_ref/shim_harness `lower`, the reference's own front-end) for the
    scripts of tests/test_integration_shim.py on the water6 topology (seed 77): the MDLOWER3 byte stream as written."""
    from test_integration_shim import SCRIPT, SCRIPT_NEW
    script = SCRIPT + " " + SCRIPT_NEW
    gro, o = os.path.join(tmp, "sl.gro"), os.path.join(tmp, "sl.bin")
    run(SYNTH, "water-gro", "6", "77", gro)
    run(SHIM, "lower", "--sys", gro, "--script", script, "--out", o)
    np.savez_compressed(os.path.join(HERE, "shim_lowered.npz"), script=np.array(script), lowered=np.fromfile(o, np.uint8))


def backbone(tmp):
    """phi / psi of every backbone segment per frame from the reference's md_util_backbone_angles_compute (harness mode `backbone`: the loop body of
    VIAMD's "Backbone Operations" task, src/viamd.cpp:488-520) on the 50 ala50 frames: the segments' five atoms (-1 rows: no angles) + angles[F][nseg][2]."""
    o = os.path.join(tmp, "bb.bin")
    run(HARNESS, "backbone", "--sys", "/root/reference/datasets/1ALA-500.pdb", "--traj", "sys", "--frames", "0:50", "--out", o)
    b = open(o, "rb").read(); assert b[:8] == b"MDBACKBN"
    F, ns = np.frombuffer(b, np.uint64, 2, 8); F, ns = int(F), int(ns)
    five = np.frombuffer(b, np.int32, ns * 5, 24).reshape(ns, 5).copy()
    ang = np.frombuffer(b, np.float32, F * ns * 2, 24 + ns * 20).reshape(F, ns, 2).copy()
    np.savez_compressed(os.path.join(HERE, "backbone.npz"), five=five, angles=ang)


def _write_gro(path, n, L):
    with open(path, "w") as f:
        f.write("synthetic\n%d\n" % n)
        for i in range(n):
            f.write("%5d%-5s%5s%5d%8.3f%8.3f%8.3f\n" % (i + 1, "ARG", "AR", i + 1, 0.1 * (i % 7), 0.1 * (i % 5), 0.1 * (i % 3)))
        f.write("%10.5f%10.5f%10.5f\n" % (L, L, L))


def xtc_cases(tmp):
    """XTC frames written by the reference's bundled xdrfile writer and decoded by the reference's md_xtc reader:
      water6    4 frames of the water6 trajectory (the common path: packed big + small integers, runs)
      tric6     4 frames with a triclinic cell that changes every frame (unit cell from the box matrix)
      water16   2 frames, 12 288 atoms (sha256 of the decoded arrays only)
      small5    5 atoms: stored uncompressed (natoms <= 9)
      wide12    12 atoms spread over ~5000 nm per axis: packed field wider than 64 bits
      huge12    12 atoms spread over ~20000 nm: per-axis integers (sizeint > 0xffffff branch)
      lowprec   water6 at precision 100 (different small-integer table positions)"""
    import hashlib
    out = {}

    def case(name, gro, raw, extra=(), hash_only=False):
        xtc = os.path.join(tmp, name + ".xtc"); dec = os.path.join(tmp, name + ".dec")
        run(HARNESS, "xtcwrite", "--sys", gro, "--traj", f"raw:{raw}", "--out", xtc, *extra)
        run(HARNESS, "dumptraj", "--sys", gro, "--traj", f"xtc:{xtc}", "--out", dec)
        fr, cells, flags = refio.read_raw_traj(dec)
        out[name + "__xtc"] = np.fromfile(xtc, np.uint8); out[name + "__cells"] = cells; out[name + "__flags"] = flags
        out[name + "__na"] = np.int32(fr.shape[2])
        if hash_only: out[name + "__sha"] = np.array([hashlib.sha256(np.ascontiguousarray(f).tobytes()).hexdigest() for f in fr])
        else: out[name + "__frames"] = fr

    gro, raw = os.path.join(tmp, "xw.gro"), os.path.join(tmp, "xw.raw")
    run(SYNTH, "water-gro", "6", "77", gro); run(SYNTH, "water-raw", "6", "77", "4", raw)
    case("water6", gro, raw); case("lowprec", gro, raw, ("--precision", "100"))
    g = np.load(os.path.join(HERE, "tric6.npz")); traw = os.path.join(tmp, "xt.raw")
    refio.write_raw_traj(traw, g["frames"], g["cells"], g["cell_flags"]); case("tric6", gro, traw)
    gro16, raw16 = os.path.join(tmp, "x16.gro"), os.path.join(tmp, "x16.raw")
    run(SYNTH, "water-gro", "16", "5", gro16); run(SYNTH, "water-raw", "16", "5", "2", raw16); case("water16", gro16, raw16, hash_only=True)
    rng = np.random.default_rng(99)
    for name, n, span in (("small5", 5, 30.0), ("wide12", 12, 5.0e4), ("huge12", 12, 2.0e5)):
        g2, r2 = os.path.join(tmp, name + ".gro"), os.path.join(tmp, name + ".raw"); _write_gro(g2, n, 3.0)
        fr = (rng.random((3, 3, n)) * span - span / 2).astype(np.float32)
        refio.write_raw_traj(r2, fr, np.tile([30.0, 0, 0, 30.0, 0, 30.0], (3, 1)), np.full(3, 29, np.uint32)); case(name, g2, r2)
        out[name + "__orig"] = fr   # what was written: the reference reader mis-decodes wide12 / huge12, the format's truth is the input
    np.savez_compressed(os.path.join(HERE, "xtc_cases.npz"), **out)


if __name__ == "__main__":
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "oracle"])
    only = sys.argv[1:]   # e.g. `python make_golden.py water32_full water12_avg` regenerates just those
    gens = dict(water6=water6, ala50=ala50, membrane6=membrane6, tric6=tric6, tric6_rmsd=tric6_rmsd, pairs6=pairs6, shapes=shapes, xtc_cases=xtc_cases,
                water32_full=water32_full, water12_avg=water12_avg, backbone=backbone, dyn6=dyn6, arrargs=arrargs, bigcut6=bigcut6, rdftrg6=rdftrg6,
                forms45=forms45, shim_lowered=shim_lowered)
    with tempfile.TemporaryDirectory() as tmp:
        for name, fn in gens.items():
            if not only or name in only: fn(tmp)
    for f in (n + ".npz" for n in gens if not only or n in only):
        print(f, os.path.getsize(os.path.join(HERE, f)), "bytes")
