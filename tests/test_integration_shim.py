"""The drop-in boundary, end to end: the reference's own md_script.c + integration/md_script_mdgpu.inl compiled as one translation
unit (oracle/_ref/shim_harness, which `make -C oracle ref` builds where the reference sources are present; the tests that run it skip elsewhere).
 - CPU: the shim's lowering of a compiled md_script IR, stored in tests/golden/shim_lowered.npz, equals viamd_b200.script's lowering (same ops,
   index lists, cutoffs).
 - GPU: md_script_eval_frame_range (reference CPU path) vs md_script_gpu_eval_frame_range (libmdgpu) on the same script."""
import json
import os
import struct
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHIM = os.path.join(ROOT, "oracle", "_ref", "shim_harness")
TOOL = os.path.join(ROOT, "oracle", "build", "synth_tool")

SCRIPT = ("r = rdf(element('O'), element('O'), 6.0); v = sdf(residue(1:20), element('O'), 5.0); dz = density_z(element('O')); "
          "d = distance(1,10); rr = rdf(element('O'), element('H'), 1.5:6.0); a = angle(1,2,3); t = dihedral(1,4,7,10); "
          "rc = rdf(residue(1:20), element('O'), 5.0);")
# forms added after the last GPU run: lowered identically by the shim and the Python mirror (CPU check); their GPU tests are in test_zz_gpu_new_ops.py
SCRIPT_NEW = ("rm = rmsd(residue(1:10)); dp = distance_pair(atom(1:5), atom(20:30)); c = com(residue(1)); ci = com(5); pl = plane(atom(1:30)); "
              "cw = count(within(4.0, residue(1))); dmn = distance_min(residue(1), atom(100:648)); dc = distance(residue(1), residue(5)); "
              "rw = rdf(within(4.0, residue(1)), element('O'), 6.0); cwr = count(within(2.5:5.0, residue(1))); rwr = rdf(within(3.0:6.0, residue(2)), element('O'), 1.0:6.5); "
              "anc = angle(2,1,3) in residue(1:10); ddc = distance(1,3) in residue(:); cz = coord_z(atom(5:40)); dpg = distance_pair(residue(1:4), residue(10:15)); cwg = count(within(6.0, residue(1:5))); cwo = count(element('O') and within(4.0, residue(1))); rwo = rdf(element('H') and within(5.0, residue(2)), element('O'), 6.0); dcm = distance(com(atom(1:30)), 200); acm = angle(com(residue(1)), com(residue(2)), residue(3)); "
              "rwt = rdf(element('O'), within(4.0, residue(1)), 6.0); rww = rdf(within(4.0, residue(1)), within(5.0, residue(2)), 6.0); vw = sdf(residue(1:20), within(6.0, residue(1:5)), 5.0); "
              "dzw = density_z(within(5.0, residue(1))); dw = distance(within(4.0, residue(1)), 200); cmw = com(within(4.0, residue(1))); dmw = distance_min(within(3.5, residue(1)), residue(30)); "
              "rwo2 = rdf(element('O') and within(5.0, residue(2)), element('H') and within(6.0, residue(3)), 5.0); aw = angle(within(2.5:5.0, residue(4)), 10, residue(7)); "
              "cc = contact_count(residue(1:5), residue(10:40), 4.0); cc2 = contact_count(residue(3:20), element('O') and residue(50:216), 3.5); "
              # an ARRAY of selections as one position argument: centre of the selections' centres for angle / dihedral / com, the union for distance (FLAG_FLATTEN)
              "aar = angle(residue(1:2), residue(5:7), 30); har = dihedral(residue(1:2), residue(3:4), residue(5:6), residue(7:9)); car = com(residue(1:6)); "
              "dar = distance(residue(1:4), residue(10)); ddr = distance(com(residue(1:4)), residue(50:52)); acr = angle(com(residue(1:3)), 100, residue(20)); "
              # an ARRAY of selections as rdf target: one centre of mass per selection is the target point
              "rta = rdf(residue(1:20), residue(10:30), 5.0); rtb = rdf(element('O'), residue(10:60), 6.0); "
              "dmg = distance_min(residue(1:4), residue(10:30)); dxg = distance_max(residue(3:5), element('O')); cxg = coord_x(residue(1:5)); plg = plane(residue(1:10)); "
              # selections inside `in` contexts (the shim evaluates context-relative arguments with the reference's own evaluator)
              "dctx = distance(element('O'), element('H')) in residue(1:10); ectx = distance(element('O'), atom(2:3)) in residue(2:5); hctx = dihedral(1, element('O'), atom(2:3), 3) in residue(:);")


# forms only the shim lowers (the Python mirror rejects them): arguments that are relative to the context — residue(1) inside `in residue(2:4)` is the
# context's own first residue, `element('O') and atom(1:2)` counts atoms from the context's first atom. The shim evaluates them per context with
# mdlib's own evaluate_node, as evaluate_context does.
SCRIPT_SHIM_ONLY = ("xr = distance(residue(1), 2) in residue(2:4); ya = distance(element('O') and atom(1:2), 3) in residue(2:4); "
                    "dcx = distance(com(element('H')), 1) in residue(10:20);")


def _need():
    if not os.path.exists(SHIM):
        pytest.skip("oracle/_ref/shim_harness not built (needs the reference sources: make -C oracle ref)")
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "oracle"])


def _read_lowered(b):
    assert b[:8] == b"MDLOWER3"
    n, = struct.unpack_from("<Q", b, 8); off = 16; out = []
    for _ in range(n):
        name = b[off:off + 64].split(b"\0")[0].decode(); off += 64
        op, ns, ss = struct.unpack_from("<3Q", b, off); off += 24
        cmin, cmax = struct.unpack_from("<2f", b, off); off += 8
        lists = []
        for _k in range(4):
            c, = struct.unpack_from("<Q", b, off); off += 8
            lists.append(np.frombuffer(b, np.int32, c, off).copy()); off += 4 * c
        dyn = {}
        for k in range(4):
            rmin, rmax = struct.unpack_from("<2f", b, off); off += 8
            has_and, c = struct.unpack_from("<2Q", b, off); off += 16
            a = np.frombuffer(b, np.int32, c, off).copy(); off += 4 * c
            if rmax > 0: dyn[k] = (rmin, rmax, a if has_and else None)
        nb, = struct.unpack_from("<Q", b, off); off += 8
        eoff = None
        if nb: eoff = np.frombuffer(b, np.uint32, nb + 1, off).copy(); off += 4 * (nb + 1)
        parts = {}
        for k in range(4):
            c, = struct.unpack_from("<Q", b, off); off += 8
            if c: parts[k] = np.frombuffer(b, np.uint32, c + 1, off).copy(); off += 4 * (c + 1)
        out.append(dict(name=name, op=op, ns=ns, ss=ss, cmin=cmin, cmax=cmax, idx=lists, dyn=dyn, eoff=eoff, parts=parts))
    return out


def test_shim_lowering_matches_python_lowering():
    """The shim's lowering of the md_script IR (stored in tests/golden/shim_lowered.npz by tests/golden/make_golden.py, which runs
    oracle/_ref/shim_harness `lower` on the water6 topology) equals viamd_b200.script's lowering of the same script."""
    import viamd_b200 as vb
    from helpers import load_golden
    g = load_golden("shim_lowered.npz"); script = SCRIPT + " " + SCRIPT_NEW
    assert str(g["script"]) == script, "shim_lowered.npz is stale: regenerate it with make_golden.py shim_lowered"
    low = _read_lowered(g["lowered"].tobytes())
    props = vb.compile_script(script, vb.water_system(6))
    assert [p["name"] for p in low] == [p.name for p in props]
    for a, b in zip(low, props):
        assert a["op"] == b.op and a["cmin"] == np.float32(b.cutoff_min) and a["cmax"] == np.float32(b.cutoff_max), a["name"]
        if b.op == vb.OP_SDF:
            assert a["ns"] == b.num_structures and a["ss"] == b.structure_size
        if b.op == vb.OP_RDF:   # array-of-selections reference -> centre-of-mass groups
            assert a["ns"] == b.num_structures
        for k, arr in enumerate(b.idx):
            if b.op == vb.OP_RDF and b.ref_within > 0 and k == 2: continue   # the round-1 spelling keeps the AND mask in idx[2]; compared through dyn below
            assert np.array_equal(a["idx"][k], arr), (a["name"], k)
        want = dict(b.dyn)
        if b.op == vb.OP_RDF and b.ref_within > 0: want[0] = (b.ref_within_min, b.ref_within, b.idx[2] if b.com_args & 1 else None)
        assert a["dyn"].keys() == want.keys(), a["name"]
        for k, (rmin, rmax, cand) in want.items():
            assert a["dyn"][k][0] == np.float32(rmin) and a["dyn"][k][1] == np.float32(rmax) and ((cand is None) == (a["dyn"][k][2] is None)), (a["name"], k)
            if cand is not None: assert np.array_equal(a["dyn"][k][2], cand), (a["name"], k)
        if b.op == vb.OP_CONTACT_COUNT: assert np.array_equal(a["eoff"], b.structure_offsets_b) and a["ns"] == b.num_structures
        if b.op in (vb.OP_RDF, vb.OP_DISTANCE_MIN, vb.OP_DISTANCE_MAX, vb.OP_DISTANCE_PAIR):
            assert (a["eoff"] is None) == (b.structure_offsets_b is None) and (a["eoff"] is None or np.array_equal(a["eoff"], b.structure_offsets_b)), a["name"]
        if b.op in (vb.OP_DISTANCE_MIN, vb.OP_DISTANCE_MAX, vb.OP_DISTANCE_PAIR, vb.OP_COORD_X, vb.OP_PLANE): assert a["ns"] == b.num_structures, a["name"]
        assert a["parts"].keys() == b.arg_offsets.keys(), a["name"]
        for k, o in b.arg_offsets.items(): assert np.array_equal(a["parts"][k], o), (a["name"], k)


@pytest.mark.gpu
def test_md_script_api_cpu_vs_gpu_through_the_shim(tmp_path):
    _need()
    gro = str(tmp_path / "w8.gro")
    subprocess.check_call([TOOL, "water-gro", "8", "1008", gro])
    script = "r = rdf(element('O'), element('O'), 10.0); v = sdf(residue(1:50), element('O'), 6.0); dz = density_z(element('O')); d = distance(1,10); rc = rdf(residue(1:50), element('O'), 6.0);"
    p = subprocess.run([SHIM, "eval", "--sys", gro, "--traj", "synthwater:8:1008:12", "--script", script], capture_output=True, text=True)
    line = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert line, p.stdout + p.stderr
    res = json.loads(line[-1])
    assert p.returncode == 0 and res["parity"] is True, res
    assert all(q["out_of_tol"] == 0 and q["frame_mask_equal"] for q in res["properties"])


def test_md_script_api_through_the_shim_against_the_emulated_library(tmp_path):
    """The drop-in boundary on the CPU: the reference's own md_script.c + the shim, with the library behind the C ABI replaced by its emulated
    build (tests/emul: same sources, kernels run by host threads). md_script_eval_frame_range (reference CPU path) vs
    md_script_gpu_eval_frame_range on one script that holds the GPU-validated ops and every op added since (rmsd, distance_pair, com, plane,
    count(within())): values within tolerance (the new temporals: equal), frame masks equal. The binary finds `libmdgpu.so` through
    LD_LIBRARY_PATH, which the loader searches before the binary's RUNPATH."""
    _need()
    import shutil
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tests", "emul"))
    import build_emul
    libdir = tmp_path / "lib"; libdir.mkdir(); shutil.copy(build_emul.build_library(), str(libdir / "libmdgpu.so"))
    gro = str(tmp_path / "w6.gro")
    subprocess.check_call([TOOL, "water-gro", "6", "1008", gro])
    script = ("r = rdf(element('O'), element('O'), 6.0); d = distance(1,10); rc = rdf(residue(1:20), element('O'), 5.0); v = sdf(residue(1:20), element('O'), 5.0); "
              "dz = density_z(element('O')); " + SCRIPT_NEW + " " + SCRIPT_SHIM_ONLY)
    env = dict(os.environ, LD_LIBRARY_PATH=str(libdir))
    p = subprocess.run([SHIM, "eval", "--sys", gro, "--traj", "synthwater:6:1008:5", "--script", script], capture_output=True, text=True, env=env)
    line = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert line, p.stdout + p.stderr
    res = json.loads(line[-1])
    assert p.returncode == 0 and res["parity"] is True, res
    assert all(q["out_of_tol"] == 0 and q["frame_mask_equal"] for q in res["properties"])
    exact = {q["name"]: q["max_abs"] for q in res["properties"]}
    assert all(exact[k] == 0 for k in ("d", "rm", "dp", "c", "ci", "pl", "cw", "dmn", "dc", "v", "xr", "ya", "dcx", "dctx", "ectx", "car", "dar", "ddr", "dmg", "cxg", "plg")), exact



DROPIN_SCRIPT = "r = rdf(element('O'), element('O'), 6.0); d = distance(1,10); dz = density_z(element('O')); dp = distance_pair(atom(1:5), atom(20:30)); v = sdf(residue(1:20), element('O'), 5.0);"


def _run_dropin(args, env=None):
    p = subprocess.run([SHIM, "dropin", *args], capture_output=True, text=True, env=env)
    line = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert line, p.stdout + p.stderr
    return p.returncode, json.loads(line[-1])


def test_zero_edit_dropin_viamd_call_pattern_against_the_emulated_library(tmp_path):
    """integration/md_script_mdgpu.c = md_script_mdgpu_pre.h + the UNMODIFIED md_script.c + md_script_mdgpu.inl: the public
    md_script_eval_frame_range IS the dispatcher. The harness drives it the way VIAMD does (src/main.cpp:993-997 via task_system.cpp:73-87,
    à la mdlib/unittest/test_script.c:1352-1417): 4 threads pull disjoint 1-frame ranges on ONE eval while the main thread polls the frame
    mask; then md_script_eval_interrupt mid-run, md_script_eval_clear_data, a full re-evaluation, md_script_eval_free. Results equal the
    reference's own evaluation (`__cpu` symbols of the same TU); partial frame masks were visible while it ran. CPU: emulated library."""
    _need()
    import shutil
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tests", "emul"))
    import build_emul
    libdir = tmp_path / "lib"; libdir.mkdir(); shutil.copy(build_emul.build_library(), str(libdir / "libmdgpu.so"))
    gro = str(tmp_path / "w6.gro"); subprocess.check_call([TOOL, "water-gro", "6", "1008", gro])
    rc, res = _run_dropin(["--sys", gro, "--traj", "synthwater:6:1008:6", "--script", DROPIN_SCRIPT.split(" v = ")[0], "--threads", "4", "--chunk", "1", "--interrupt-at", "2"],
                          env=dict(os.environ, LD_LIBRARY_PATH=str(libdir)))
    assert rc == 0 and res["parity"] is True, res
    assert res["frames_done"] == 6 and res["partial_mask_views"] >= 2 and res["frames_done_at_interrupt"] < 6 and res["frames_done_after_restart"] == 6
    exact = {q["name"]: q["max_abs"] for q in res["properties"]}
    assert exact["d"] == 0 and exact["dp"] == 0 and all(q["out_of_tol"] == 0 and q["min_max_equal"] for q in res["properties"] + res["after_restart"])


@pytest.mark.gpu
def test_zero_edit_dropin_viamd_call_pattern_on_the_gpu(tmp_path):
    """The same on the B200 with libmdgpu.so itself: 8 threads x enkiTS-sized ranges over 192 frames of a 1536-atom box, interrupt, restart."""
    _need()
    gro = str(tmp_path / "w8.gro"); subprocess.check_call([TOOL, "water-gro", "8", "1008", gro])
    rc, res = _run_dropin(["--sys", gro, "--traj", "synthwater:8:1008:192", "--script", DROPIN_SCRIPT, "--threads", "8", "--interrupt-at", "40"])
    assert rc == 0 and res["parity"] is True, res
    assert res["frames_done"] == 192 and res["frames_done_after_restart"] == 192 and res["frames_done_at_interrupt"] <= 192
    assert all(q["out_of_tol"] == 0 and q["min_max_equal"] for q in res["properties"] + res["after_restart"])
    rc, res = _run_dropin(["--sys", gro, "--traj", "synthwater:8:1008:64", "--script", DROPIN_SCRIPT, "--threads", "1", "--chunk", "64"])   # one call over the whole range
    assert rc == 0 and res["parity"] is True and res["partial_mask_views"] >= 0, res
