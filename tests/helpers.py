"""Shared helpers for the parity tests (TEST INFRASTRUCTURE)."""
from __future__ import annotations

import os

import numpy as np

import oracle_lib as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def load_golden(name):
    return np.load(os.path.join(ROOT, "tests", "golden", name), allow_pickle=False)


def cell_from_row(row, flags):
    return O.UnitCell.from_params(row[0], row[1], row[2], row[3], row[4], row[5], int(flags))


def dense_from_sparse(idx, val, n=128 ** 3):
    v = np.zeros(n, np.float32); v[idx] = val; return v


def dense_from_mask(mask, val, n=128 ** 3):
    """volume stored as the np.packbits mask of its non-zero voxels + their values in index order"""
    v = np.zeros(n, np.float32); v[np.unpackbits(mask, count=n).astype(bool)] = val; return v


def golden_system(g):
    """(mass, z, names, comp_off, conn_off, conn_idx) -> selections by element"""
    z = g["z"].astype(int)
    return dict(mass=g["mass"], z=z, names=[str(s) for s in g["names"]], comp_off=g["comp_off"].astype(np.int64),
                conn_off=g["conn_off"], conn_idx=g["conn_idx"])


def sel_element(sysd, znum):
    return np.nonzero(sysd["z"] == znum)[0].astype(np.int32)


def vb_system(sysd):
    import viamd_b200 as vb
    sym = {1: "H", 6: "C", 7: "N", 8: "O", 16: "S"}
    return vb.System(len(sysd["mass"]), sysd["mass"], sysd["conn_off"], sysd["conn_idx"],
                     element=[sym.get(int(z), "X") for z in sysd["z"]], name=sysd["names"],
                     resname=["RES"] * (len(sysd["comp_off"]) - 1), res_atom_offset=sysd["comp_off"])


def vb_cell(row, flags):
    import viamd_b200 as vb
    return vb.UnitCell(float(row[0]), float(row[1]), float(row[2]), float(row[3]), float(row[4]), float(row[5]), int(flags))
