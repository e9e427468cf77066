"""Per-cell profile tables for the tests of dfb_set_profiles: three boundary layers of different thickness on spanwise column bands, the
row tables broadcast along the span, and the epilogue's constants restated in numpy with the library's expressions and roundings."""
import numpy as np

import _dfb_import  # noqa: F401
from digital_filtering_b200 import workloads as W

THICKNESS = (0.6, 1.0, 1.8)          # boundary-layer thickness of bands A, B, C over the plane's own


def band_rows(plane):
    """the [8][Ny] row tables A, B, C: the plane's synthetic boundary layer at each thickness"""
    yc = np.asarray(plane["yc"])
    yc = yc[:, 0] if yc.ndim == 2 else yc                  # per-cell geometry: the rows follow column 0, as the library's do
    return [W.synthetic_rows(yc, plane["d_i"] * t, plane.get("U_e", W.U_E)) for t in THICKNESS]


def band_edges(Nz):
    """columns [0, a), [a, b), [b, Nz) of bands A, B, C"""
    return (0, Nz // 5, (3 * Nz) // 5, Nz)


def band_cells(rows_abc, Nz):
    """[8][Ny][Nz]: band i's columns take row table i"""
    e = band_edges(Nz)
    Ny = rows_abc[0].shape[1]
    cells = np.empty((8, Ny, Nz))
    for i, r in enumerate(rows_abc):
        cells[:, :, e[i]:e[i + 1]] = np.asarray(r)[:, :, None]
    return cells


def broadcast(rows, Nz):
    return np.repeat(np.asarray(rows, dtype=np.float64)[:, :, None], Nz, axis=2)


def consts(cells):
    """[7][...] epilogue constants: sqrt(R11), b, sqrt(R22 - b^2), sqrt(R33), -0.5 (1.4 - 1) Ms Ms / Us (left to right), Ts, rhos"""
    R11, R21, R22, R33, Us, Ts, rhos, Ms = cells
    with np.errstate(divide="ignore", invalid="ignore"):
        b = np.where(R11 < 1e-10, 0.0, R21 / np.sqrt(R11))
        return np.stack([np.sqrt(R11), b, np.sqrt(R22 - b * b), np.sqrt(R33), -0.5 * (1.4 - 1) * Ms * Ms / Us, Ts, rhos])
