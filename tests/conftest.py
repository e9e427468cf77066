import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")

from oracle.oracle import stored_default_plane as default_plane  # noqa: E402


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def O():
    """the CPU checkers (oracle/): plain-C restatement + the reference's own object code"""
    from oracle import oracle
    oracle.build()
    return oracle


@pytest.fixture(scope="session")
def dfb():
    """the product: ctypes mirror over libdfb200.so (hard error if the library is not built)"""
    import _dfb_import  # noqa: F401
    import digital_filtering_b200
    digital_filtering_b200.lib()
    return digital_filtering_b200


@pytest.fixture(scope="session")
def W():
    import _dfb_import  # noqa: F401
    from digital_filtering_b200 import workloads
    return workloads


@pytest.fixture(scope="session")
def default_data(tmp_path_factory):
    """Input files in the reference's formats for its default plane, written from the stored tables (oracle.stored_default_plane()) into
    the reference's layout: <dir>/files/RST.dat, <dir>/line.dat, and <dir>/run as the working directory from which its
    relative paths resolve (df.cpp:16,224).  RST.dat samples 330 of the 510 rows and ends at the last one, so the setup keeps
    the same 510 rows; the friction velocity the setup derives from line.dat (df.cpp:547-549) is the one the columns are
    scaled by, so the row tables come back up to interpolation and rounding.  Returns the directory."""
    import numpy as np
    P = default_plane()
    d = tmp_path_factory.mktemp("default_data")
    os.makedirs(d / "files")
    os.makedirs(d / "run")
    yc, (R11, R21, R22, R33, Us, Ts, rhos, _) = P["yc"], P["rows"]
    line = np.zeros((len(yc), 10))
    line[:, 1], line[:, 4], line[:, 5], line[:, 8], line[:, 9] = yc, rhos, Us, Ts, rhos * 287.0 * Ts
    u_tau = np.sqrt(7.1212e-6 * (Us[1] - Us[0]) / (yc[1] - yc[0]) / rhos[0])
    i = np.unique(np.linspace(0, len(yc) - 1, 330).round().astype(int))
    rst = np.stack([np.arange(len(i)), yc[i] / P["d_i"], np.sqrt(R11[i]) / u_tau, np.sqrt(R22[i]) / u_tau, np.sqrt(R33[i]) / u_tau,
                    R21[i] / u_tau ** 2], axis=1)
    for path, a, names in ((d / "files" / "RST.dat", rst, "n y/d u' v' w' uv"), (d / "line.dat", line, "i y 2 3 rho u 6 7 T p")):
        with open(path, "w") as fh:
            fh.write("VARIABLES = %s\nZONE T=default i=%d\n" % (" ".join('"%s"' % n for n in names.split()), len(a)))
            fh.writelines(" ".join(repr(float(x)) for x in r) + "\n" for r in a)
    return d


def normwise_close(got, ref, tol=1e-12):
    """north_star's fp64 gate, in the normwise form SURVEY section 7 shows is the attainable one:
    |got - ref| <= tol * max(|ref|, rms(ref)) elementwise.  Returns (ok, worst ratio)."""
    import numpy as np
    got = np.asarray(got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    rms = float(np.sqrt(np.mean(ref * ref)))
    scale = np.maximum(np.abs(ref), rms if rms > 0 else 1.0)
    ratio = float(np.max(np.abs(got - ref) / scale)) if ref.size else 0.0
    return ratio <= tol, ratio
