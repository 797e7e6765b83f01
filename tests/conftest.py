import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with `-m gpu`)")


@pytest.fixture(scope="session")
def orc():
    from oracle import orc as _orc
    _orc.build()
    return _orc


# ---- the two long golden runs, shared by test_oracle_golden.py (sums) and test_output_format.py (reference reader + checker) ----
# tests/hydro/implosion/implosion.nml and tests/mhd/orszag-tang/orszag-tang.nml
IMPL = [dict(type="square", x_center=0.5, y_center=0.5, length_x=1.0, length_y=1.0, exp_region=10, d=1.0, p=1.0),
        dict(type="square", x_center=0.0, y_center=0.0, length_x=1.0, length_y=1.0, exp_region=1, d=0.125, p=0.4)]
# BOUNDARY_PARAMS of implosion.nml:17-24 after hydro/read_hydro_params.f90:316-407: (boundary_type, i-, j-, k-range)
IMPL_BOUND = [(1, (0, 0), (1, 1), (0, 0)), (2, (2, 2), (1, 1), (0, 0)), (4, (0, 2), (2, 2), (0, 0)), (3, (0, 2), (0, 0), (0, 0))]


def make_implosion_run():
    from oracle.amr import FastAmrRun
    r = FastAmrRun(2, 5, 8, (1, 1, 1, 1, 0, 0), 1.0, nsubcycle=[2] * 10, nexpand=[4], ngridmax=100000, riemann="hllc",
                   slope_type=2, gamma=1.4, courant_factor=0.8, err_grad_d=0.05, err_grad_u=0.05, err_grad_p=0.05,
                   interpol_type=2, interpol_var=0, regions=IMPL, tout=[0.0, 5.0], bound_regions=IMPL_BOUND)
    return r, r.run()


def make_orszag_run():
    from oracle.amr_mhd import MhdAmrRun2D
    r = MhdAmrRun2D(5, 9, 1.0, nsubcycle=[1], riemann="hlld", riemann2d="hlld", slope_type=2, gamma=1.6666667,
                    courant_factor=0.8, err_grad_p=0.1, interpol_type=2, tout=[0.5], nexpand=1, ngridmax=100000)
    return r, r.run()


@pytest.fixture(scope="session")
def implosion_run(orc):
    return make_implosion_run()


@pytest.fixture(scope="session")
def orszag_run(orc):
    return make_orszag_run()
