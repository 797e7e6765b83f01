"""ramses_b200/output.py writes the reference's snapshot format: state -> reference file format -> reference reader -> reference
checker.  The reference's own reader and checker (tests/visu/visu_ramses.py of the reference: load_snapshot + check_solution)
were run on the snapshots these tests write by tests/golden/make_snapshot_golden.py, and what they returned is stored:

  golden/snapshot_golden.json  per snapshot: the SHA-256 of every file of output_NNNNN/ the reader was given; for the two long
                               runs also the sums check_solution computed and its verdict against the reference's golden file
  golden/snapshot_<name>.npz   the per-cell arrays and scalars load_snapshot returned (short runs)

Each test writes its snapshot again and requires the same bytes, so the reference reader would return the stored arrays; those
arrays are then compared with the run as the reader's live output was."""
import hashlib
import json
import os

import numpy as np

GOLD = os.path.join(os.path.dirname(__file__), "golden")
SNAPSHOT_GOLDEN = os.path.join(GOLD, "snapshot_golden.json")


def _write_from_run(r, tmp, iout, mhd=False):
    """the oracle AMR driver's tree / state (1-based arrays with an unused element 0) -> output_NNNNN/"""
    from ramses_b200.output import write_snapshot
    m = r.m
    nb = m.nboundary
    L = r.nlevelmax
    nvs = r.nvar
    return write_snapshot(
        str(tmp), iout, ndim=r.ndim, nvar=8 if mhd else r.nvar, levelmin=r.levelmin, nlevelmax=L, ngridmax=r.ngridmax,
        ncoarse=r.ncoarse, nxyz=(m.nx, m.ny, m.nz), coarse_min=(m.icoarse_min, m.jcoarse_min, m.kcoarse_min),
        coarse_max=(m.icoarse_max, m.jcoarse_max, m.kcoarse_max), boxlen=r.p.boxlen, gamma=(r.pm.gamma if mhd else r.p.gamma),
        smallr=r.p.smallr, son=r.son[1:], father=r.father[1:], nbor=r.nbor[:, 1:], xg=r.xg[:, 1:],
        active=[r.active[l] for l in range(1, L + 1)], boundary=[[r.bound[b][l] for l in range(1, L + 1)] for b in range(nb)],
        uold=r.uold.reshape(nvs, r.ncell), t=r.t, dtold=[r.dtold[l] for l in range(1, L + 1)],
        dtnew=[r.dtnew[l] for l in range(1, L + 1)], nstep=r.nstep, nstep_coarse=r.nstep_coarse, tout=r.tout, mhd=mhd)


# ---- the snapshots (also run by tests/golden/make_snapshot_golden.py) ------------------------------------------------------
def sod_run():
    from oracle.amr import AmrRun
    from test_oracle_golden import SOD
    r = AmrRun(1, 3, 10, (1, 1, 0, 0, 0, 0), 1.0, nsubcycle=[1, 1, 1, 2], nexpand=1, ngridmax=2000, riemann="hllc",
               slope_type=2, gamma=1.4, courant_factor=0.8, err_grad_d=0.05, err_grad_u=0.05, err_grad_p=0.05,
               interpol_type=2, interpol_var=0, regions=SOD, tout=[0.245])
    return r, r.run()


def orszag_short_run():
    from oracle.amr_mhd import MhdAmrRun2D
    r = MhdAmrRun2D(4, 6, 1.0, nsubcycle=[1], riemann="hlld", riemann2d="hlld", slope_type=2, gamma=1.6666667, courant_factor=0.8,
                    err_grad_p=0.1, interpol_type=2, tout=[0.1], nexpand=1, ngridmax=20000)
    return r, r.run()


def host_mirror_commons():
    """the product's host mirror (AmrCommons from ramses_b200.tree.build_nested_tree, three levels) with a linear state"""
    from ramses_b200.tree import build_nested_tree, fill_state
    a = build_nested_tree(3, 5, half_width=2)
    a.gamma = 1.4

    def fn(x, y, z):
        u = np.zeros((5, len(x)))
        u[0] = 1.0 + x + 2 * y + 4 * z
        u[1], u[2], u[3] = 0.1 * u[0], -0.2 * u[0], 0.3 * u[0]
        u[4] = 2.5 + 0.5 * u[0] * (0.01 + 0.04 + 0.09) + x * y
        return u
    for l in range(1, 6):
        fill_state(a, l, fn)
    return a


def write_host_mirror(a, outdir):
    from ramses_b200.output import snapshot_from_commons
    return snapshot_from_commons(a, str(outdir), 1, t=0.125, levelmin=3)


def file_hashes(snapdir):
    """SHA-256 of every file of an output_NNNNN/ directory"""
    return {f: hashlib.sha256(open(os.path.join(snapdir, f), "rb").read()).hexdigest() for f in sorted(os.listdir(snapdir))}


# ---- what the reference's reader and checker returned ----------------------------------------------------------------------
def _golden(name):
    return json.load(open(SNAPSHOT_GOLDEN))[name]


def _assert_reader_input(snapdir, name):
    """the snapshot holds the bytes the reference reader was given when the golden arrays were recorded"""
    assert file_hashes(snapdir) == _golden(name)["files"], f"{name}: the snapshot files differ from those the reference reader read"


def _reader_output(name):
    z = np.load(os.path.join(GOLD, "snapshot_%s.npz" % name))
    return {k: z[k] for k in z.files}


def _assert_checker_passed(name, ref_json):
    """check_solution's sums of the reference reader's data against the reference's golden file: its verdict, and its comparison
    (relative difference <= 3e-13 per variable, tests/visu/visu_ramses.py:497 of the reference) redone on the stored sums"""
    g = _golden(name)
    assert g["check_solution"] == "PASSED"
    ref = json.load(open(os.path.join(GOLD, ref_json)))
    sums = g["sums"]
    assert sorted(sums) == sorted(ref)
    for k, v in ref.items():
        s = sums[k]
        err = 0.0 if s == v == 0.0 else abs(s - v) / min(abs(s), abs(v))
        assert err <= 3.0e-13, (name, k, s, v, err)


def test_sod_tube_snapshot_through_reference_reader(orc, tmp_path):
    r, snap = sod_run()
    # the driver stops after the output step: the state at the output time is the current one
    _assert_reader_input(_write_from_run(r, tmp_path, 2), "sod_tube")
    _assert_checker_passed("sod_tube", "sod_tube_ref.json")   # the reference's own verdict on the reference's own golden file
    data = _reader_output("sod_tube")
    assert data["ncells"] == 142 and abs(data["time"] - snap["t"]) < 1e-14
    rows = snap["rows"]
    x = np.array([q[1][0] for q in rows])
    order_ref, order_ours = np.argsort(data["x"]), np.argsort(x)
    assert np.array_equal(np.sort(data["x"]), np.sort(x))
    assert np.array_equal(data["density"][order_ref], np.array([q[2] for q in rows])[order_ours])
    assert np.array_equal(data["pressure"][order_ref], np.array([q[4] for q in rows])[order_ours])


def test_orszag_tang_snapshot_through_reference_reader(orc, tmp_path):
    """a short NDIM=2 MHD AMR run: the eleven output fields survive the file format bit for bit"""
    r, snap = orszag_short_run()
    _assert_reader_input(_write_from_run(r, tmp_path, 2, mhd=True), "orszag_tang_short")
    data = _reader_output("orszag_tang_short")
    ours = snap["rows"]
    assert data["ncells"] == len(ours["level"])
    key_ref = np.lexsort((data["y"], data["x"]))
    key_our = np.lexsort((ours["y"], ours["x"]))
    for k in ("level", "x", "y", "dx", "density", "velocity_x", "velocity_y", "velocity_z", "pressure", "B_x_left", "B_y_left",
              "B_z_left", "B_x_right", "B_y_right", "B_z_right"):
        assert np.array_equal(np.asarray(data[k])[key_ref], np.asarray(ours[k])[key_our]), k


def test_implosion_and_orszag_tang_through_reference_checker(implosion_run, orszag_run, tmp_path):
    """the two long golden runs (session fixtures shared with test_oracle_golden.py): the final state in the reference's format
    is what the REFERENCE's check_solution compared with the REFERENCE's golden file -- PASSED for orszag-tang (all sums to
    2e-15) and for implosion (within its 3e-13 tolerance)."""
    r, _ = orszag_run
    d1 = tmp_path / "ot"
    d1.mkdir()
    _assert_reader_input(_write_from_run(r, d1, 2, mhd=True), "orszag_tang")
    _assert_checker_passed("orszag_tang", "orszag_tang_ref.json")
    r, _ = implosion_run
    d2 = tmp_path / "impl"
    d2.mkdir()
    _assert_reader_input(_write_from_run(r, d2, 2), "implosion")
    _assert_checker_passed("implosion", "implosion_ref.json")


def test_snapshot_from_host_mirror_nested_tree(tmp_path):
    """the product's host mirror (AmrCommons from ramses_b200.tree.build_nested_tree, three levels) -> snapshot -> reference
    reader: every leaf cell comes back at its position with its value."""
    a = host_mirror_commons()
    _assert_reader_input(write_host_mirror(a, tmp_path), "host_mirror")
    data = _reader_output("host_mirror")
    nleaf = sum(int((a.son[a.ncoarse + ind * a.ngridmax + a.active[l].astype(np.int64) - 1] == 0).sum())
                for l in range(1, 6) for ind in range(8))
    assert data["ncells"] == nleaf and data["time"] == 0.125
    x, y, z = data["x"], data["y"], data["z"]
    assert np.array_equal(data["density"], 1.0 + x + 2 * y + 4 * z)
    assert np.allclose(data["velocity_y"], -0.2, rtol=0, atol=1e-16)
    assert np.allclose(data["pressure"], 0.4 * (2.5 + x * y), rtol=1e-14, atol=0)
    assert set(np.unique(data["level"])) == {3.0, 4.0, 5.0}


def test_snapshot_restart_round_trip(orc, tmp_path):
    """write_snapshot -> read_snapshot (the restart side, amr/init_amr.f90 + hydro/init_hydro.f90:57-250): the tree arrays and the
    lists come back identically, the conserved state to round-off (the file holds primitive variables, like the reference's own
    restart), and a second write of the restored state reproduces the amr file byte for byte."""
    from oracle.amr import AmrRun
    from ramses_b200.output import read_snapshot, write_snapshot
    from test_oracle_golden import SOD
    r = AmrRun(1, 3, 8, (1, 1, 0, 0, 0, 0), 1.0, nsubcycle=[1, 1, 1, 2], nexpand=1, ngridmax=500, riemann="hllc", slope_type=2,
               gamma=1.4, courant_factor=0.8, err_grad_d=0.05, err_grad_u=0.05, err_grad_p=0.05, interpol_type=2, interpol_var=0,
               regions=SOD, tout=[0.1])
    r.run()
    d1 = tmp_path / "a"
    d1.mkdir()
    _write_from_run(r, d1, 3)
    s = read_snapshot(str(d1), 3, smallr=r.p.smallr)
    assert s["t"] == r.t and s["nstep"] == r.nstep and s["ndim"] == 1 and s["nboundary"] == 2
    used = np.concatenate([np.asarray(r.active[l], dtype=np.int64) for l in range(1, 9)] +
                          [np.asarray(r.bound[b][l], dtype=np.int64) for b in range(2) for l in range(1, 9)])
    assert np.array_equal(s["son"][:r.ncoarse], r.son[1:r.ncoarse + 1])
    for ind in range(2):
        c = r.ncoarse + ind * r.ngridmax + used
        assert np.array_equal(s["son"][c - 1], r.son[c])
    assert np.array_equal(s["father"][used - 1], r.father[used]) and np.array_equal(s["nbor"][:, used - 1], r.nbor[:, used])
    assert np.array_equal(s["xg"][:, used - 1], r.xg[:, used])
    for l in range(1, 9):
        assert np.array_equal(s["active"][l - 1], np.asarray(r.active[l], dtype=np.int32))
    U = r.uold.reshape(3, r.ncell)
    act = np.concatenate([np.asarray(r.active[l], dtype=np.int64) for l in range(1, 9)])
    for ind in range(2):
        c = r.ncoarse + ind * r.ngridmax + act - 1
        assert np.array_equal(s["uold"][0, c], U[0, c])
        assert np.allclose(s["uold"][1:, c], U[1:, c], rtol=4e-16, atol=1e-300)
    d2 = tmp_path / "b"
    d2.mkdir()
    write_snapshot(str(d2), 3, ndim=1, nvar=3, levelmin=3, nlevelmax=8, ngridmax=s["ngridmax"], ncoarse=s["ncoarse"], nxyz=s["nxyz"],
                   coarse_min=(1, 0, 0), coarse_max=(1, 0, 0), boxlen=s["boxlen"], gamma=s["gamma"], smallr=r.p.smallr, son=s["son"],
                   father=s["father"], nbor=s["nbor"], xg=s["xg"], active=s["active"], boundary=s["boundary"], uold=s["uold"],
                   t=s["t"], dtold=s["dtold"], dtnew=s["dtnew"], nstep=s["nstep"], nstep_coarse=s["nstep_coarse"], tout=s["tout"],
                   flag1=s["flag1"], cpu_map=s["cpu_map"])
    f = "output_00003/amr_00003.out00001"
    assert open(d1 / f, "rb").read() == open(d2 / f, "rb").read()
