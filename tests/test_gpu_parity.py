"""GPU parity tests proper: the CUDA path, called through the C-ABI, against the CPU oracle on the same
seeded inputs.  Bit-exact wherever libm `pow` is not involved (every solver except 'exact')."""
import numpy as np
import pytest

from helpers import Case, SEDOV3D_REGIONS, SEDOV1D_REGIONS, SOD_REGIONS, smooth_state, max_rel_err

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gpu():
    from ramses_b200 import lib
    lib.load()
    return lib


def run_level0(case, dt):
    from ramses_b200.hydro import HydroGPU
    a = case.amr_commons()
    h = HydroGPU(a)
    h.bind_level(case.level)
    a.dtnew[case.level] = dt
    a.unew[:, :] = a.uold          # state right after set_unew
    h.godunov_fine(case.level)
    info = h.level_info(case.level)
    h.finalize()
    return a.unew.copy(), info


@pytest.mark.parametrize("riemann", ["llf", "hllc", "hll", "acoustic", "exact"])
@pytest.mark.parametrize("order", [0, 2])
def test_godunov_fine_3d_smooth_bitwise(gpu, riemann, order):
    c = Case(3, 5, riemann=riemann, slope_type=1, order=order, seed=7)
    c.init_dense(smooth_state(3, 32))
    dt, _ = c.oracle_courant()
    ref = c.oracle_godunov(dt).reshape(c.nvar, -1)
    got, info = run_level0(c, dt)
    assert info.dense == 1
    idx = c.active_cells()
    if riemann == "exact":
        assert max_rel_err(got[:, idx], ref[:, idx]) <= 1e-12   # libm pow vs CUDA pow
    else:
        assert np.array_equal(got[:, idx], ref[:, idx])


@pytest.mark.parametrize("slope_type", [0, 1, 2, 3, 7, 8])
def test_godunov_fine_3d_slopes_bitwise(gpu, slope_type):
    c = Case(3, 4, riemann="hllc", slope_type=slope_type, order=2, seed=3)
    c.init_dense(smooth_state(3, 16))
    dt, _ = c.oracle_courant()
    ref = c.oracle_godunov(dt).reshape(c.nvar, -1)
    got, _ = run_level0(c, dt)
    idx = c.active_cells()
    assert np.array_equal(got[:, idx], ref[:, idx])


@pytest.mark.parametrize("riemann", ["llf", "hllc", "exact"])
def test_sedov3d_steps(gpu, riemann):
    """sedov3d (BASELINE config 2 at reduced size): 10 fused steps vs the oracle, conserved state <= 1e-12."""
    from ramses_b200.hydro import HydroGPU
    c = Case(3, 5, riemann=riemann, slope_type=1, boxlen=0.5)
    c.init_regions(SEDOV3D_REGIONS)
    ref, dts_ref = c.oracle_steps(10)
    a = c.amr_commons()
    h = HydroGPU(a)
    h.bind_level(c.level)
    h.upload_state(c.level)
    dts, sums = h.level_steps(c.level, 10)
    h.download_state(c.level)
    h.finalize()
    idx = c.active_cells()
    ref = ref.reshape(c.nvar, -1)
    if riemann == "exact":
        assert np.allclose(dts, dts_ref, rtol=1e-12, atol=0)
        assert max_rel_err(a.uold[:, idx], ref[:, idx]) <= 1e-12
    else:
        assert np.array_equal(dts, dts_ref)
        assert np.array_equal(a.uold[:, idx], ref[:, idx])
    # conservation to round-off on the periodic box
    d0 = c.dense()
    d1 = c.dense(a.uold.reshape(-1))
    assert abs(d1[0].sum() - d0[0].sum()) <= 1e-13 * abs(d0[0].sum())
    assert abs(d1[4].sum() - d0[4].sum()) <= 1e-12 * abs(d0[4].sum())


@pytest.mark.parametrize("ndim,level,regions", [(1, 7, SEDOV1D_REGIONS), (1, 8, SOD_REGIONS)])
@pytest.mark.parametrize("riemann,slope_type", [("hllc", 2), ("llf", 1), ("exact", 2), ("hll", 7), ("acoustic", 8)])
def test_1d_reflexive(gpu, ndim, level, regions, riemann, slope_type):
    """BASELINE config 1 (sedov1d, levelmin=levelmax=7, reflexive walls) and the Sod tube of tube1d.nml."""
    from ramses_b200.hydro import HydroGPU
    c = Case(ndim, level, riemann=riemann, slope_type=slope_type, bound=(1, 1, 0, 0, 0, 0),
             boxlen=0.5 if regions is SEDOV1D_REGIONS else 1.0)
    c.init_regions(regions)
    ref, dts_ref = c.oracle_steps(25)
    a = c.amr_commons()
    h = HydroGPU(a)
    h.bind_level(c.level)
    h.upload_state(c.level)
    dts, _ = h.level_steps(c.level, 25)
    h.download_state(c.level)
    h.finalize()
    idx = c.active_cells()
    ref = ref.reshape(c.nvar, -1)
    if riemann == "exact":
        assert max_rel_err(a.uold[:, idx], ref[:, idx]) <= 1e-12
    else:
        assert np.array_equal(dts, dts_ref)
        assert np.array_equal(a.uold[:, idx], ref[:, idx])


@pytest.mark.parametrize("bound", [(0,) * 6, (1, 1, 1, 1, 0, 0), (2, 2, 0, 0, 0, 0)])
@pytest.mark.parametrize("riemann,slope_type", [("hllc", 2), ("llf", 3)])
def test_2d_steps(gpu, bound, riemann, slope_type):
    from ramses_b200.hydro import HydroGPU
    c = Case(2, 5, riemann=riemann, slope_type=slope_type, bound=bound, order=2, seed=11)
    c.init_dense(smooth_state(2, 32))
    ref, dts_ref = c.oracle_steps(8)
    a = c.amr_commons()
    h = HydroGPU(a)
    h.bind_level(c.level)
    h.upload_state(c.level)
    dts, _ = h.level_steps(c.level, 8)
    h.download_state(c.level)
    h.finalize()
    idx = c.active_cells()
    assert np.array_equal(dts, dts_ref)
    assert np.array_equal(a.uold[:, idx], ref.reshape(c.nvar, -1)[:, idx])


def test_3d_reflexive_and_outflow(gpu):
    from ramses_b200.hydro import HydroGPU
    c = Case(3, 4, riemann="hllc", slope_type=2, bound=(1, 1, 2, 2, 1, 1), order=2, seed=5)
    c.init_dense(smooth_state(3, 16))
    ref, dts_ref = c.oracle_steps(6)
    a = c.amr_commons()
    h = HydroGPU(a)
    h.bind_level(c.level)
    h.upload_state(c.level)
    dts, _ = h.level_steps(c.level, 6)
    h.download_state(c.level)
    h.finalize()
    idx = c.active_cells()
    assert np.array_equal(dts, dts_ref)
    assert np.array_equal(a.uold[:, idx], ref.reshape(c.nvar, -1)[:, idx])


@pytest.mark.parametrize("amr_mode", [False, True])
def test_imposed_boundary_inflow(gpu, orc, amr_mode):
    """bound_type=3 (imposed, hydro/hydro_boundary.f90:229-252 with the default boundana): a denser supersonic inflow through the
    left face of a 1-D tube (outflow right face), dense kernel and oct-batch kernel: bit-identical to the oracle; the mass of the
    domain grows by the inflow."""
    import ctypes as C
    from ramses_b200.hydro import HydroGPU
    L = orc.lib()
    L.orc_set_boundary_var.argtypes = [C.c_int, C.POINTER(C.c_double), C.c_int]
    n = 64
    c = Case(1, 6, riemann="hllc", slope_type=1, bound=(3, 2, 0, 0, 0, 0))
    rho, u, p = 1.0, 3.0, 1.0
    cons = np.array([rho, rho * u, p / 0.4 + 0.5 * rho * u * u])
    cons2 = np.array([2.0, 2.0 * u, p / 0.4 + 0.5 * 2.0 * u * u])
    L.orc_set_boundary_var(0, orc.dptr(cons2), 3)
    d = np.zeros((3, 1, 1, n))
    d[:, 0, 0, :] = cons[:, None]
    c.init_dense(d)
    ref, dts_ref = c.oracle_steps(12, nthreads=1)
    a = c.amr_commons()
    h = HydroGPU(a, amr_mode=amr_mode)
    h.set_boundary_var(1, cons2)
    h.bind_level(c.level)
    h.upload_state(c.level)
    if amr_mode:
        from ramses_b200.hydro import amr_step
        dtnew = {l: 0.0 for l in range(0, c.level + 2)}
        dtold = dict(dtnew)
        dts = []
        for _ in range(12):
            amr_step(h, c.level, 1, c.level, [1] * 64, dtnew, dtold)
            dts.append(dtnew[c.level])
        dts = np.array(dts)
    else:
        dts, _ = h.level_steps(c.level, 12)
    h.download_state(c.level)
    h.finalize()
    idx = c.active_cells()
    assert np.array_equal(dts, dts_ref)
    assert np.array_equal(a.uold[:, idx], ref.reshape(c.nvar, -1)[:, idx])
    assert a.uold[0, idx].sum() > 1.05 * n


def test_courant_fine_parity(gpu):
    from ramses_b200.hydro import HydroGPU
    c = Case(3, 5, riemann="hllc", slope_type=1)
    c.init_dense(smooth_state(3, 32))
    dt_ref, sums_ref = c.oracle_courant()
    a = c.amr_commons()
    h = HydroGPU(a)
    h.bind_level(c.level)
    h.upload_state(c.level)
    a.dtnew[c.level] = c.p.boxlen / c.p.smallc
    dt = h.courant_fine(c.level)
    h.finalize()
    assert dt == dt_ref                     # min-reduction is order independent: exact
    assert np.allclose([a.mass_tot, a.ekin_tot, a.eint_tot], sums_ref, rtol=1e-13, atol=0)


def test_split_calls_match_fused(gpu):
    """Level-1 contract called routine by routine (amr_step order) equals the fused rgpu_level_steps."""
    from ramses_b200.hydro import HydroGPU
    c = Case(3, 4, riemann="hllc", slope_type=1, bound=(1, 1, 0, 0, 0, 0))
    c.init_dense(smooth_state(3, 16))
    ref, dts_ref = c.oracle_steps(3)
    a = c.amr_commons()
    h = HydroGPU(a)
    h.bind_level(c.level)
    h.upload_state(c.level)
    h.make_boundary_hydro(c.level)
    for s in range(3):
        a.dtnew[c.level] = c.p.boxlen / c.p.smallc
        h.courant_fine(c.level)
        assert a.dtnew[c.level] == dts_ref[s]
        h.set_unew(c.level)
        h.godunov_fine_dev(c.level)
        h.set_uold(c.level)
        h.make_boundary_hydro(c.level)
    h.download_state(c.level)
    h.finalize()
    idx = c.active_cells()
    assert np.array_equal(a.uold[:, idx], ref.reshape(c.nvar, -1)[:, idx])


def test_fast_div_sqrt_match_ieee(gpu):
    """The branch-free reciprocal / shared-reciprocal quotient / square root used in the kernels are bit-identical to
    the IEEE `1/b`, `a/b`, sqrt(a) on 2^28 random / adversarial operand pairs (exponents within 2^+-100)."""
    import ctypes as C
    from ramses_b200.hydro import HydroGPU
    c = Case(3, 2)
    h = HydroGPU(c.amr_commons())
    bad = C.c_longlong(-1)
    from ramses_b200 import lib
    lib.check(h.L.rgpu_selftest_div(1 << 28, 12345, C.byref(bad)))
    h.finalize()
    assert bad.value == 0


@pytest.mark.parametrize("level", [5, 7])
def test_multi_gpu_bit_identical_to_single_gpu(gpu, level):
    """2 (or more) GPUs with NCCL ghost-oct exchange == the same global problem on one GPU, bit for bit.  level 5: 32^3 per
    rank (one tile ring: the exchange is serial with the sweep); level 7: 128^3 per rank, where rgpu_level_steps splits the sweep
    into interior and frame launches and overlaps the fused exchange of the previous step with the interior (stream s_x)."""
    import os
    import subprocess
    import sys
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    n = 2 if n < 4 else (4 if n < 8 else 8)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr", "127.0.0.1",
           "--master-port", str(29617 + level), os.path.join(root, "tests", "mgpu_check.py"), str(level), "6", "hllc"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "state identical=True" in r.stdout


@pytest.mark.parametrize("args", [("2",), ("3",), ("3", "empty")])
def test_multi_gpu_amr_matches_single_gpu(gpu, args):
    """AMR mode with NCCL ghost-oct exchange (forward copy + reverse reflux accumulation) on 2 GPUs == one GPU
    (<= 1e-13: refluxes arriving from different ranks are summed in a different order), through the library's amr_step and
    through rgpu_amr_steps; "empty": the last rank owns no oct of the finest level and still takes part in that level's
    all-reduce and exchanges (numbtot gating, amr/amr_step.f90:33,345)."""
    import os
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", str(29641 + len(args) + int(args[0])), os.path.join(root, "tests", "mgpu_amr_check.py"), *args]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]


def test_full_size_256_properties(gpu):
    """BASELINE config 2 at full size (sedov3d 256^3, exact Riemann, 10 level steps) through size-independent
    properties: mass and energy conserved to round-off on the periodic box (mcons/econs of doc/wiki/Start.md), the
    x<->y<->z permutation symmetry of the corner blast, positivity, and dt of the first step equal to the oracle's
    closed form for the initial state."""
    import sys, os
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from bench import sedov_ic
    from ramses_b200.hydro import HydroGPU
    from ramses_b200.tree import build_uniform_tree, fill_state
    level, n = 8, 256
    a = build_uniform_tree(3, level, order="creation", boxlen=0.5)
    a.gamma, a.courant_factor, a.slope_type, a.riemann = 1.4, 0.8, 1, "exact"
    fill_state(a, level, sedov_ic(0.5, 1, level))
    ig = a.active[level].astype(np.int64)
    cells = np.concatenate([a.ncoarse + ind * a.ngridmax + ig - 1 for ind in range(8)])
    m0, e0 = a.uold[0, cells].sum(), a.uold[4, cells].sum()
    h = HydroGPU(a)
    h.bind_level(level)
    h.upload_state(level)
    dts, sums = h.level_steps(level, 10)
    h.download_state(level)
    h.finalize()
    u = a.uold[:, cells]
    assert abs(u[0].sum() - m0) <= 1e-13 * m0
    assert abs(u[4].sum() - e0) <= 1e-12 * e0
    assert u[0].min() > 0 and np.isfinite(u).all()
    # dt of step 1: the hottest cell (the one holding the blast energy) sets it, cmpdt (godunov_utils.f90:5-120)
    dx = 0.5 / n
    pmax = 1e-5 + 0.4 * 0.125 / dx ** 3
    ws = 3 * np.sqrt(1.4 * pmax / 1.0)
    g = 1e-4
    assert abs(dts[0] - dx / ws * (np.sqrt(1 + 2 * 0.8 * g) - 1) / g) <= 1e-14 * dts[0]
    assert np.all(np.diff(dts) != 0)
    # permutation symmetry: gather a 16^3 corner block (the blast has not left it after 10 steps)
    pos = a._pos[level][ig - a._igrid0[level]]
    dense = np.zeros((5, 16, 16, 16))
    for ind in range(8):
        c = 2 * pos + np.array([(ind >> d) & 1 for d in range(3)])[None, :]
        sel = (c < 16).all(axis=1)
        dense[:, c[sel, 2], c[sel, 1], c[sel, 0]] = a.uold[:, a.ncoarse + ind * a.ngridmax + ig[sel] - 1]
    assert np.abs(dense[0] - dense[0].transpose(0, 2, 1)).max() <= 1e-12 * dense[0].max()
    assert np.abs(dense[0] - dense[0].transpose(2, 1, 0)).max() <= 1e-12 * dense[0].max()
    assert np.abs(dense[1] - dense[2].transpose(0, 2, 1)).max() <= 1e-11 * np.abs(dense[1]).max()
    assert dense[0].max() > 1.05          # the blast is there


@pytest.mark.parametrize("bound", [(0,) * 6, (1, 1, 0, 0, 2, 2)])
@pytest.mark.parametrize("riemann", ["hllc", "llf"])
def test_level0_pipelined_equals_serial_and_oracle(gpu, riemann, bound):
    """rgpu_godunov_fine on host arrays with a spatially coherent (lattice) oct numbering runs as the three-stream z-slab pipeline
    (H2D | gather + sweep + scatter | D2H): same bits as the serial order of the same call and as the oracle; periodic box and
    a box with reflexive x walls / outflow z faces (ghost shells in the slab direction)."""
    from ramses_b200.hydro import HydroGPU
    c = Case(3, 6, riemann=riemann, slope_type=1, bound=bound, order=1, seed=5)
    d0 = smooth_state(3, 64)
    d0[0] *= 1 + 0.3 * (np.random.default_rng(11).standard_normal(d0[0].shape) > 1.0)
    c.init_dense(d0)
    dt, _ = c.oracle_courant()
    ref = c.oracle_godunov(dt).reshape(c.nvar, -1)
    a = c.amr_commons()
    h = HydroGPU(a)
    h.bind_level(c.level)
    info = h.level_info(c.level)
    assert info.dense == 1 and info.pipeline_slabs >= 3
    a.dtnew[c.level] = dt
    h.host_register(a.uold); h.host_register(a.unew)
    out = {}
    for mode in (1, 0):
        h.set_pipeline(mode)
        a.unew[:, :] = a.uold
        h.godunov_fine(c.level)
        out[mode] = a.unew.copy()
    h.host_unregister(a.uold); h.host_unregister(a.unew)
    h.finalize()
    idx = c.active_cells()
    assert np.array_equal(out[1], out[0])                       # every cell of the host array, ghosts and other levels included
    assert np.array_equal(out[1][:, idx], ref[:, idx])


def test_level0_creation_order_keeps_serial_path(gpu):
    """the reference's creation order scatters a z-slab over the whole igrid window: no pipeline plan, serial order"""
    from ramses_b200.hydro import HydroGPU
    c = Case(3, 6, riemann="hllc", slope_type=1, order=0)
    c.init_dense(smooth_state(3, 64))
    a = c.amr_commons()
    h = HydroGPU(a)
    h.bind_level(c.level)
    info = h.level_info(c.level)
    h.finalize()
    assert info.dense == 1 and info.pipeline_slabs == 0


@pytest.mark.parametrize("riemann,level,nstep", [("hllc", 7, 8), ("llf", 7, 8), ("exact", 7, 8), ("exact", 8, 4), ("hllc", 8, 4)])
def test_sedov3d_large_grid_vs_oracle(gpu, riemann, level, nstep):
    """GPU vs oracle at the sizes the bench measures (VERDICT r1 weak #1b): sedov3d on 128^3 and 256^3, fused level steps.
    hllc / llf: dt history and conserved state bit for bit (np.array_equal); exact: <= 1e-12 relative (CUDA pow vs libm pow in
    the rarefaction branch, hydro/godunov_utils.f90:415,453), the tolerance north_star states."""
    from ramses_b200.hydro import HydroGPU
    c = Case(3, level, riemann=riemann, slope_type=1, boxlen=0.5)
    c.init_regions(SEDOV3D_REGIONS)
    ref, dts_ref = c.oracle_steps(nstep, nthreads=16)
    a = c.amr_commons()
    h = HydroGPU(a)
    h.bind_level(c.level)
    h.upload_state(c.level)
    dts, _ = h.level_steps(c.level, nstep)
    h.download_state(c.level)
    h.finalize()
    idx = c.active_cells()
    ref = ref.reshape(c.nvar, -1)
    assert np.abs(ref[:, idx] - c.u.reshape(c.nvar, -1)[:, idx]).max() > 0          # the blast moved
    if riemann == "exact":
        assert np.allclose(dts, dts_ref, rtol=1e-12, atol=0)
        assert max_rel_err(a.uold[:, idx], ref[:, idx]) <= 1e-12
    else:
        assert np.array_equal(dts, dts_ref)
        assert np.array_equal(a.uold[:, idx], ref[:, idx])


@pytest.mark.parametrize("riemann", ["hllc", "exact", "llf", "hll", "acoustic"])
@pytest.mark.parametrize("ic", ["sedov", "smooth"])
def test_fast_mode_within_tolerance(gpu, riemann, ic):
    """rgpu_params.fast = 1 (FMA contraction, reciprocal-multiply quotients, <= 2 ulp reciprocal / sqrt in the 3-D dense sweep):
    after 12 fused level steps the conserved state and the dt history stay within north_star's tolerance (1e-12 relative) of the
    STRICT path and of the oracle; the strict path itself remains bit-identical to the oracle (other tests)."""
    from ramses_b200.hydro import HydroGPU
    c = Case(3, 6, riemann=riemann, slope_type=1, boxlen=0.5)
    if ic == "sedov":
        c.init_regions(SEDOV3D_REGIONS)
    else:
        c.init_dense(smooth_state(3, 64))
    ref, dts_ref = c.oracle_steps(12, nthreads=8)
    ref = ref.reshape(c.nvar, -1)
    out = {}
    for fast in (False, True):
        a = c.amr_commons()
        a.fast = fast
        h = HydroGPU(a)
        h.bind_level(c.level)
        h.upload_state(c.level)
        dts, _ = h.level_steps(c.level, 12)
        h.download_state(c.level)
        h.finalize()
        out[fast] = (a.uold.copy(), dts)
    idx = c.active_cells()
    us, uf = out[False][0][:, idx], out[True][0][:, idx]
    assert not np.array_equal(us, uf)                      # the fast build really is a different arithmetic
    assert max_rel_err(uf, us) <= 1e-12
    assert max_rel_err(uf, ref[:, idx]) <= 1e-12
    assert np.allclose(out[True][1], out[False][1], rtol=1e-12, atol=0)
    assert np.allclose(out[True][1], dts_ref, rtol=1e-12, atol=0)


def test_bench_dump_outputs(gpu, tmp_path):
    """bench.py --dump-outputs: after the --steps timed steps it writes their time steps and the seeded sample of the state they
    computed, in float64; the run's own check finds that state equal to the recorded single-GPU hashes (bench_hashes.json), and a
    second run with the same arguments writes the same arrays bit for bit."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = []
    for run in ("a", "b"):
        d = tmp_path / run
        cmd = [sys.executable, os.path.join(root, "bench.py"), "--workload", "sedov3d_128_hllc", "--steps", "5", "--warmup", "3",
               "--no-cpu-baseline", "--no-fast", "--e2e-steps", "1", "--dump-outputs", str(d)]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
        assert line["steps"] == 5 and line["check"]["equals_single_gpu_golden"] is True
        assert sorted(os.listdir(d)) == ["sedov3d_128_hllc_dt.npy", "sedov3d_128_hllc_state.npy"]
        out.append({f: np.load(d / f) for f in os.listdir(d)})
    dt, state = out[0]["sedov3d_128_hllc_dt.npy"], out[0]["sedov3d_128_hllc_state.npy"]
    assert dt.dtype == np.float64 and dt.shape == (5,) and (dt > 0).all()
    assert state.dtype == np.float64 and state.shape == (5, 1 << 17) and np.isfinite(state).all()
    for f in out[0]:
        assert np.array_equal(out[0][f], out[1][f]), f
