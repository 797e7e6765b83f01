"""Snapshot files in the reference's on-disk format (SURVEY 8f-4: the data format on the far side of the hot path).

After `rgpu_download_state` the host arrays hold the conserved state in the layout of `hydro_commons`; `write_snapshot`
turns them into an `output_NNNNN/` directory that the reference's own tools read:

    info_NNNNN.txt               amr/output_amr.f90:408-492  output_info
    amr_NNNNN.out00001           amr/output_amr.f90:205-403  backup_amr   (Fortran unformatted records)
    hydro_NNNNN.out00001         hydro/output_hydro.f90:50-240 backup_hydro (primitive variables: density, velocities,
                                 [B left, B right for the MHD build, mhd/output_hydro.f90:82-137], pressure, scalars)
    hydro_file_descriptor.txt    io/dump_utils.f90:127-139
    header_NNNNN.txt             amr/output_amr.f90:497-575  output_header (particle families, all zero)

`read_snapshot` is the restart side (amr/init_amr.f90:227-520, hydro/init_hydro.f90:57-250).
Serial runs (ncpu=1) and the Hilbert ordering header only.  tests/test_output_format.py holds the files to the bytes the
reference's reader and checker (tests/visu/visu_ramses.py: load_snapshot + check_solution) read, with what they returned
stored under tests/golden/, and so closes the loop state -> reference file format -> reference reader -> reference golden sums.
"""
import os
import struct

import numpy as np


class _Records:
    """Fortran sequential unformatted file: every record is <int32 nbytes> payload <int32 nbytes>."""

    def __init__(self, path):
        self.f = open(path, "wb")

    def rec(self, *parts):
        payload = b"".join(parts)
        n = struct.pack("i", len(payload))
        self.f.write(n + payload + n)

    def ints(self, *v):
        self.rec(np.asarray(v, dtype=np.int32).tobytes())

    def dbls(self, *v):
        self.rec(np.asarray(v, dtype=np.float64).tobytes())

    def iarr(self, a):
        self.rec(np.ascontiguousarray(a, dtype=np.int32).tobytes())

    def darr(self, a):
        self.rec(np.ascontiguousarray(a, dtype=np.float64).tobytes())

    def close(self):
        self.f.close()


def _e23(x):
    """Fortran E23.15: 0.dddddddddddddddE+ee right-justified in 23 columns"""
    if x == 0.0:
        s = "0.000000000000000E+00"
    else:
        m, e = ("%.14E" % x).split("E")
        e = int(e) + 1
        neg = m.startswith("-")
        digits = m.replace("-", "").replace(".", "")
        s = ("-" if neg else "") + "0." + digits + ("E%+03d" % e)
    return s.rjust(23)


def write_snapshot(outdir, iout, *, ndim, nvar, levelmin, nlevelmax, ngridmax, ncoarse, nxyz, coarse_min, coarse_max, boxlen,
                   gamma, smallr, son, father, nbor, xg, active, boundary=(), uold, t=0.0, dtold=None, dtnew=None, nstep=0,
                   nstep_coarse=0, tout=(0.0,), flag1=None, cpu_map=None, mhd=False):
    """Write output_<iout>/ for a serial run.

    son[ncell], father[ngridmax], nbor[2*ndim][ngridmax], xg[ndim][ngridmax]: the tree arrays, 0-based views of the 1-based
    Fortran arrays (element i-1 = Fortran element i).  active[l-1] / boundary[b][l-1]: igrid lists (1-based values) of level l
    in linked-list order.  uold[nvar_stored][ncell] with nvar_stored = nvar (+3 for the MHD build).  Returns the directory."""
    T, twondim = 1 << ndim, 2 * ndim
    ncell = ncoarse + T * ngridmax
    nvs = nvar + 3 if mhd else nvar
    son, father, xg = np.asarray(son), np.asarray(father), np.asarray(xg)
    nbor, uold = np.asarray(nbor), np.asarray(uold)
    assert son.shape == (ncell,) and father.shape == (ngridmax,) and nbor.shape == (twondim, ngridmax)
    assert xg.shape == (ndim, ngridmax) and uold.shape == (nvs, ncell)
    flag1 = np.zeros(ncell, dtype=np.int32) if flag1 is None else np.asarray(flag1, dtype=np.int32)
    cpu_map = np.ones(ncell, dtype=np.int32) if cpu_map is None else np.asarray(cpu_map, dtype=np.int32)
    nboundary = len(boundary)
    nchar = "%05d" % iout
    d = os.path.join(outdir, "output_" + nchar)
    os.makedirs(d, exist_ok=True)
    dtold = np.zeros(nlevelmax) if dtold is None else np.asarray(dtold, dtype=float)
    dtnew = np.zeros(nlevelmax) if dtnew is None else np.asarray(dtnew, dtype=float)
    lists = [[np.asarray(active[l], dtype=np.int64)] + [np.asarray(boundary[b][l], dtype=np.int64) for b in range(nboundary)]
             for l in range(nlevelmax)]                    # [level][domain]: cpu 1, then the boundary regions
    nx, ny, nz = nxyz
    nx_loc = coarse_max[0] - coarse_min[0] + 1
    scale = boxlen / float(nx_loc)

    # ---- info file (output_info) ------------------------------------------------------------------------------------
    with open(os.path.join(d, "info_" + nchar + ".txt"), "w") as f:
        for k, v in (("ncpu", 1), ("ndim", ndim), ("levelmin", levelmin), ("levelmax", nlevelmax), ("ngridmax", ngridmax),
                     ("nstep_coarse", nstep_coarse)):
            f.write("%-12s=%11d\n" % (k, v))
        f.write("\n")
        for k, v in (("boxlen", scale), ("time", t), ("aexp", 1.0), ("H0", 1.0), ("omega_m", 1.0), ("omega_l", 0.0),
                     ("omega_k", 0.0), ("omega_b", 0.0), ("unit_l", 1.0), ("unit_d", 1.0), ("unit_t", 1.0)):
            f.write("%-12s=%s\n" % (k, _e23(v)))
        f.write("\n")
        f.write("ordering type=" + "hilbert".ljust(80) + "\n")
        f.write("   DOMAIN   ind_min                 ind_max\n")
        f.write("%8d %s %s\n" % (1, _e23(0.0), _e23(float(2 ** (ndim * (nlevelmax + 1))))))

    # ---- header file (output_header, amr/output_amr.f90:497-575): particle families, all empty ----------------------------------
    with open(os.path.join(d, "header_" + nchar + ".txt"), "w") as f:
        f.write("#%12s%10s\n" % ("Family", "Count"))
        for fam in ("other_tracer", "debris_tracer", "cloud_tracer", "star_tracer", "other_tracer", "gas_tracer", "DM", "star",
                    "cloud", "debris", "other", "undefined"):
            f.write("%13s%10d\n" % (fam, 0))
        f.write(" Particle fields\n")
        f.write("pos vel mass iord level family tag ")

    # ---- amr file (backup_amr) ----------------------------------------------------------------------------------------
    # linked lists (headl/taill/numbl, next/prev) rebuilt from the list order
    nxt, prv = np.zeros(ngridmax, dtype=np.int32), np.zeros(ngridmax, dtype=np.int32)
    headl, taill, numbl = (np.zeros(nlevelmax, dtype=np.int32) for _ in range(3))
    headb, tailb, numbb = (np.zeros((nlevelmax, max(nboundary, 1)), dtype=np.int32) for _ in range(3))
    for l in range(nlevelmax):
        for dom, g in enumerate(lists[l]):
            if len(g) == 0:
                continue
            nxt[g[:-1] - 1], prv[g[1:] - 1] = g[1:], g[:-1]
            if dom == 0:
                headl[l], taill[l], numbl[l] = g[0], g[-1], len(g)
            else:
                headb[l, dom - 1], tailb[l, dom - 1], numbb[l, dom - 1] = g[0], g[-1], len(g)
    ngrid_current = int(sum(len(g) for lv in lists for g in lv))
    numbtot = np.zeros((nlevelmax, 10), dtype=np.int32)
    numbtot[:, 0] = numbtot[:, 1] = numbtot[:, 2] = numbl
    numbtot[:, 3] = numbl
    noutput = len(tout)
    r = _Records(os.path.join(d, "amr_" + nchar + ".out00001"))
    r.ints(1); r.ints(ndim); r.ints(nx, ny, nz); r.ints(nlevelmax); r.ints(ngridmax); r.ints(nboundary); r.ints(ngrid_current)
    r.dbls(boxlen)
    r.ints(noutput, min(iout, noutput), 1)
    r.darr(tout); r.darr(np.ones(noutput))
    r.dbls(t)
    r.darr(dtold); r.darr(dtnew)
    r.ints(nstep, nstep_coarse)
    r.dbls(0.0, 0.0, 0.0)                                  # einit, mass_tot_0, rho_tot
    r.dbls(1.0, 0.0, 0.0, 0.0, 1.0, 1.0, boxlen)           # omega_m, omega_l, omega_k, omega_b, h0, aexp_ini, boxlen_ini
    r.dbls(1.0, 0.0, 1.0, 0.0, 0.0)                        # aexp, hexp, aexp_old, epot_tot_int, epot_tot_old
    r.dbls(0.0)                                            # mass_sph
    r.iarr(headl); r.iarr(taill); r.iarr(numbl)            # (1:ncpu, 1:nlevelmax) with ncpu = 1
    r.iarr(numbtot.reshape(-1))                            # numbtot(1:10, 1:nlevelmax): ten values per level
    if nboundary > 0:
        r.iarr(headb[:, :nboundary].reshape(-1)); r.iarr(tailb[:, :nboundary].reshape(-1)); r.iarr(numbb[:, :nboundary].reshape(-1))
    used = set(int(x) for lv in lists for g in lv for x in g)
    free = [i for i in range(1, ngridmax + 1) if i not in used] if ngridmax <= 200000 else []
    r.ints(free[0] if free else 0, free[-1] if free else 0, ngridmax - ngrid_current, 0, 0)   # headf, tailf, numbf, used_mem, used_mem_tot
    r.rec("hilbert".ljust(128).encode())
    r.dbls(0.0, float(2 ** (ndim * (nlevelmax + 1))))      # bound_key(0:ndomain), qdp = real*8
    r.iarr(son[:ncoarse]); r.iarr(flag1[:ncoarse]); r.iarr(cpu_map[:ncoarse])
    for l in range(nlevelmax):
        for g in lists[l]:
            if len(g) == 0:
                continue
            gi = g - 1
            r.iarr(g); r.iarr(nxt[gi]); r.iarr(prv[gi])
            for k in range(ndim):
                r.darr(xg[k, gi])
            r.iarr(father[gi])
            for j in range(twondim):
                r.iarr(nbor[j, gi])
            for arr in (son, cpu_map, flag1):
                for ind in range(T):
                    r.iarr(arr[ncoarse + ind * ngridmax + gi])
    r.close()

    # ---- hydro file (backup_hydro) + descriptor ---------------------------------------------------------------------------
    names = ["density"] + ["velocity_" + "xyz"[k] for k in range(3 if mhd else ndim)]
    if mhd:
        names += ["B_%s_left" % c for c in "xyz"] + ["B_%s_right" % c for c in "xyz"]
    names += ["pressure"] + ["scalar_%02d" % k for k in range(nvar - (8 if mhd else ndim + 2))]   # hydro/output_hydro.f90: ivar-ndim-3-nener, 0-based
    with open(os.path.join(d, "hydro_file_descriptor.txt"), "w") as f:
        f.write("# version:  1\n# ivar, variable_name, variable_type\n")
        for i, nm in enumerate(names):
            f.write("%2d, %s, d\n" % (i + 1, nm))
    r = _Records(os.path.join(d, "hydro_" + nchar + ".out00001"))
    r.ints(1); r.ints(nvs); r.ints(ndim); r.ints(nlevelmax); r.ints(nboundary); r.dbls(gamma)
    for l in range(nlevelmax):
        for g in lists[l]:
            r.ints(l + 1); r.ints(len(g))
            if len(g) == 0:
                continue
            for ind in range(T):
                c = ncoarse + ind * ngridmax + g - 1
                u = uold[:, c]
                dmax = np.maximum(u[0], smallr)
                r.darr(u[0])
                nvel = 3 if mhd else ndim
                for k in range(nvel):
                    r.darr(u[1 + k] / dmax)
                if mhd:
                    for k in range(3):
                        r.darr(u[5 + k])
                    for k in range(3):
                        r.darr(u[nvar + k])
                    vx, vy, vz = u[1] / dmax, u[2] / dmax, u[3] / dmax
                    A, B, C = 0.5 * (u[5] + u[nvar]), 0.5 * (u[6] + u[nvar + 1]), 0.5 * (u[7] + u[nvar + 2])
                    e = u[4] - 0.5 * dmax * (vx ** 2 + vy ** 2 + vz ** 2) - 0.5 * (A ** 2 + B ** 2 + C ** 2)
                    r.darr((gamma - 1.0) * e)
                    first_scalar = 8
                else:
                    e = u[ndim + 1].copy()
                    for k in range(ndim):
                        e = e - 0.5 * u[1 + k] ** 2 / dmax
                    r.darr((gamma - 1.0) * e)
                    first_scalar = ndim + 2
                for k in range(first_scalar, nvar):
                    r.darr(u[k] / dmax)
    r.close()
    return d


def snapshot_from_commons(a, outdir, iout, t=0.0, levelmin=None, nstep=0, nstep_coarse=0):
    """write_snapshot for the host mirror of one rank (ramses_b200.hydro.AmrCommons as filled by the tree fabricators of
    ramses_b200.tree, i.e. carrying the integer oct positions `_pos`): what a run does after `HydroGPU.download_state()`."""
    L = a.nlevelmax
    xg = np.zeros((a.ndim, a.ngridmax))
    for l in range(1, L + 1):
        if l not in a._pos:
            continue
        pos, ig0 = a._pos[l], a._igrid0[l]
        ig = np.arange(ig0, ig0 + len(pos))
        for k in range(a.ndim):
            xg[k, ig - 1] = (pos[:, k] + 0.5) / 2.0 ** (l - 1)
    empty = np.zeros(0, dtype=np.int32)
    nb = len(a.boundary_type)
    return write_snapshot(
        outdir, iout, ndim=a.ndim, nvar=a.nvar, levelmin=levelmin or L, nlevelmax=L, ngridmax=a.ngridmax, ncoarse=a.ncoarse,
        nxyz=(a.nx, a.ny, a.nz), coarse_min=(a.icoarse_min, a.jcoarse_min, a.kcoarse_min),
        coarse_max=(a.icoarse_max, a.jcoarse_max, a.kcoarse_max), boxlen=a.boxlen, gamma=a.gamma, smallr=a.smallr, son=a.son,
        father=a.father, nbor=a.nbor, xg=xg, active=[a.active.get(l, empty) for l in range(1, L + 1)],
        boundary=[[(a.boundary.get(l) or [empty] * nb)[b] for l in range(1, L + 1)] for b in range(nb)], uold=a.uold, t=t,
        dtold=[getattr(a, "dtold", a.dtnew).get(l, 0.0) for l in range(1, L + 1)], dtnew=[a.dtnew.get(l, 0.0) for l in range(1, L + 1)], nstep=nstep,
        nstep_coarse=nstep_coarse, mhd=a.mhd)


class _Reader:
    def __init__(self, path):
        self.b = open(path, "rb").read()
        self.o = 0

    def rec(self):
        n = struct.unpack_from("i", self.b, self.o)[0]
        payload = self.b[self.o + 4:self.o + 4 + n]
        assert struct.unpack_from("i", self.b, self.o + 4 + n)[0] == n, "corrupt Fortran record"
        self.o += n + 8
        return payload

    def ints(self):
        return np.frombuffer(self.rec(), dtype=np.int32)

    def dbls(self):
        return np.frombuffer(self.rec(), dtype=np.float64)


def read_snapshot(outdir, iout, smallr=1e-10):
    """The restart side (amr/init_amr.f90:227-520 for the tree, hydro/init_hydro.f90:57-250 for the state) of a serial
    hydro snapshot: returns a dict with the header scalars, the tree arrays in the 0-based-view convention of write_snapshot, the
    per-level igrid lists and `uold[nvar][ncell]` rebuilt from the primitive records exactly as init_hydro does
    (momentum = v*max(rho,smallr), E = P/(gamma-1) + sum 0.5*mom^2/max(rho,smallr))."""
    nchar = "%05d" % iout
    d = os.path.join(outdir, "output_" + nchar)
    r = _Reader(os.path.join(d, "amr_" + nchar + ".out00001"))
    ncpu = int(r.ints()[0]); ndim = int(r.ints()[0]); nx, ny, nz = (int(v) for v in r.ints())
    nlevelmax = int(r.ints()[0]); ngridmax = int(r.ints()[0]); nboundary = int(r.ints()[0]); ngrid_current = int(r.ints()[0])
    boxlen = float(r.dbls()[0])
    noutput, iout2, ifout = (int(v) for v in r.ints())
    tout = r.dbls().copy(); r.dbls()
    t = float(r.dbls()[0])
    dtold = r.dbls().copy(); dtnew = r.dbls().copy()
    nstep, nstep_coarse = (int(v) for v in r.ints())
    for _ in range(4):
        r.dbls()
    assert ncpu == 1
    headl = r.ints().copy(); taill = r.ints().copy(); numbl = r.ints().copy(); r.ints()
    numbb = np.zeros((nlevelmax, max(nboundary, 1)), dtype=np.int32)
    if nboundary > 0:
        r.ints(); r.ints(); numbb = r.ints().reshape(nlevelmax, nboundary).copy()
    r.ints()                                               # headf, tailf, numbf, used_mem, used_mem_tot
    ordering = r.rec().decode().strip()
    r.rec()                                                # bound_key
    T, twondim = 1 << ndim, 2 * ndim
    ncoarse = nx * ny * nz
    ncell = ncoarse + T * ngridmax
    son = np.zeros(ncell, dtype=np.int32); flag1 = np.zeros(ncell, dtype=np.int32); cpu_map = np.zeros(ncell, dtype=np.int32)
    father = np.zeros(ngridmax, dtype=np.int32); nbor = np.zeros((twondim, ngridmax), dtype=np.int32)
    xg = np.zeros((ndim, ngridmax))
    son[:ncoarse] = r.ints(); flag1[:ncoarse] = r.ints(); cpu_map[:ncoarse] = r.ints()
    active = [np.zeros(0, dtype=np.int32) for _ in range(nlevelmax)]
    boundary = [[np.zeros(0, dtype=np.int32) for _ in range(nlevelmax)] for _ in range(nboundary)]
    for l in range(nlevelmax):
        for dom in range(1 + nboundary):
            ncache = int(numbl[l]) if dom == 0 else int(numbb[l, dom - 1])
            if ncache == 0:
                continue
            g = r.ints().copy(); r.ints(); r.ints()
            if dom == 0:
                active[l] = g
            else:
                boundary[dom - 1][l] = g
            gi = g.astype(np.int64) - 1
            for k in range(ndim):
                xg[k, gi] = r.dbls()
            father[gi] = r.ints()
            for j in range(twondim):
                nbor[j, gi] = r.ints()
            for arr in (son, cpu_map, flag1):
                for ind in range(T):
                    arr[ncoarse + ind * ngridmax + gi] = r.ints()
    h = _Reader(os.path.join(d, "hydro_" + nchar + ".out00001"))
    h.ints(); nvar = int(h.ints()[0]); h.ints(); h.ints(); h.ints(); gamma = float(h.dbls()[0])
    if nvar != ndim + 2 and nvar < ndim + 2 or nvar == 11 and ndim == 3:
        raise ValueError("read_snapshot rebuilds hydro builds only (nvar = ndim+2 [+ passive scalars]); an MHD snapshot "
                         "(11 records per cell: 3 velocities, 6 face fields) is not supported")
    uold = np.zeros((nvar, ncell))
    for l in range(nlevelmax):
        for dom in range(1 + nboundary):
            h.ints(); ncache = int(h.ints()[0])
            if ncache == 0:
                continue
            g = (active[l] if dom == 0 else boundary[dom - 1][l]).astype(np.int64)
            for ind in range(T):
                c = ncoarse + ind * ngridmax + g - 1
                uold[0, c] = h.dbls()
                dmax = np.maximum(uold[0, c], smallr)
                for k in range(ndim):
                    uold[1 + k, c] = h.dbls() * dmax
                e = h.dbls() / (gamma - 1.0)
                for k in range(ndim):
                    e = e + 0.5 * uold[1 + k, c] ** 2 / dmax
                uold[ndim + 1, c] = np.where(uold[0, c] > 0.0, e, 0.0)
                for k in range(ndim + 2, nvar):
                    uold[k, c] = h.dbls() * dmax
    return dict(ndim=ndim, nxyz=(nx, ny, nz), nlevelmax=nlevelmax, ngridmax=ngridmax, nboundary=nboundary, ncoarse=ncoarse,
                ngrid_current=ngrid_current, boxlen=boxlen, t=t, dtold=dtold, dtnew=dtnew, nstep=nstep, nstep_coarse=nstep_coarse,
                tout=tout, ordering=ordering, gamma=gamma, nvar=nvar, son=son, father=father, nbor=nbor, xg=xg, flag1=flag1,
                cpu_map=cpu_map, active=active, boundary=boundary, uold=uold)
