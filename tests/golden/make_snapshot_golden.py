#!/usr/bin/env python
"""Records what the reference's snapshot reader and checker return for the snapshots of tests/test_output_format.py:

  python tests/golden/make_snapshot_golden.py <reference>/tests/visu

For every snapshot the test writes, the reference's load_snapshot reads it and check_solution (where the test has a golden
file of the reference) compares it.  Written here:

  snapshot_golden.json   {name: {"files": {file: sha256}, "sums": {variable: check_solution's sum}, "check_solution": verdict}}
  snapshot_<name>.npz    load_snapshot's per-cell arrays and scalars (the short runs; the long runs keep sums only)
"""
import contextlib
import io
import json
import os
import sys
import tempfile

import numpy as np

OUT = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(OUT)
sys.path[:0] = [os.path.dirname(TESTS), TESTS]

import conftest                   # noqa: E402
import test_output_format as t    # noqa: E402


def read_and_check(visu, snapdir, iout, test_name=None, ref_json=None):
    """load_snapshot (and check_solution against tests/golden/<ref_json>) in the directory holding output_NNNNN/"""
    cwd = os.getcwd()
    os.chdir(os.path.dirname(snapdir))
    try:
        data = visu.load_snapshot(iout)["data"]
        rec = {"files": t.file_hashes(snapdir)}
        if test_name:
            os.mkdir("sums")
            os.chdir("sums")            # overwrite=True: check_solution writes its own sums as <test_name>-ref.dat
            with contextlib.redirect_stdout(io.StringIO()):
                visu.check_solution(data, test_name, overwrite=True)
            rec["sums"] = {k.strip(): float(v) for k, v in (line.split(":") for line in open(test_name + "-ref.dat"))}
            os.chdir("..")
            ref = json.load(open(os.path.join(OUT, ref_json)))
            with open(test_name + "-ref.dat", "w") as f:
                for k in sorted(ref):
                    f.write("%s : %.16e\n" % (k, ref[k]))
            buf = io.StringIO()
            with contextlib.redirect_stdout(buf):
                visu.check_solution(data, test_name)
            rec["check_solution"] = "PASSED" if "PASSED" in buf.getvalue() else "FAILED"
    finally:
        os.chdir(cwd)
    return data, rec


def save_arrays(name, data):
    arrays = {k: np.asarray(v) for k, v in data.items() if np.asarray(v).dtype.kind in "fiub"}
    np.savez_compressed(os.path.join(OUT, "snapshot_%s.npz" % name), **arrays)


def main():
    sys.path.insert(0, os.path.abspath(sys.argv[1]))
    import visu_ramses
    gold = {}
    with tempfile.TemporaryDirectory() as tmp:
        def new_dir(name):
            d = os.path.join(tmp, name)
            os.mkdir(d)
            return d
        r, _ = t.sod_run()
        data, gold["sod_tube"] = read_and_check(visu_ramses, t._write_from_run(r, new_dir("sod"), 2), 2, "sod-tube", "sod_tube_ref.json")
        save_arrays("sod_tube", data)
        r, _ = t.orszag_short_run()
        data, gold["orszag_tang_short"] = read_and_check(visu_ramses, t._write_from_run(r, new_dir("ots"), 2, mhd=True), 2)
        save_arrays("orszag_tang_short", data)
        data, gold["host_mirror"] = read_and_check(visu_ramses, t.write_host_mirror(t.host_mirror_commons(), new_dir("hm")), 1)
        save_arrays("host_mirror", data)
        r, _ = conftest.make_orszag_run()
        _, gold["orszag_tang"] = read_and_check(visu_ramses, t._write_from_run(r, new_dir("ot"), 2, mhd=True), 2, "orszag-tang",
                                                "orszag_tang_ref.json")
        r, _ = conftest.make_implosion_run()
        _, gold["implosion"] = read_and_check(visu_ramses, t._write_from_run(r, new_dir("impl"), 2), 2, "implosion",
                                              "implosion_ref.json")
    json.dump(gold, open(t.SNAPSHOT_GOLDEN, "w"), indent=1, sort_keys=True)
    print({k: v.get("check_solution") for k, v in gold.items()})


if __name__ == "__main__":
    main()
