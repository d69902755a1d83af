"""Worker of tests/test_matrix_shapes_gpu.py::test_env_selected_paths.  The engine reads FDB_BDB_SYM and
FDB_MAT_NO_RANK once per process, so each runs here in a process of its own:

* FDB_BDB_SYM=0: the generic B^T D B kernel (bdb_matrix_kernel) at p = 3 and p = 4, where the
  symmetric tilings are used otherwise;
* FDB_MAT_NO_RANK=1: no rank table, so every scatter binary-searches its row, on full extruded sets.

Prints ``MATRIX_ENV_OK <name>`` when every case passes."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from firedrake_b200 import _lib                 # noqa: E402
import test_matrix_shapes_gpu as T              # noqa: E402

engine = _lib.init(0)


def with_kernel(value, fn, *args):
    _lib.check(engine.fdb_set_option(b"matrix_kernel", value))
    try:
        fn(*args)
    finally:
        _lib.check(engine.fdb_set_option(b"matrix_kernel", -1))


if os.environ.get("FDB_BDB_SYM") == "0":
    name = "FDB_BDB_SYM"
    for p in (3, 4):
        for alpha, beta in T.FORMS:
            with_kernel(1, T.check_forms_multipass, p, alpha, beta, False)
        with_kernel(1, T.check_short_columns, p, 2)
        with_kernel(1, T.check_ranges, p)
        with_kernel(1, T.check_lgmaps, p)
elif os.environ.get("FDB_MAT_NO_RANK") == "1":
    name = "FDB_MAT_NO_RANK"
    for kernel in (0, 1):
        for p in (1, 2, 3, 4):
            with_kernel(kernel, T.check_forms_multipass, p, 1.0, 0.7)
            for nz in (1, 2, 3):
                with_kernel(kernel, T.check_short_columns, p, nz)
            with_kernel(kernel, T.check_ranges, p)
            with_kernel(kernel, T.check_lgmaps, p)
else:
    sys.exit("set FDB_BDB_SYM=0 or FDB_MAT_NO_RANK=1")
print("MATRIX_ENV_OK", name, flush=True)
