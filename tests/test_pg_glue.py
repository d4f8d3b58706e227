"""The PostgreSQL-side glue (pg_glue/*.c) and a plain C caller of the library (tests/c/driver.c).

The image has no PostgreSQL headers, so the glue cannot be linked here; it is type-checked: every file must compile
with -fsyntax-only -Wall -Wextra -Werror against pg_glue/stub/postgres.h (PostgreSQL's and Citus's declarations, restated) and
the real include/citus_gpu.h -- so every call into the library, every struct field and every callback signature is
checked by the compiler.  The C driver is built here and run on the GPU box."""
import glob
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_pg_glue_type_checks_against_the_stub_headers():
    files = sorted(glob.glob(os.path.join(ROOT, "pg_glue", "*.c")))
    assert len(files) >= 5
    for f in files:
        r = subprocess.run(["gcc", "-fsyntax-only", "-std=gnu11", "-Wall", "-Wextra", "-Wno-unused-parameter", "-Werror",
                            "-I", os.path.join(ROOT, "pg_glue", "stub"), "-I", os.path.join(ROOT, "include"), f],
                           capture_output=True, text=True)
        assert r.returncode == 0, f"{f}:\n{r.stderr}"


def test_glue_registers_the_reference_hook_points():
    src = open(os.path.join(ROOT, "pg_glue", "gpu_columnar_agg.c")).read()
    for needle in ("RegisterCustomScanMethods", "create_upper_paths_hook", "StripesForRelfilelocator", "ReadStripeSkipList",
                   "ExecStoreVirtualTuple", "cg_scan_relation", "cg_partial_fetch"):
        assert needle in src, needle
    shim = open(os.path.join(ROOT, "pg_glue", "gpu_aggregate_shim.c")).read()
    for sig in ("gpu_worker_partial_agg_sfunc", "gpu_worker_partial_agg_ffunc", "gpu_coord_combine_agg_sfunc", "gpu_coord_combine_agg_ffunc"):
        assert f"PG_FUNCTION_INFO_V1({sig})" in shim


def _build_driver(tmp_path):
    exe = str(tmp_path / "driver")
    subprocess.check_call(["gcc", "-O2", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "c", "driver.c"), "-ldl", "-o", exe])
    return exe


def test_c_driver_builds_and_fails_loudly_without_a_gpu(tmp_path):
    from citus_b200 import build
    from oracle import oracle as orc
    build.build()
    orc.build()
    exe = _build_driver(tmp_path)
    # where a GPU is present, the driver is shown none (CUDA_VISIBLE_DEVICES empty)
    r = subprocess.run([exe, os.path.join(ROOT, "citus_b200", "lib", "libcitus_gpu.so"), os.path.join(ROOT, "oracle", "liboracle.so")],
                       capture_output=True, text=True, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 1 and "cg_init" in r.stderr            # no device: an error, never a CPU fallback


@pytest.mark.gpu
def test_c_driver_runs_c1_bit_exact(tmp_path):
    from citus_b200 import build
    from oracle import oracle as orc
    build.build()
    orc.build()
    exe = _build_driver(tmp_path)
    r = subprocess.run([exe, os.path.join(ROOT, "citus_b200", "lib", "libcitus_gpu.so"), os.path.join(ROOT, "oracle", "liboracle.so")],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "bit-exact" in r.stdout
