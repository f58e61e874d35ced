"""CPU-side checks of the drop-in boundary: the shared library loads, exports every symbol
include/raytrace_b200.h declares, and refuses to compute without a GPU (no CPU fallback)."""
import os
import re
import subprocess

import numpy as np
import pytest

import raytracerfortran_b200 as rt
from raytracerfortran_b200 import _lib, build, workloads

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _cuobjdump():
    # the toolkit that built the library, which need not be on PATH (build.nvcc_path falls back)
    return os.path.join(os.path.dirname(build.nvcc_path()), "cuobjdump")


@pytest.fixture(scope="module")
def lib():
    build.build_library()
    return _lib.load()


def _header_functions():
    src = open(os.path.join(ROOT, "include", "raytrace_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return set(re.findall(r"\b([A-Za-z_][A-Za-z0-9_]*)\s*\(", src)) - {"defined"}


def test_header_and_exports_agree(lib):
    declared = _header_functions()
    assert declared == set(_lib.EXPORTS)
    out = subprocess.check_output(["nm", "-D", "--defined-only", _lib.LIB_PATH], text=True)
    exported = {l.split()[-1] for l in out.splitlines() if " T " in l}
    missing = declared - exported
    assert not missing, missing
    for name in declared:
        assert getattr(lib, name) is not None


def test_library_is_sm100a_only(lib):
    out = subprocess.run([_cuobjdump(), "-lelf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


def test_kernels_stage_tiles_with_tma_bulk_copies(lib):
    """The batch kernels bring a tile's rows in with cp.async.bulk + mbarrier: the SASS carries
    UBLKCP (the bulk copy) and SYNCS (mbarrier arrive/wait), and fp64 math only (no tensor-core
    instructions: the path is not a contraction)."""
    sass = subprocess.run([_cuobjdump(), "-sass", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert sass.count("UBLKCP") >= 3 and sass.count("SYNCS") >= 3          # one per kernel variant at least
    assert "DFMA" in sass and "MUFU.RSQ64H" in sass
    assert not re.search(r"\b(HMMA|IMMA|UTCHMMA|UTCMMA|HGMMA)\b", sass)


def test_shard_range_partitions_the_model_axis(lib):
    for B in (0, 1, 7, 64, 1_000_003):
        for world in (1, 2, 3, 8):
            spans = [rt.shard_range(B, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == B
            for (a0, a1), (b0, b1) in zip(spans, spans[1:]):
                assert a1 == b0 and a0 <= a1
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1


def test_no_cpu_fallback(lib):
    if lib.rtb200_device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(rt.RayTraceError):
        rt.dff([3100.0, 4270.0], [2000.0], [100.0], [2500.0])
    with pytest.raises(rt.RayTraceError):
        v, z, nl = workloads.make_models(4, 3, 1)
        so, sd = workloads.make_sources(5, 1)
        rt.dff_batch(v, z, nl, so, sd)


def test_argument_validation():
    v, z, nl = workloads.make_models(4, 3, 1)
    so, sd = workloads.make_sources(5, 1)
    with pytest.raises(ValueError):
        rt.dff_batch(v, z, nl + 1, so, sd)                # nlayers exceeds the row length
    with pytest.raises(ValueError):
        rt.dff_batch(v, z, nl, so, sd, tobs=np.zeros(4), sigma=np.ones(4))   # tobs size != NSrc


def test_workloads_are_seeded_and_well_formed():
    v1, z1, nl1 = workloads.make_models(100, 10, 2)
    v2, z2, _ = workloads.make_models(100, 10, 2)
    assert np.array_equal(v1, v2) and np.array_equal(z1, z2)
    assert v1.min() >= 1500 and v1.max() <= 10000
    h = np.diff(np.concatenate([np.zeros((100, 1)), z1], axis=1), axis=1)
    assert h.min() >= 100.1 - 1e-9 and z1.max() <= 10000.1
    k, vp, zi = workloads.make_transd_models(500, 30, 3)
    assert k.min() >= 1 and k.max() <= 30
    for b in range(50):
        zz = zi[b, :k[b] - 1]
        assert np.all(np.diff(zz) >= 100.1 - 1e-9) and np.all(vp[b, :k[b]] >= 1500)
    so, sd = workloads.make_sources(64, 2)
    assert so.shape == sd.shape == (64,) and sd.min() >= 1050


def test_product_never_touches_the_oracle():
    """The oracle is test infrastructure: nothing under raytracerfortran_b200/ (Python, C++, CUDA)
    or include/ may import, link or mention it."""
    pkg = os.path.join(ROOT, "raytracerfortran_b200")
    offenders = []
    for base in (pkg, os.path.join(ROOT, "include"), os.path.join(ROOT, "shim")):
        for dirpath, _, files in os.walk(base):
            for f in files:
                if f.endswith((".py", ".cu", ".h", ".cuh", ".cpp", ".f90")):
                    text = open(os.path.join(dirpath, f), errors="ignore").read()
                    if re.search(r"\boracle\b|liboracle|raymod_oracle", text):
                        offenders.append(os.path.join(dirpath, f))
    assert not offenders, offenders
    out = subprocess.run(["ldd", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "oracle" not in out


def test_fortran_shim_binds_only_exported_symbols():
    """shim/raymod_b200.f90 cannot be compiled here (no Fortran compiler); at least every C name it
    binds must be one the library exports and the header declares."""
    import re
    src = open(os.path.join(ROOT, "shim", "raymod_b200.f90")).read()
    names = set(re.findall(r'bind\(C,\s*name="([A-Za-z0-9_]+)"\)', src))
    assert {"tracerays_", "dff_batch", "loglhood_batch"} <= names
    assert names <= set(_lib.EXPORTS), names - set(_lib.EXPORTS)


def test_header_is_plain_c_and_a_c_caller_links(tmp_path):
    """include/raytrace_b200.h is valid C99 and C++ (extern "C", plain pointers), and a C program
    written against it links with the library; without a GPU it fails loudly, never silently."""
    hdr = os.path.join(ROOT, "include", "raytrace_b200.h")
    cc, cxx = "/usr/bin/gcc", "/usr/bin/g++"
    if not (os.path.exists(cc) and os.path.exists(cxx)):
        pytest.skip("no host compiler")
    assert subprocess.run([cc, "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-fsyntax-only", "-x", "c", hdr]).returncode == 0
    assert subprocess.run([cxx, "-std=c++11", "-Wall", "-Werror", "-fsyntax-only", "-x", "c++", hdr]).returncode == 0
    exe = str(tmp_path / "dff_batch_example")
    libdir = os.path.dirname(_lib.LIB_PATH)
    r = subprocess.run([cc, "-std=c99", "-Wall", "-Wextra", os.path.join(ROOT, "examples", "dff_batch_example.c"),
                        "-I" + os.path.join(ROOT, "include"), "-L" + libdir, "-lraytrace_b200",
                        "-Wl,-rpath," + libdir, "-o", exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    run = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    if run.returncode == 0:
        assert "logL" in run.stdout                      # a GPU was there
    else:
        assert "no usable CUDA device" in run.stderr or "sm_100a" in run.stderr
