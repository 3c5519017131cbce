"""Build the reference's OWN CPU operators for the hot path from a checkout of the reference (rusty1s/pytorch_sparse,
read-only; nothing is copied into this repo) into oracle/_ref/. The checkout is $TSB200_REFERENCE or, when that is
unset, the directory `reference` beside this repository:

    _spmm_cpu.so      <- csrc/spmm.cpp + csrc/cpu/spmm_cpu.cpp
    _convert_cpu.so   <- csrc/convert.cpp + csrc/cpu/convert_cpu.cpp
    _version_cpu.so   <- csrc/version.cpp

Recipe: g++ directly on those files against the installed libtorch headers (no setup.py / cmake),
flags as the reference's setup.py:67-83 (-O3 -fopenmp -DAT_PARALLEL_OPENMP). OpenMP is NOT passed
at link time (this image's g++ has no libgomp.spec; libtorch already provides libgomp).

oracle/_ref is git-ignored; where no readable checkout exists nothing is built, the reference-suite test skips and
the other tests rely on the outputs of the reference stored under tests/golden/. TEST / BASELINE INFRASTRUCTURE ONLY
(see oracle/__init__.py).
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
OUT = ROOT / "oracle" / "_ref"
REF = Path(os.environ.get("TSB200_REFERENCE") or ROOT.parent / "reference")

LIBS = {
    "_spmm_cpu": ["csrc/spmm.cpp", "csrc/cpu/spmm_cpu.cpp"],
    "_convert_cpu": ["csrc/convert.cpp", "csrc/cpu/convert_cpu.cpp"],
    "_version_cpu": ["csrc/version.cpp"],
}


def _cmd(name, srcs):
    import sysconfig

    import torch
    from torch.utils import cpp_extension as ce
    inc = [f"-I{p}" for p in ce.include_paths()] + [f"-I{sysconfig.get_paths()['include']}",
                                                    f"-I{REF / 'csrc'}", f"-I{REF / 'third_party/parallel-hashmap'}"]
    tl = Path(torch.__file__).parent / "lib"
    cxx = "/usr/bin/g++" if Path("/usr/bin/g++").exists() else "g++"
    return [cxx, "-O3", "-std=c++17", "-fPIC", "-shared", "-fopenmp", "-DAT_PARALLEL_OPENMP", "-DWITH_PYTHON",
            "-Wno-sign-compare", f"-D_GLIBCXX_USE_CXX11_ABI={int(torch._C._GLIBCXX_USE_CXX11_ABI)}",
            f"-DTORCH_EXTENSION_NAME={name}", *inc, *[str(REF / s) for s in srcs], "-o", str(OUT / f"{name}.so"),
            f"-L{tl}", "-ltorch", "-ltorch_cpu", "-lc10", "-ltorch_python", f"-Wl,-rpath,{tl}"]


def _one(item):
    name, srcs = item
    so = OUT / f"{name}.so"
    if so.exists() and all(so.stat().st_mtime_ns >= (REF / s).stat().st_mtime_ns for s in srcs):
        return so
    res = subprocess.run(_cmd(name, srcs), capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(f"reference build of {name} failed:\n{res.stderr[-4000:]}")
    return so


REF_TESTS = ["test_matmul.py", "test_spmm.py", "test_spspmm.py", "test_coalesce.py", "test_storage.py",
             "test_transpose.py", "test_add.py", "test_mul.py", "test_tensor.py", "test_overload.py"]


def stage_tests() -> Path:
    """Stage the reference's own test files for the hot path, byte for byte, next to its compiled operators in
    oracle/_ref/ref_tests/ (git-ignored: they never enter this repo's history; tests/test_reference_suite_gpu.py runs
    them unmodified against pytorch_sparse_b200 where they have been staged)."""
    import shutil
    dst = OUT / "ref_tests"
    dst.mkdir(parents=True, exist_ok=True)
    for name in REF_TESTS:
        shutil.copyfile(REF / "test" / name, dst / name)
    return dst


def sources_available() -> bool:
    """True when REF is a readable checkout of the reference (an unreadable one is treated as absent)."""
    try:
        return (REF / "csrc/cpu/spmm_cpu.cpp").is_file()
    except OSError:
        return False


def build() -> Path:
    if not sources_available():
        raise FileNotFoundError(f"reference sources not found in {REF} "
                                "(set TSB200_REFERENCE to a checkout of the reference)")
    OUT.mkdir(parents=True, exist_ok=True)
    with ThreadPoolExecutor(max_workers=3) as ex:
        list(ex.map(_one, LIBS.items()))
    stage_tests()
    return OUT


ALL_LIBS = ["version", "convert", "diag", "spmm", "metis", "rw", "saint", "sample", "ego_sample", "hgt_sample",
            "neighbor_sample", "relabel"]


def build_full(out_dir: Path) -> Path:
    """All 12 CPU operator libraries (what torch_sparse/__init__.py:8-21 insists on loading), so the
    UNMODIFIED reference package can be imported for golden-vector generation. Not needed at test
    or bench time; kept out of the repo tree."""
    global OUT
    out_dir.mkdir(parents=True, exist_ok=True)
    saved, OUT = OUT, out_dir
    try:
        items = []
        for n in ALL_LIBS:
            srcs = [f"csrc/{n}.cpp"]
            if (REF / f"csrc/cpu/{n}_cpu.cpp").exists():
                srcs.append(f"csrc/cpu/{n}_cpu.cpp")
            items.append((f"_{n}_cpu", srcs))
        with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 2)) as ex:
            list(ex.map(_one, items))
    finally:
        OUT = saved
    return out_dir


def available() -> bool:
    return all((OUT / f"{n}.so").exists() for n in LIBS)


def load() -> None:
    """Register the reference's operators as torch.ops.torch_sparse.* in THIS process. Must not be
    combined with pytorch_sparse_b200's own torch_sparse-namespace registration
    (set TSB200_REGISTER_TORCH_SPARSE=0 or use a separate process)."""
    import torch
    for n in LIBS:
        torch.ops.load_library(str(OUT / f"{n}.so"))


if __name__ == "__main__":
    print(build())
