"""CPU-only checks of the drop-in boundary: libgangpack.so builds for sm_100a, loads, exports every
symbol include/gangpack.h declares, and refuses to run without a GPU (no CPU fallback)."""
import ctypes
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def native():
    import k8s_spark_scheduler_b200 as g
    g.native.build()
    return g.native


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "gangpack.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(gp_[a-z_]+)\s*\(", text)))


def test_header_and_binding_agree(native):
    assert _declared_symbols() == sorted(native.EXPORTS)


def test_library_exports_every_declared_symbol(native):
    out = subprocess.check_output(["nm", "-D", "--defined-only", native.LIB_PATH], text=True)
    exported = {line.split()[-1] for line in out.splitlines() if " T " in line}
    missing = [s for s in _declared_symbols() if s not in exported]
    assert not missing, missing
    lib = native.load()
    for s in _declared_symbols():
        assert getattr(lib, s) is not None
    assert lib.gp_abi_version() == 1


def test_rebuild_tracks_every_source():
    """build() recompiles when any file under csrc/ or the header is newer than the library."""
    import k8s_spark_scheduler_b200 as g
    csrc = os.path.join(ROOT, "k8s-spark-scheduler_b200", "csrc")
    tracked = {os.path.abspath(s) for s in g.native._SOURCES}
    missing = [f for f in sorted(os.listdir(csrc)) if os.path.join(csrc, f) not in tracked]
    assert not missing, missing
    assert os.path.join(ROOT, "include", "gangpack.h") in tracked


def test_library_contains_sm100a_code(native):
    cuobjdump = os.path.join(os.path.dirname(native._nvcc()), "cuobjdump")   # the toolkit that built the library
    out = subprocess.check_output([cuobjdump, "-lelf", native.LIB_PATH], text=True)
    assert "sm_100a" in out


def test_struct_layout_matches_header(native):
    """ctypes mirrors vs a C compiler's view of include/gangpack.h."""
    src = r'''
    #include <stdio.h>
    #include <stddef.h>
    #include "gangpack.h"
    int main(void) {
      printf("%zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(gp_config), sizeof(gp_nodes), sizeof(gp_apps), sizeof(gp_results), sizeof(gp_stats),
             sizeof(gp_sort_input), sizeof(gp_usage_input), sizeof(gp_reschedule));
      printf("%zu %zu %zu %zu %zu %zu %zu\n", offsetof(gp_nodes, n_groups), offsetof(gp_apps, exec_out_off), offsetof(gp_results, executor_nodes_cap),
             offsetof(gp_sort_input, executor_label_rank), offsetof(gp_usage_input, res_gpu), offsetof(gp_reschedule, min_frag),
             offsetof(gp_reschedule, host_nodes));
      return 0; }'''
    import tempfile
    with tempfile.TemporaryDirectory() as td:
        c = os.path.join(td, "t.c"); exe = os.path.join(td, "t")
        open(c, "w").write(src)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        lines = subprocess.check_output([exe], text=True).split("\n")
    sizes = [int(x) for x in lines[0].split()]
    offs = [int(x) for x in lines[1].split()]
    assert sizes == [ctypes.sizeof(native.gp_config), ctypes.sizeof(native.gp_nodes), ctypes.sizeof(native.gp_apps),
                     ctypes.sizeof(native.gp_results), ctypes.sizeof(native.gp_stats), ctypes.sizeof(native.gp_sort_input),
                     ctypes.sizeof(native.gp_usage_input), ctypes.sizeof(native.gp_reschedule)]
    assert offs == [native.gp_nodes.n_groups.offset, native.gp_apps.exec_out_off.offset,
                    native.gp_results.executor_nodes_cap.offset, native.gp_sort_input.executor_label_rank.offset,
                    native.gp_usage_input.res_gpu.offset, native.gp_reschedule.min_frag.offset,
                    native.gp_reschedule.host_nodes.offset]


def test_no_cpu_fallback(native):
    """Without a CUDA device context creation fails loudly; with one it reports the CUDA backend."""
    import torch
    if torch.cuda.is_available():
        p = native.GangPacker()
        assert native.load().gp_backend(p._h) == 1
        p.close()
    else:
        with pytest.raises(native.GangpackError) as ei:
            native.GangPacker()
        assert ei.value.status == 3  # GP_ERR_NO_DEVICE


def test_product_never_imports_the_oracle():
    """oracle/ is test infrastructure: nothing under the product package references it."""
    pkg = os.path.join(ROOT, "k8s-spark-scheduler_b200")
    offenders = []
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".hpp", ".cpp", ".go")):
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                if re.search(r"(from|import)\s+oracle|gangpack_oracle|oracle/", text):
                    offenders.append(os.path.join(dirpath, f))
    assert not offenders, offenders
