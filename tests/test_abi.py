"""The C-ABI library: builds, loads, exports every symbol include/anyseq.h declares,
and fails loudly (no CPU fallback) when there is no GPU.  No compute here."""
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_functions():
    src = open(os.path.join(ROOT, "include", "anyseq.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    names = re.findall(r"\b([a-z_][a-z0-9_]*)\s*\(", src)
    return sorted({n for n in names if n.startswith("anyseq_") or n.endswith("_alignment_score") or n.startswith("construct_")})


def test_library_builds_and_loads():
    import __graft_entry__ as G
    G.build()
    from anyseq_b200 import capi
    assert os.path.exists(capi.LIB_PATH)
    capi.load_library()


def test_exports_every_declared_symbol():
    from anyseq_b200 import capi
    L = capi.load_library()
    declared = _declared_functions()
    assert len(declared) >= 24
    for name in declared:
        assert hasattr(L, name), f"{name} declared in include/anyseq.h but not exported"
    assert sorted(capi.EXPORTED_SYMBOLS) == declared
    # the six symbols of the reference's src/import.h:14-41
    for name in ("global_alignment_score", "semiglobal_alignment_score", "local_alignment_score",
                 "construct_global_alignment", "construct_semiglobal_alignment", "construct_local_alignment"):
        assert name in declared


def test_sass_is_sm100a_with_dpx():
    """the shipped cubin targets sm_100a and the hot loop uses DPX (VIADDMNMX / VIMNMX3) + IMAD"""
    from anyseq_b200 import capi
    out = subprocess.run(["cuobjdump", "-lelf", capi.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    # the mixed-cell kernel (wide local Gotoh launches): strip_kernel<LOCAL=1, AFFINE=1, K=32, MASK=1, TRACK=0, FORM=2>
    hot = "_ZN6anyseq12strip_kernelILb1ELb1ELi32ELb1ELb0ELi2EEEvNS_10KernelArgsE"
    sass = subprocess.run(["cuobjdump", "-sass", "-fun", hot, capi.LIB_PATH], capture_output=True, text=True).stdout
    assert "Function : " + hot in sass, "hot kernel not found in the library (mangled name changed?)"
    n_dpx = sass.count("VIADDMNMX") + sass.count("VIMNMX3")
    assert n_dpx >= 500 and sass.count("VIMNMX3") >= 50 and sass.count("IMAD") >= 500 and "R2P" in sass, (n_dpx, sass.count("IMAD"))
    # the headline kernel (FORM=1, decoupled cells): four VIADDMNMX per cell, no VIMNMX3 in the cells
    dec = subprocess.run(["cuobjdump", "-sass", "-fun", "_ZN6anyseq12strip_kernelILb0ELb1ELi32ELb1ELb0ELi1EEEvNS_10KernelArgsE",
                          capi.LIB_PATH], capture_output=True, text=True).stdout
    assert dec.count("VIADDMNMX") >= 1000
    # the local and the linear-gap kernels use the .RELU / two-operand forms
    loc = subprocess.run(["cuobjdump", "-sass", "-fun", "_ZN6anyseq12strip_kernelILb1ELb0ELi32ELb1ELb0ELi1EEEvNS_10KernelArgsE",
                          capi.LIB_PATH], capture_output=True, text=True).stdout
    assert "VIADDMNMX.RELU" in loc
    # packed batch kernels: two 16-bit cells per DPX instruction, predicates from R2P
    sass = subprocess.run(["cuobjdump", "-sass", "-fun", "_ZN6anyseq15batch_x2_kernelILi1ELb1ELi16EEEvNS_9BatchArgsE",
                           capi.LIB_PATH], capture_output=True, text=True).stdout
    assert "VIADDMNMX.S16x2" in sass and "VIMNMX3.S16x2" in sass and "R2P" in sass


def test_no_cpu_fallback():
    """without a CUDA device the engine refuses to start; checked in a child process that sees no device, so that a
    machine with a GPU runs the check too"""
    child = ("import anyseq_b200 as A\n"
             "try:\n"
             "    A.Aligner(0)\n"
             "except A.AnyseqError as e:\n"
             "    assert e.code == -1 and 'no CPU fallback' in str(e), (e.code, str(e))\n"
             "    print('refused')\n")
    r = subprocess.run([sys.executable, "-c", child], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.strip() == "refused", r.stdout + r.stderr


def test_product_never_touches_the_oracle():
    """only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may use oracle/"""
    for dp, _, files in os.walk(os.path.join(ROOT, "anyseq_b200")):
        if "_build" in dp:
            continue
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                txt = open(os.path.join(dp, f), errors="ignore").read()
                assert "oracle" not in txt.lower(), os.path.join(dp, f)
    hdr = open(os.path.join(ROOT, "include", "anyseq.h")).read()
    assert "oracle" not in hdr.lower()


def test_reference_host_program_links_against_the_library(oracle):
    """the drop-in boundary, exercised by the reference's OWN caller: /root/reference/src/main.cpp (+ sequence_io,
    alignment_io) compiled unmodified and linked against libanyseq_b200.so in place of the AnyDSL object code
    (recipe: oracle/Makefile ref_host).  Needs the reference sources; on the GPU box the prebuilt binary is used."""
    from anyseq_b200 import build
    build.build()
    exe = oracle.build_reference_host()
    if exe is None:
        pytest.skip("reference sources not on this machine and no prebuilt oracle/_ref/align_reference_host")
    und = subprocess.run(["nm", "-u", exe], capture_output=True, text=True).stdout
    for sym in ("global_alignment_score", "semiglobal_alignment_score", "local_alignment_score",
                "construct_global_alignment", "construct_semiglobal_alignment", "construct_local_alignment"):
        assert sym in und, sym                      # resolved by our library at load time
    ldd = subprocess.run(["ldd", exe], capture_output=True, text=True).stdout
    assert "libanyseq_b200.so" in ldd and "not found" not in ldd
    r = subprocess.run([exe], capture_output=True, text=True)     # no arguments: the reference's usage text
    assert r.returncode == 0 and "SYNOPSIS" in r.stdout
