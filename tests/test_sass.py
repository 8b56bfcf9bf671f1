"""CPU: what the built library's machine code must contain (cuobjdump on the in-tree libr3g.so).  These are the SASS
mnemonics that prove the Blackwell paths are the ones compiled in -- tcgen05 MMAs (UTCHMMA), TMA loads (UTMALDG), TMEM
loads/stores (LDTM/STTM), the packed fp32 pipe (FFMA2/FADD2) -- and guards against two regressions found by profiling:
a GPU-scope membar in the GEMM pipeline (a `.release.cluster` remote arrive) and register spills in the hot kernels."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "3d-re-gen_b200", "r3g", "libr3g.so")


@pytest.fixture(scope="module")
def sass():
    # the CUDA toolkit's own location when it is not on PATH, as the build does for nvcc
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not found")
    import sys
    sys.path.insert(0, ROOT)
    import __graft_entry__ as ge
    ge.build()
    txt = subprocess.run([cuobjdump, "-sass", LIB], capture_output=True, text=True, check=True).stdout
    funcs = {}
    for blk in re.split(r"\n\s*Function : ", txt)[1:]:
        name, _, body = blk.partition("\n")
        funcs[name.strip()] = body
    res = subprocess.run([cuobjdump, "-res-usage", LIB], capture_output=True, text=True, check=True).stdout
    usage = {m.group(1): (int(m.group(2)), int(m.group(3)))
             for m in re.finditer(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+)", res)}
    return funcs, usage


def _one(funcs, *needles):
    hits = [n for n in funcs if all(s in n for s in needles)]
    assert hits, f"no kernel matching {needles}"
    return hits


def test_gemm_is_tcgen05_tma_and_has_no_gpu_scope_membar(sass):
    funcs, usage = sass
    for name in _one(funcs, "linear_kernel_2cta") + _one(funcs, "linear_kernelILi256E"):
        body = funcs[name]
        assert "UTCHMMA" in body and "UTMALDG" in body and "LDTM" in body, name
        # the only GPU-scope membars allowed are the two cluster barriers (start / end of the kernel)
        ins = [ln for ln in body.split("\n") if re.match(r"\s*/\*[0-9a-f]{4}\*/", ln)]
        for i, ln in enumerate(ins):
            if "MEMBAR.ALL.GPU" in ln:
                assert any("UCGABAR_ARV" in x for x in ins[i:i + 5]), \
                    name + ": a GPU-scope membar outside the cluster barriers (a .release.cluster arrive in the pipeline?)"
        assert sum("MEMBAR.ALL.GPU" in ln for ln in ins) <= 2, name
        assert usage[name][1] <= 64, f"{name}: {usage[name][1]} bytes of stack (spills)"
    assert "UTCHMMA.2CTA" in funcs[_one(funcs, "linear_kernel_2cta")[0]]


def test_default_attention_uses_tmem_operand_mma_and_packed_fp32(sass):
    funcs, usage = sass
    name = _one(funcs, "attention_kernelILb1ELb1ELi4ELi2ELb1E")[0]     # <P in TMEM, f32 exps, 1/4 poly, 2 stages, FFMA2>
    body = funcs[name]
    assert re.search(r"UTCHMMA\s+tmem\[", body), "P V must take its A operand from TMEM"
    assert re.search(r"UTCHMMA\s+gdesc\[", body), "Q K^T is the shared-memory form"
    for op in ("UTMALDG", "LDTM", "STTM.x32", "FFMA2", "FADD2", "MUFU.EX2", "FMNMX3"):
        assert op in body, op
    assert "MUFU.EX2.F16" not in body          # the f16x2 form splits into two MUFU + a PRMT
    assert usage[name][1] == 0, "register spills in the softmax loop"
    assert "NANOSLEEP.SYNCS" in body           # mbarrier.try_wait carries the suspend-time hint


def test_row_kernels_use_the_packed_fp32_pipe(sass):
    funcs, _ = sass
    for needle in ("layernorm_kernelILi4E", "lnpost_dot_kernelILi4E"):
        body = funcs[_one(funcs, needle)[0]]
        assert "FFMA2" in body and "FADD2" in body, needle
    # every fp16 row moves as 16-byte accesses (a `__half2 v[4]` payload is copied member-wise: four 32-bit LDG/STG)
    for needle in ("layernorm_kernelILi4E", "lnpost_dot_kernelILi4E", "qk_norm_kernel", "gemv_kernel"):
        body = funcs[_one(funcs, needle)[0]]
        assert "LDG.E.128" in body or "LDG.E.CONSTANT.128" in body or "LD.E.128" in body, needle
    for needle in ("layernorm_kernelILi4E", "grid_fourier_kernel"):
        assert "STG.E.128" in funcs[_one(funcs, needle)[0]], needle


def test_no_spills_in_row_kernels(sass):
    funcs, usage = sass
    # (grid_fourier_kernel keeps 32 bytes of stack: sinf/cosf's Payne-Hanek branch, unreachable for fp16 arguments)
    for needle in ("layernorm_kernelILi4E", "lnpost_dot_kernelILi4E", "qk_norm_kernel", "cfg_euler_kernel"):
        name = _one(funcs, needle)[0]
        assert usage[name][1] == 0, f"{name}: {usage[name][1]} bytes of stack"


def test_marching_cubes_emit_has_no_output_atomics(sass):
    funcs, _ = sass
    for needle in ("mc_vertex_kernel", "mc_face_kernel"):
        body = funcs[_one(funcs, needle)[0]]
        assert "ATOMG" not in body and "RED." not in body, needle + ": output order must come from the scans"
