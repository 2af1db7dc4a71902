"""Static checks on the built SASS (no GPU): the Blackwell-specific instructions the design relies on are there, and the
column-walk forward does not wait for its own B / C prefetch (profiles/r2zz_fwd_prefetch_wait.md)."""
import os
import shutil
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BUILD = os.path.join(ROOT, "medical_image_analysis_b200", "build")
sys.path.insert(0, os.path.join(ROOT, "tools"))

needs_objects = pytest.mark.skipif(shutil.which("cuobjdump") is None or not os.path.exists(os.path.join(BUILD, "scan_fwd_bf16.o")),
                                   reason="needs cuobjdump and the in-tree objects (python -c 'import __graft_entry__ as g; g.build()')")

FWD = "_ZN3mia16ss_fwd_cw_kernelI13__nv_bfloat16Lb1ELb0ELi%dEEEv14CUtensorMap_stS2_S2_NS_9CwFwdArgsE"


def _prefetch_waiters(ins, after, slot):
    """Arithmetic / branch instructions after index `after` that wait for scoreboard slot `slot`."""
    import sass_waits
    out = []
    for _, t, hi in ins[after + 1:]:
        toks = t.split()
        op = (toks[1] if toks[0].startswith("@") else toks[0]).split(".")[0]
        if sass_waits.ctrl(hi)["wait"] & (1 << slot) and op in ("FMUL2", "FFMA2", "FADD2", "FMUL", "FFMA", "FADD", "BRA", "MUFU", "FMNMX"):
            out.append(t)
    return out


@needs_objects
@pytest.mark.parametrize("g", [1, 4])
def test_forward_does_not_wait_for_its_own_prefetch(g):
    import sass_waits
    ins = sass_waits.load(os.path.join(BUILD, "scan_fwd_bf16.o"), FWD % g)
    assert len(ins) > 1000
    pre = [(i, sass_waits.ctrl(hi)["wbar"]) for i, (_, t, hi) in enumerate(ins) if t.startswith("LDG.E.U16")]
    assert pre, "the B / C prefetch loads are gone?"
    slot = pre[-1][1]
    assert all(s == slot for _, s in pre)
    # the parameter loads are settled by a LOP3 with a uniform register right after they are issued ...
    settles = [t for _, t, hi in ins if t.startswith("LOP3.LUT") and ", UR" in t and "0x3c" in t]
    assert len(settles) >= 2, settles
    # ... so between the last prefetch load and the end of the window body nothing arithmetic waits for the prefetch's slot
    # (before the fix: the window's first FMUL2 with A, or for g > 1 the branch into the column loop)
    offenders = _prefetch_waiters(ins, pre[-1][0], slot)
    assert not offenders, offenders


@needs_objects
def test_planner_object_compiles_no_scan_kernel():
    """scan_api.cu reaches the kernels only through the launchers in scan_args.h: its object holds the finalize kernel (one
    per dtype) and no second copy of a kernel that the per-dtype objects instantiate."""
    out = subprocess.run(["cuobjdump", "-sass", os.path.join(BUILD, "scan_api.o")], capture_output=True, text=True, check=True).stdout
    kernels = [l.split("Function :", 1)[1].strip() for l in out.splitlines() if "Function :" in l]
    assert len(kernels) == 3 and all("ss_finalize_kernel" in k for k in kernels), kernels


@needs_objects
def test_blackwell_instructions_present():
    def count(obj, needle):
        out = subprocess.run(["cuobjdump", "-sass", os.path.join(BUILD, obj)], capture_output=True, text=True, check=True).stdout
        return out.count(needle)
    assert count("scan_fwd_bf16.o", "UTMALDG.2D") > 0 and count("scan_fwd_bf16.o", "UTMASTG.2D") > 0      # tensor-map TMA
    assert count("scan_bwd_bf16.o", "UTMALDG.2D") > 0 and count("scan_bwd_bf16.o", "FFMA2") > 0          # + packed f32x2
    assert count("gemm_tcgen05.o", "UTCHMMA") > 0 and count("gemm_tcgen05.o", "LDTM") > 0                # tcgen05.mma / tcgen05.ld
