"""Source-level rules of the sweep kernels that the hardware taught (DESIGN.md section 4, round 2), checked without a
GPU so that a later edit cannot quietly undo them.

csrc/sell.cu issues the loads of CONSTANT data (matrix stream, inverse diagonal, dense inverse) before
``griddepcontrol.wait`` and everything a kernel of the chain writes after it.  ptxas moves non-coherent loads
(``__ldg`` / loads through ``const T *__restrict__`` kernel parameters -> LDG.CONSTANT) freely across the wait: it sank
early loads below it and -- the bug that produced wrong sweeps on the GPU -- hoisted the gathers of the iterate above
it.  So: vectors are read with plain loads, ``__ldg`` is reserved for constant data, and only constant pointers may be
``__restrict__`` kernel parameters."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SELL = os.path.join(ROOT, "control_b200", "csrc", "sell.cu")

# what __ldg may be applied to in sell.cu: stencil / dictionary tables, per-entry codes, the inverse diagonal, the
# dense inverse
LDG_ALLOWED = (r"__ldg\(&st\[", r"__ldg\(code \+", r"__ldg\(dinv\.x \+", r"__ldg\(A \+")
RESTRICT_ALLOWED = ("dinv", "A")


def test_ldg_only_on_constant_data():
    src = open(SELL).read()
    code = "\n".join(l for l in src.splitlines() if not l.lstrip().startswith("//"))
    for m in re.finditer(r"__ldg\([^;]*", code):
        text = m.group(0)
        for part in re.findall(r"__ldg\([^,;]*", text):
            assert any(re.match(p, part) for p in LDG_ALLOWED), f"__ldg on something that may not be constant: {part}"


def test_only_constant_pointers_are_restrict_kernel_parameters():
    src = open(SELL).read()
    for m in re.finditer(r"const\s+double\s*\*\s*__restrict__\s+(\w+)", src):
        assert m.group(1) in RESTRICT_ALLOWED, f"const double *__restrict__ {m.group(1)}: vectors must not be restrict"
    assert "double *__restrict__" not in re.sub(r"const\s+double\s*\*\s*__restrict__", "", src)


@pytest.mark.skipif(shutil.which("cuobjdump") is None and not os.path.exists("/usr/local/cuda/bin/cuobjdump"),
                    reason="needs cuobjdump")
def test_early_loads_precede_the_wait_in_the_sass():
    """In the built object every sweep kernel triggers its dependents (PREEXIT), and on the one-GPU path of the hot
    kernels plain loads (the early matrix loads) stand BEFORE the first griddepcontrol.wait (ACQBULK) that follows the
    multi-GPU prologue -- i.e. the early loads did not sink -- and no LDG.CONSTANT stands before that wait."""
    obj = os.path.join(ROOT, "control_b200", "lib", "obj", "sell.o")
    if not os.path.exists(obj):
        pytest.skip("control_b200/lib/obj/sell.o not built")
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    out = subprocess.run([tool, "-sass", obj], capture_output=True, text=True, timeout=300).stdout
    funcs = re.split(r"\n\s*Function : ", out)[1:]
    hot = [f for f in funcs if re.match(r"\S*(sell_cheb_kernel|sell_spmv_kernel|sell_first2_kernel|csrv_cheb_kernel|"
                                        r"csrv_spmv_kernel|csrv_first2_kernel|dense_gemv_kernel)", f)]
    assert len(hot) >= 20
    for f in hot:
        name = f.split("\n", 1)[0]
        ops = re.findall(r"/\*[0-9a-f]{4}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", f)
        assert "PREEXIT" in ops, name
        waits = [i for i, o in enumerate(ops) if o == "ACQBULK"]
        assert waits, name
        # the last wait of the listing belongs to the regular (non-push) path or to a later chunk; between the trigger
        # and the FIRST wait only the epoch word may be loaded -- never a read-only load
        first = waits[0]
        assert not any(o.startswith("LDG") and "CONSTANT" in o for o in ops[:first]), name
        # and somewhere a plain load precedes a wait directly (the early matrix loads were kept in place)
        assert any(any(o.startswith("LDG") and "CONSTANT" not in o for o in ops[(waits[k - 1] if k else 0):w])
                   for k, w in enumerate(waits)), name


CSRC = os.path.join(ROOT, "control_b200", "csrc")


def test_device_resources_are_released_only_by_their_owning_types():
    """Per-call device resources are scoped (csrc/common.cuh): scratch vectors are leased from a ScratchPool and given
    back by the lease, events are destroyed by an EventPair.  No other file destroys an event or pushes to / pops from
    a pool's free list by hand, and the retired get / put functions stay retired -- releasing by hand leaked on the
    error paths."""
    owner = "common.cuh"
    names = sorted(f for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".cpp", ".h")))
    assert owner in names
    for name in names:
        src = open(os.path.join(CSRC, name)).read()
        for retired in ("ctl_scratch_get", "ctl_scratch_put", "outer_get"):
            assert not re.search(rf"\b{retired}\b", src), f"{name}: {retired}"
        if name == owner:
            continue
        assert "cudaEventDestroy" not in src, f"{name}: events are destroyed by EventPair ({owner})"
        assert not re.search(r"\b(pool|free_)\s*\.\s*(push_back|pop_back)\b", src), \
            f"{name}: scratch vectors are leased with ScratchPool::take ({owner})"
