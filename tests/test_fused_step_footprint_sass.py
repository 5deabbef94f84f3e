"""CPU check (no GPU): the instruction stream of the single-GPU flat step carries no grid-barrier fault path.

Every phase of the step runs once per launch and the L2 flush between training steps evicts the kernel's code, so
each instruction on the way through the kernel body is fetched again on every step.  The barrier time-out (globaltimer
sampling, fault-code store, system fence, trap) therefore lives in one out-of-line subroutine placed after the body,
and the body stays below a size ceiling.  The only traps left in the body are the bounded mbarrier waits, whose
one-instruction trap is smaller than a call would be."""
import os
import re
import shutil
import subprocess
import tempfile

import multimodal_baby_b200 as cv

SINGLE = "_ZN4cvcl5fused16flat_step_kernelILb0EEEvNS0_8StepMapsENS0_10StepParamsE"
BODY_CEILING = 9100          # instructions in the kernel body: 8952 with nvcc 12.9 (9683 with the time-out inline)
INSN = re.compile(r"^\s+/\*[0-9a-f]+\*/\s+(.*?)\s*;")


def _tool(name):
    return shutil.which(name) or os.path.join("/usr/local/cuda/bin", name)


def _kernel_and_subroutines(sym):
    """(instructions of the kernel body, {subroutine: instructions}) from the section of kernel `sym`"""
    tmp = tempfile.mkdtemp(prefix="footprint_sass_")
    try:
        subprocess.run([_tool("cuobjdump"), "-xelf", "all", os.path.abspath(cv._cabi.LIB_PATH)], cwd=tmp,
                       check=True, capture_output=True)
        cubin = [f for f in os.listdir(tmp) if f.endswith(".cubin") and "sm_100" in f][0]
        text = subprocess.run([_tool("nvdisasm"), "-c", os.path.join(tmp, cubin)], check=True,
                              capture_output=True, text=True).stdout
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    sect = text.split("//--------------------- .text.%s " % sym, 1)[1].split("\n//----", 1)[0]
    funcs, cur = {}, None
    for line in sect.splitlines():
        m = re.match(r"\s+\.type\s+([^,]+),@function", line)
        if m:
            cur = funcs.setdefault(m.group(1), [])
            continue
        m = INSN.match(line)
        if m and cur is not None:
            cur.append(m.group(1))
    body = funcs.pop(sym)
    return body, funcs


def test_single_gpu_step_body_has_no_barrier_fault_path():
    cv._cabi.load()                                  # builds the library if it is missing or stale
    body, subs = _kernel_and_subroutines(SINGLE)
    # each trap left in the body ends a bounded mbarrier wait: the try-wait probe is a few instructions before it
    for i, ins in enumerate(body):
        if "BPT.TRAP" in ins:
            assert any("SYNCS.PHASECHK" in x for x in body[max(0, i - 6):i]), \
                "trap at instruction %d of the body is not an mbarrier wait's" % i
    assert not any("MEMBAR.SC.SYS" in x for x in body), "a fault path's system fence is inline in the body"
    cold = [k for k in subs if "grid_wait_cold" in k]
    assert len(cold) == 1, "no out-of-line barrier time-out subroutine: %s" % sorted(subs)
    cold_ins = subs[cold[0]]
    for mnemonic in ("GLOBALTIMER", "ATOMG.E.EXCH", "MEMBAR.SC.SYS", "BPT.TRAP"):
        assert any(mnemonic in x for x in cold_ins), "the barrier time-out subroutine lacks %s" % mnemonic
    calls = [x for x in body if x.startswith("CALL") and "grid_wait_cold" in x]
    assert len(calls) >= 5, "the grid barriers do not reach the time-out subroutine (%d calls)" % len(calls)
    assert len(body) <= BODY_CEILING, "kernel body of %d instructions, ceiling %d" % (len(body), BODY_CEILING)
