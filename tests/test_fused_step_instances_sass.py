"""CPU check (no GPU): both instances of the one-kernel flat step in the built library are the real tcgen05 / TMA
kernel, and only the sharded instance carries the cross-rank barrier (system-scope release / acquire on the peer
flag words).  The single-GPU instance is the one `cvcl_flat_step_fused` launches; it is compiled without that code."""
import re
import subprocess

import multimodal_baby_b200 as cv

SHARDED = "_ZN4cvcl5fused16flat_step_kernelILb1EEEvNS0_8StepMapsENS0_10StepParamsE"
SINGLE = "_ZN4cvcl5fused16flat_step_kernelILb0EEEvNS0_8StepMapsENS0_10StepParamsE"


def _functions():
    sass = subprocess.run(["cuobjdump", "-sass", cv._cabi.LIB_PATH], capture_output=True, text=True).stdout
    parts = re.split(r"\n\s*Function : (\S+)", sass)
    return dict(zip(parts[1::2], parts[2::2]))


def test_both_flat_step_instances_are_tcgen05_tma_kernels():
    cv._cabi.load()                                  # builds the library if it is missing or stale
    fns = _functions()
    for name in (SHARDED, SINGLE):
        assert name in fns, "%s not in the library" % name
        for mnemonic in ("UTCHMMA", "LDTM", "UTMALDG.2D", "UTMASTG.2D", "SYNCS.PHASECHK"):
            assert mnemonic in fns[name], "%s lacks %s" % (name, mnemonic)
    for mnemonic in ("STG.E.STRONG.SYS", "LDG.E.STRONG.SYS"):
        assert mnemonic in fns[SHARDED], "sharded instance lacks %s" % mnemonic
        assert mnemonic not in fns[SINGLE], "single-GPU instance still carries the cross-rank barrier (%s)" % mnemonic
