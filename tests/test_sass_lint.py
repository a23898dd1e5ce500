"""Static checks on the SASS of the built library (cuobjdump, no GPU).

* the Blackwell instructions the design claims are really there (tcgen05 MMA / TMEM load / commit, TMA tensor
  and bulk copies, st.async, packed FFMA2);
* two code-generation pitfalls found with the profiler in round 1 stay fixed:
    - a tcgen05.mma / TMA issue whose operands the compiler cannot prove warp-uniform is wrapped in an
      ELECT + R2UR.BROADCAST + BRA.U.ANY loop (~55 cycles per MMA instead of ~16): kernels that issue UTCHMMA or
      UTMALDG must contain no BRA.U.ANY;
    - a shared-memory pointer aligned through an integer round trip becomes generic (LD.E / ST.E instead of
      LDS / STS) and its loads queue behind outstanding global loads: the tensor-core kernels must not contain
      generic loads/stores at all (their global traffic is LDG/STG).
"""
import re
import shutil
import subprocess

import pytest

from b200rnn import _lib

cuobjdump = shutil.which("cuobjdump") or shutil.which("/usr/local/cuda/bin/cuobjdump")
pytestmark = pytest.mark.skipif(cuobjdump is None, reason="cuobjdump not available")


@pytest.fixture(scope="module")
def functions():
    txt = subprocess.run([cuobjdump, "-sass", _lib.LIB_PATH], capture_output=True, text=True, timeout=300).stdout
    out, name = {}, None
    for line in txt.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            name = m.group(1)
            out[name] = []
        elif name is not None:
            m = re.search(r"\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_.]*)", line)
            if m:
                out[name].append(m.group(1))
    assert out, "cuobjdump produced no functions"
    return out


def _has(ops, prefix):
    return any(o.startswith(prefix) for o in ops)


def test_expected_blackwell_instructions_are_present(functions):
    all_ops = [o for ops in functions.values() for o in ops]
    for prefix, what in [("UTCHMMA", "tcgen05.mma"), ("LDTM", "tcgen05.ld"), ("UTCBAR", "tcgen05.commit"),
                         ("UTMALDG", "TMA tensor load"), ("UBLKCP", "TMA bulk copy"), ("STAS", "st.async"),
                         ("FFMA2", "packed fp32 FMA"), ("SYNCS", "mbarrier")]:
        assert _has(all_ops, prefix), f"no {prefix} ({what}) in the library"


def test_tensor_core_issue_stays_on_the_uniform_datapath(functions):
    tc = {n: ops for n, ops in functions.items() if _has(ops, "UTCHMMA") or _has(ops, "UTMALDG")}
    assert len(tc) >= 1, sorted(tc)   # the 3xTF32 GEMM
    for name, ops in tc.items():
        assert not _has(ops, "BRA.U.ANY"), f"{name}: tcgen05 / TMA issue inside a register-broadcast loop"


def test_tensor_core_kernels_keep_the_shared_state_space(functions):
    for name, ops in functions.items():
        if _has(ops, "UTCHMMA"):
            generic = [o for o in ops if re.fullmatch(r"(LD|ST)(\.E)?(\.\d+)?", o)]
            assert not generic, f"{name}: generic loads/stores {sorted(set(generic))}"
            assert _has(ops, "LDS") or _has(ops, "STS"), name
