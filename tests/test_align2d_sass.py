"""align2d_kernel must contain no fused multiply-add: the reference computes every product and sum of Align2D separately, and
ptxas contracts a paired FMUL2 feeding a paired FADD2 into FFMA2 even when both come from the _rn intrinsics. Reads the SASS of
the built library, so it needs no GPU."""
import re
import shutil
import subprocess


def _functions(sass):
    """{mangled name: [instruction text]} of a cuobjdump -sass listing"""
    out, cur = {}, None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = out.setdefault(m.group(1), [])
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4}\*/\s+(.*?);", line)
        if m and cur is not None:
            cur.append(m.group(1).strip())
    return out


def _opcode(ins):
    return re.sub(r"^@!?U?P\w+\s+", "", ins).split()[0].split(".")[0]


def test_align2d_kernel_has_no_fma(built):
    from dsdtm_b200 import capi
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    r = subprocess.run([tool, "-sass", capi.lib_path()], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    fns = {k: v for k, v in _functions(r.stdout).items() if "align2d_kernel" in k}
    assert len(fns) == 1, sorted(fns)
    ins = next(iter(fns.values()))
    ops = [_opcode(i) for i in ins]
    # the kernel does run paired fp32: without it this test would guard nothing
    assert "FMUL2" in ops and "FADD2" in ops
    assert "FFMA2" not in ops
    # the one FFMA allowed is the fp64 division's range test 0 * x + y (an exact move, not a contracted product)
    fused = [i for i, o in zip(ins, ops) if o == "FFMA" and not re.match(r"(@!?P\w+\s+)?FFMA\S*\s+R\d+,\s*RZ,", i)]
    assert not fused, fused
