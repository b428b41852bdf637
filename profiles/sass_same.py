"""Is every device function of one libdronecu.so compiled to the same SASS in another?

    python profiles/sass_same.py OLD.so NEW.so

Splits `cuobjdump -sass` of both libraries into functions and compares every function of OLD with its counterpart in NEW,
instruction for instruction and encoding for encoding (the scheduling control bits included).  A kernel template that
gained a trailing `bool` parameter defaulting to false (the rollout kernels' TIMEOUT, DESIGN.md section 11) has a new
mangled name: OLD's `<R, N>` is matched with NEW's `<R, N, false>`.  Exit status 0 when all functions match.
"""
from __future__ import annotations

import re
import subprocess
import sys

CUOBJDUMP = "/usr/local/cuda/bin/cuobjdump"
EXTENDED = ("policy_rollout_kernel", "policy_rollout_warp_kernel", "policy_rollout_tc_kernel")


def functions(path: str) -> dict:
    text = subprocess.run([CUOBJDUMP, "-sass", path], check=True, capture_output=True, text=True).stdout
    out, name = {}, None
    for line in text.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = m.group(1)
            out[name] = []
        elif name is not None and re.match(r"\s*/\*", line):      # address, instruction and its encoding (control bits)
            out[name].append(line.strip())
    return out


def counterpart(name: str) -> str:
    if any(k in name for k in EXTENDED):
        return re.sub(r"I(Lb[01]ELb[01]E)EEv", r"I\1Lb0EEEv", name)
    return name


def main(old: str, new: str) -> int:
    a, b = functions(old), functions(new)
    bad = 0
    for name, body in a.items():
        other = b.get(counterpart(name))
        if other != body:
            bad += 1
            print(f"DIFFERS: {name}" if other is not None else f"MISSING: {name}")
    print(f"{len(a) - bad} of {len(a)} functions identical ({len(b) - len(a)} new functions)")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main(*sys.argv[1:3]))
