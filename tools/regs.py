#!/usr/bin/env python
"""Registers / spills per step, rollout and reset kernel from a `nvcc -Xptxas -v` log (stdin or file)."""
import re, sys
t = open(sys.argv[1]).read() if len(sys.argv) > 1 else sys.stdin.read()
pat = re.compile(r"Compiling entry function '([^']+)'[^\n]*\n[^\n]*\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads\n[^\n]*Used (\d+) registers")
for m in pat.finditer(t):
    # G = lanes per env (thread-per-env kernels: 1); rollouts: Philox or caller-supplied actions
    k = re.search(r'\d+((?:simple_)?(?:step|rollout|reset)(?:_call|_tpe)?_kernel)(?:I(?:Li(\d+)E)?(?:Lb([01])E)?E)?', m.group(1))
    if k:
        acts = {"0": "philox", "1": "caller"}.get(k.group(3), "")
        print(f"{k.group(1):22s} G={k.group(2) or '1':>2s} {acts:6s} regs={m.group(5):>3s} spill_st={m.group(3):>3s} spill_ld={m.group(4):>3s}")
