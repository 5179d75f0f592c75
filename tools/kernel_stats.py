#!/usr/bin/env python
"""What the BUILT step kernels execute, counted from their SASS (cuobjdump of libmvrl.so).

    python tools/kernel_stats.py [libmvrl.so]          -> JSON on stdout
    kernel_stats.collect(lib_path) -> dict             (used by __graft_entry__.build(), which writes
                                                        marinevehiclereinforcementlearning_b200/kernel_stats.json;
                                                        bench.py reads that file for roofline.executed_*)

Per kernel: the instruction mix of the RK4 sub-step loop (the largest backward branch; rare-path blocks skipped by a
forward branch over more than 64 instructions are dropped), the floating-point operations one trip executes per
environment (FFMA2 = 2 lanes x 2 flop, FMUL2 / FADD2 = 2 x 1, scalar FFMA / DFMA = 2, other scalar FP = 1; packed
kernels carry two environments per thread), the same count for the straight-line code outside the loop (prologue +
epilogue, out-of-line rare paths excluded as far as they sit behind long forward branches), and a lower bound on
FMA-pipe cycles per trip (a packed instruction holds the pipe 2 cycles, 3 when all three sources are vector
registers: tools/ffma_regs.cu).  This replaces the hand-pasted "933 n_sub + 100" of round 1: the numbers follow the
kernel.
"""
import collections
import json
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEFAULT_LIB = os.path.join(ROOT, "marinevehiclereinforcementlearning_b200", "libmvrl.so")

# name -> (mangled-name regex, environments per thread)
# the fp32 force / set-point kernels the default vehicle runs are the instantiations with compile-time constants (last
# template argument CONSTP = true); "_runtime_constants" = the same kernel reading the constants from the kernel argument
KERNELS = {
    "rov6_step_f32x2_rpm": (r"rov6_step_kernelINS_2F2ELi0ELb1ELb0ELb0E", 2),
    "rov6_step_f32x2_force": (r"rov6_step_kernelINS_2F2ELi1ELb1ELb0ELb1E", 2),
    "rov6_step_f32x2_setpoint": (r"rov6_step_kernelINS_2F2ELi2ELb1ELb0ELb1E", 2),
    "rov6_step_f32x2_setpoint_runtime_constants": (r"rov6_step_kernelINS_2F2ELi2ELb1ELb0ELb0E", 2),
    "rov6_step_f64_rpm": (r"rov6_step_kernelIdLi0ELb1ELb0", 1),
    "rov6_step_f64_setpoint": (r"rov6_step_kernelIdLi2ELb1ELb0", 1),
}

PACKED = {"FFMA2": 4, "FMUL2": 2, "FADD2": 2}
SCALAR = {"FFMA": 2, "FMUL": 1, "FADD": 1, "DFMA": 2, "DMUL": 1, "DADD": 1, "FMNMX": 1, "FSET": 1, "FSETP": 1, "FSEL": 1, "DSETP": 1, "DMNMX": 1}
# min / max / compare / select count as one flop each in SURVEY.md 8(d)'s convention ("every add/mul/abs/min/max/compare-select = 1")


def _functions(lib):
    names = subprocess.run(["cuobjdump", "-elf", lib], capture_output=True, text=True).stdout
    return sorted(set(re.findall(r"_ZN4mvrl\w+", names)))


def _sass(lib, fn):
    out = subprocess.run(["cuobjdump", "-sass", "-fun", fn, lib], capture_output=True, text=True).stdout
    ins = []
    for line in out.splitlines():
        m = re.match(r"\s+/\*([0-9a-f]{4,6})\*/\s+(.*?);", line)
        if m:
            ins.append((int(m.group(1), 16), m.group(2).strip()))
    return ins


def _flops(instrs):
    mix, packed3, cycles, flop = collections.Counter(), 0, 0, 0
    for _, t in instrs:
        t = re.sub(r"^@!?U?P\d+\s+", "", t)
        op = t.split()[0].split(".")[0]
        mix[op] += 1
        if op in PACKED:
            srcs = [o.strip() for o in t.split(None, 1)[1].split(",")[1:]]
            nreg = sum(1 for o in srcs if re.match(r"^[-|]*R\d+", o))
            packed3 += nreg == 3
            cycles += 3 if nreg == 3 else 2
            flop += PACKED[op]
        elif op in SCALAR:
            flop += SCALAR[op]
            if op in ("FFMA", "FMUL", "FADD"):
                cycles += 1
    return mix, packed3, cycles, flop


def analyse(lib, pattern, envs_per_thread):
    fn = [f for f in _functions(lib) if re.search(pattern, f)]
    if not fn:
        return None
    fn = min(fn, key=len)
    ins = _sass(lib, fn)
    lo = hi = None
    for a, t in ins:
        m = re.search(r"BRA(?:\.U)? !?U?P\d+, 0x([0-9a-f]+)", t)
        if m and int(m.group(1), 16) < a and (hi is None or a - int(m.group(1), 16) > hi - lo):
            lo, hi = int(m.group(1), 16), a
    if lo is None:
        return None
    rare = []
    for a, t in ins:
        m = re.search(r"@!?U?P\d BRA(?:\.U)? 0x([0-9a-f]+)", t)
        if m and int(m.group(1), 16) - a > 0x400:
            rare.append((a + 0x10, int(m.group(1), 16)))
    skip = lambda a: any(x <= a < y for x, y in rare)
    loop = [(a, t) for a, t in ins if lo <= a <= hi and not skip(a)]
    end = next((a for a, t in ins if a > hi and t.startswith("EXIT")), ins[-1][0])   # code after the first EXIT past the loop = out-of-line paths
    outside = [(a, t) for a, t in ins if (a < lo or hi < a <= end) and not skip(a)]
    mix, p3, cyc, flop = _flops(loop)
    omix, _, _, oflop = _flops(outside)
    alu = sum(mix[o] for o in ("FMNMX", "FSET", "FSETP", "FSEL", "LOP3", "MOV", "IMAD", "IADD3", "SHF", "PRMT", "CS2R", "ISETP", "SEL", "VIADD"))
    fma = sum(mix[o] for o in ("FFMA2", "FMUL2", "FADD2", "FFMA", "FMUL", "FADD"))
    return {"function": fn, "envs_per_thread": envs_per_thread,
            "loop_bytes": hi - lo + 16, "loop_instructions_per_trip": len(loop), "outside_instructions": len(outside),
            "loop_mix": dict(mix.most_common(16)), "packed_three_register": p3, "fma_pipe_cycles_per_trip_min": cyc,
            "loop_fma_pipe_instructions": fma, "loop_alu_pipe_instructions": alu,
            "flop_per_env_per_substep": flop / envs_per_thread, "flop_per_env_outside_loop": oflop / envs_per_thread}


def collect(lib=DEFAULT_LIB):
    out = {"library": os.path.relpath(lib, ROOT) if lib.startswith(ROOT) else lib, "kernels": {}}
    for name, (pat, ept) in KERNELS.items():
        r = analyse(lib, pat, ept)
        if r is not None:
            out["kernels"][name] = r
    return out


if __name__ == "__main__":
    print(json.dumps(collect(sys.argv[1] if len(sys.argv) > 1 else DEFAULT_LIB), indent=1))
