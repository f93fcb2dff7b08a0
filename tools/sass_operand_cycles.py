"""Static FMA-pipe cost of the substep loop of each step kernel, read from the SASS (no GPU needed).

    python tools/sass_operand_cycles.py [path/to/libvine_b200.so] [--json]

The free-space step kernel is bound by the register-file operand reads of its FP32 instructions (profiles/README.md, r02a
probe: 256 B/clk of register-file read per SM sub-partition feeds two 32-lane f32 operands per cycle, so an FFMA that reads
three registers occupies the FMA pipe 1.5 cycles and anything reading at most two, 1 cycle). Nsight Compute's pipe metrics
are not the only way to see this: the cost is fixed by the instructions of the loop, so it can be counted from
`cuobjdump -sass`.

The substep loop of a kernel is taken as the innermost backward branch whose body holds the LDL^T's reciprocals (at least
five MUFU.RCP). The free-space loops are branch-free, so their static count is what every substep executes; the contact
variant's loop also holds its narrow phase, which runs only where something touches.

Per loop it reports:
  fp32      FFMA / FMUL / FADD (packed FFMA2 / FMUL2 / FADD2 counted apart), FLOPs (2 per FMA and lane)
  ffma3     FFMAs (FFMA2s) whose three sources are all registers
  reads     register-file operand reads of the FP32 instructions: a register source (RZ excluded) is read unless the previous
            instruction flagged the same register with .reuse in the same operand slot; a packed .F32x2 source reads two
  cycles    FMA-pipe operand cycles: per FP32 instruction max(issue cycles, reads / 2), issue cycles 1 (scalar) or 2 (packed)
  mufu      MUFU instructions by function
"""
import argparse
import collections
import json
import os
import re
import shutil
import subprocess
import sys

LIB = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "vine_robot_isaacgymenvs_b200", "csrc", "libvine_b200.so")
KERNELS = {  # mangled name -> short name
    "_Z16vine_step_kernelILb0EEv10VineParams8StepArgs": "vine_step_kernel<false>",
    "_Z17vine_step2_kernel10VineParams8StepArgs": "vine_step2_kernel",
    "_Z20vine_step_far_kernel10VineParams8StepArgs": "vine_step_far_kernel",
    "_Z16vine_step_kernelILb1EEv10VineParams8StepArgs": "vine_step_kernel<true>",
    "_Z20vine_simulate_kernelILb0EEv10VineParamsl14VineSimulateIO": "vine_simulate_kernel<false>",
}
FP32 = {"FFMA": 1, "FMUL": 1, "FADD": 1, "FFMA2": 2, "FMUL2": 2, "FADD2": 2}
INST = re.compile(r"/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;")
REG = re.compile(r"^[-!|]*(R\d+)(\.reuse)?")


def sass_functions(lib):
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    out = subprocess.run([cuobjdump, "-sass", lib], capture_output=True, text=True, check=True).stdout
    funcs, name = {}, None
    for line in out.splitlines():
        if "Function :" in line:
            name = line.split("Function :")[1].strip()
            funcs[name] = []
        elif name is not None:
            m = INST.search(line)
            if m:
                funcs[name].append((int(m.group(1), 16), m.group(2)))
    return funcs


def parse(text):
    """'@P0 FFMA R1, R2.reuse, -R3, c[0x0][0x10]' -> ('FFMA', ['R1', 'R2.reuse', '-R3', 'c[0x0][0x10]'])"""
    text = re.sub(r"^@!?U?P\w+\s+", "", text)
    op, _, rest = text.partition(" ")
    return op, [t.strip() for t in rest.split(",")] if rest else []


def substep_loop(insts):
    """(start, end) index range of the innermost backward branch holding >= 5 MUFU.RCP, or None"""
    addr_index = {a: i for i, (a, _) in enumerate(insts)}
    loops = []
    for i, (a, text) in enumerate(insts):
        op, ops = parse(text)
        if op.startswith("BRA") and ops:
            m = re.search(r"0x([0-9a-f]+)", ops[-1])
            if m and int(m.group(1), 16) <= a and int(m.group(1), 16) in addr_index:
                loops.append((addr_index[int(m.group(1), 16)], i))
    rcp = [sum(parse(t)[0] == "MUFU.RCP" for _, t in insts[s:e + 1]) for s, e in loops]
    cands = [(e - s, s, e) for (s, e), r in zip(loops, rcp) if r >= 5]
    return min(cands)[1:] if cands else None


def count(insts):
    c = collections.Counter()
    mufu = collections.Counter()
    prev = []   # (register, reuse flag) per operand slot of the previous instruction
    for _, text in insts:
        op, ops = parse(text)
        base = op.split(".")[0]
        srcs = ops[1:]
        slots = [REG.match(t) for t in srcs]
        if base == "MUFU":
            mufu[op.split(".")[1]] += 1
        if base in FP32:
            c[base] += 1
            regs = [m for m in slots if m and m.group(1) != "RZ"]
            if base in ("FFMA", "FFMA2") and len(regs) == 3:
                c["ffma3"] += 1
            reads = 0
            for k, (m, t) in enumerate(zip(slots, srcs)):
                if not m or m.group(1) == "RZ":
                    continue
                if k < len(prev) and prev[k] == (m.group(1), True):
                    c["reuse_hits"] += 1
                    continue
                reads += 2 if (FP32[base] == 2 and ".F32x2" in t) else 1
            c["reads"] += reads
            c["cycles"] += max(FP32[base], reads / 2)
            lanes = FP32[base]
            c["flops"] += lanes * (2 if base.startswith("FFMA") else 1)
        c["instructions"] += 1
        prev = [(m.group(1), bool(m.group(2))) if m else None for m in slots]
    c["fp32"] = sum(c[k] for k in FP32)
    return c, mufu


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("lib", nargs="?", default=LIB)
    ap.add_argument("--json", action="store_true", help="one JSON object instead of the table")
    args = ap.parse_args()
    funcs = sass_functions(args.lib)
    result = {}
    for mangled, short in KERNELS.items():
        insts = funcs.get(mangled)
        if insts is None:
            sys.exit(f"{short} ({mangled}) not in {args.lib}")
        loop = substep_loop(insts)
        if loop is None:
            sys.exit(f"{short}: no loop with the LDL^T's reciprocals found")
        s, e = loop
        c, mufu = count(insts[s:e + 1])
        result[short] = {"loop": [hex(insts[s][0]), hex(insts[e][0])], **{k: c[k] for k in
                         ("instructions", "fp32", "FFMA", "FMUL", "FADD", "FFMA2", "FMUL2", "FADD2", "ffma3", "reads",
                          "reuse_hits", "cycles", "flops")}, "mufu": dict(sorted(mufu.items()))}
    if args.json:
        print(json.dumps(result, indent=1))
        return
    print(f"{os.path.relpath(args.lib)}: substep loop of each step kernel (static SASS count per loop iteration)")
    hdr = f"{'kernel':28s} {'loop':>15s} {'inst':>5s} {'fp32':>5s} {'FFMA':>5s} {'FMUL':>5s} {'FADD':>5s} {'ffma3':>5s} " \
          f"{'reads':>5s} {'reuse':>5s} {'cycles':>6s} {'flops':>5s}  mufu"
    print(hdr)
    for short, r in result.items():
        packed = r["FFMA2"] + r["FMUL2"] + r["FADD2"] > 0
        f = lambda k: r[k + "2"] if packed else r[k]  # noqa: E731
        print(f"{short:28s} {r['loop'][0] + '-' + r['loop'][1]:>15s} {r['instructions']:5d} {r['fp32']:5d} {f('FFMA'):5d} "
              f"{f('FMUL'):5d} {f('FADD'):5d} {r['ffma3']:5d} {r['reads']:5d} {r['reuse_hits']:5d} {r['cycles']:6.1f} "
              f"{r['flops']:5d}  " + " ".join(f"{k} {v}" for k, v in r["mufu"].items()) + ("  (packed: FFMA2/FMUL2/FADD2)" if packed else ""))


if __name__ == "__main__":
    main()
