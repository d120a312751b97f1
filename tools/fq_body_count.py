#!/usr/bin/env python3
"""Static instruction count of the out-of-line field multiplier bodies (fq_mul_ool, fq_sqr_ool) as the curve kernel
k_curve_p<0> and the challenge kernel k_run<OP_CHALLENGE> call them, priced with the issue model of DESIGN 4.0
(4.0 sub-partition cycles per IMAD.WIDE, 1.29 per other instruction).  The squaring is also split by source line into its
product part (the limb products of a^2 and their carries) and the rest (Montgomery reduction, final addition and
subtraction, call overhead).

usage: tools/fq_body_count.py [--lib LIB --src FQ_CUH] [--json OUT]
Without --lib the library is compiled into a temporary directory with the flags of __graft_entry__.build().  --src names
the fq.cuh that LIB was built from (default: this tree's), whose lines the split reads."""
import argparse
import collections
import glob
import json
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KERNELS = {"k_curve_p<0>": "k_curve_pILi0E", "k_run<OP_CHALLENGE>": "k_runILi18E"}
BODIES = ("fq_mul_ool", "fq_sqr_ool")
WIDE_CYCLES, OTHER_CYCLES = 4.0, 1.29
# The split goes by the function of fq.cuh that holds an instruction's innermost source line (the "inlined at" chains
# ptxas records are not reliable; the innermost line is).  Reduction, final addition / subtraction and call overhead:
REST_FUNCS = {"mont_reduce16", "blk_fold_red_odd", "blk_red_even_q", "blk_sqr_red_row", "add8", "add8c", "sub8",
              "cond_sub_p", "fq_sqr_ool"}
# ... and lines of fq_sqr_inl itself that belong to the product (parent: the doubling shift; now: the limbs of 2a)
PRODUCT_LINE = re.compile(r"<< 1|funnelshift")
FUNC_DEF = re.compile(r"^(?:SB_HD|static __device__|template).*?\b(\w+)\(")


def build(tmp):
    sys.path.insert(0, ROOT)
    import __graft_entry__ as g
    lib = os.path.join(tmp, "libschnorr_b200.so")
    subprocess.check_call(["nvcc"] + g.NVCC_FLAGS + ["-o", lib, os.path.join(g.CSRC, "schnorr_b200.cu")])
    return lib


def disassemble(lib, tmp):
    subprocess.check_call(["cuobjdump", "-xelf", "all", os.path.abspath(lib)], cwd=tmp, stdout=subprocess.DEVNULL)
    cubin = sorted(glob.glob(os.path.join(tmp, "*sm_100a*.cubin")))[0]
    return subprocess.run(["nvdisasm", "-gi", "-c", cubin], capture_output=True, text=True, check=True).stdout.split("\n")


def body(lines, kernel_key, func):
    """(opcode, inline line stack) of every instruction of the subroutine `func` that kernel `kernel_key` calls"""
    start = re.compile(r"^\$\S*%s\S*\$\S*%s\S*:$" % (kernel_key, func))
    out, stack, inside, closed = [], [], False, True
    for ln in lines:
        if not inside:
            inside = bool(start.match(ln))
            continue
        if ln.startswith(("$", ".text", "//----", "\t.section")):
            break
        # one group of line records per instruction: innermost frame first, the group ends with the frame that has no
        # "inlined at"; only the last group before an instruction describes it
        m = re.match(r'\s*//## File "[^"]*", line (\d+)', ln)
        if m:
            if closed:
                stack = []
            stack.append(int(m.group(1)))
            closed = "inlined at" not in ln
            continue
        m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P[T\d]\s+)?([A-Z0-9_.]+)", ln)
        if m:
            if stack:
                cur = stack
            out.append((m.group(1), tuple(cur)))
            stack = []
    if not out:
        raise SystemExit("no %s body found in %s" % (func, kernel_key))
    return out


def price(instrs):
    wide = sum(op.startswith("IMAD.WIDE") for op, _ in instrs)
    other = len(instrs) - wide
    return {"instructions": len(instrs), "imad_wide": wide, "others": other,
            "issue_model_cycles": round(WIDE_CYCLES * wide + OTHER_CYCLES * other, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib")
    ap.add_argument("--src", default=os.path.join(ROOT, "schnorr_b200", "csrc", "fq.cuh"))
    ap.add_argument("--json")
    args = ap.parse_args()
    src = open(args.src).read().split("\n")
    funcs, cur = [], "?"  # enclosing function of every source line
    for ln in src:
        m = FUNC_DEF.match(ln)
        cur = m.group(1) if m else cur
        funcs.append(cur)
    res = {"model": "%.1f cycles per IMAD.WIDE + %.2f per other instruction (DESIGN 4.0)" % (WIDE_CYCLES, OTHER_CYCLES)}
    with tempfile.TemporaryDirectory() as tmp:
        lines = disassemble(args.lib or build(tmp), tmp)
        for kname, key in KERNELS.items():
            r = res[kname] = {}
            for f in BODIES:
                ins = body(lines, key, f)
                r[f] = price(ins)
                r[f]["opcodes"] = dict(collections.Counter(op for op, _ in ins).most_common())
                if f == "fq_sqr_ool":
                    parts = collections.defaultdict(list)
                    for op, st in ins:
                        line = st[0]
                        fn = funcs[line - 1] if line <= len(funcs) else "?"
                        rest = fn in REST_FUNCS or (fn == "fq_sqr_inl" and not PRODUCT_LINE.search(src[line - 1]))
                        parts["reduction_epilogue_call" if rest else "product"].append((op, st))
                    r[f]["split"] = {k: price(v) for k, v in sorted(parts.items())}
            r["sqr_over_mul"] = round(r["fq_sqr_ool"]["issue_model_cycles"] / r["fq_mul_ool"]["issue_model_cycles"], 3)
    for kname in KERNELS:
        print(kname)
        for f in BODIES:
            p = res[kname][f]
            print("  %-11s %4d instr  %3d IMAD.WIDE  %3d others  %6.1f cycles" % (f, p["instructions"], p["imad_wide"], p["others"],
                                                                               p["issue_model_cycles"]))
            for k, s in p.get("split", {}).items():
                print("    %-25s %4d instr  %3d IMAD.WIDE  %3d others" % (k, s["instructions"], s["imad_wide"], s["others"]))
        print("  squaring / product = %.3f" % res[kname]["sqr_over_mul"])
    if args.json:
        with open(args.json, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
