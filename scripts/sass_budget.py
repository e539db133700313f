"""Opcode histogram of the render kernel's hot loops, from the SASS of a compiled object (no GPU needed).

    python scripts/sass_budget.py [object] [--kernel SUBSTRING]

object defaults to build/obj/vs_render.o (`make lib`); the kernel defaults to the bench instance
vs_render_kernel<SYNTH, GEN_FAST, noise=0, FILT_INT, raw=0, tract=0>.  A hot loop is an innermost backward branch:
the F loop is one 24-sample block of the recurrence (one copy per preset: the first is shown, the others are
counted to check they are alike), the G loop one or more 8-sample groups of gen_fast (one DMUL per sample).  Per sample, an FP64 instruction
holds the sub-partition's issue port two cycles and every other instruction one (DESIGN.md 4.1)."""
import argparse
import collections
import os
import pathlib
import re
import subprocess

ROOT = pathlib.Path(__file__).resolve().parents[1]
BENCH = "vs_render_kernelILi1ELi0ELb0ELi0ELb0ELb0E"
FP64 = ("DFMA", "DMUL", "DADD")
INS = re.compile(r"/\*([0-9a-f]{4,})\*/\s+(@!?U?P[T0-9]\s+)?([A-Z][A-Z0-9_.]*)\s*([^;]*);")


def sass(obj, kernel):
    cuobjdump = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")
    out = subprocess.run([cuobjdump, "-sass", obj], check=True, capture_output=True, text=True).stdout
    funcs = re.split(r"\n\s*Function : ", out)
    hits = [f for f in funcs[1:] if kernel in f.split("\n", 1)[0]]
    if len(hits) != 1:
        raise SystemExit(f"{len(hits)} functions match {kernel!r}")
    return [(int(m.group(1), 16), m.group(3), m.group(4)) for m in INS.finditer(hits[0])]


def loops(ins):
    """innermost loops: [target, branch] of backward branches that contain no other backward branch"""
    addr = [a for a, _, _ in ins]
    spans = []
    for i, (a, op, args) in enumerate(ins):
        m = re.match(r"0x([0-9a-f]+)", args.strip())
        if op == "BRA" and m and int(m.group(1), 16) < a:
            spans.append((addr.index(int(m.group(1), 16)), i))
    return [(s, e) for s, e in spans if not any(s <= s2 and e2 <= e and (s2, e2) != (s, e) for s2, e2 in spans)]


def key(op, args):
    """opcode with the modifiers that matter for the accounting"""
    if op.startswith("IMAD") and not op.startswith("IMAD.MOV"):
        return op + (" (x+0)" if args.rstrip().endswith("RZ") else "")
    if op.startswith(("IMAD.MOV", "I2F", "F2I")):
        return op
    return op.split(".")[0]


def report(name, body, samples):
    h = collections.Counter(key(op, args) for _, op, args in body)
    fp = sum(n for k, n in h.items() if k.startswith(FP64))
    other = len(body) - fp
    print(f"{name}: {len(body)} instructions per {samples} samples, FP64 {fp}, others {other} = {other / samples:.2f} per sample, "
          f"issue cycles per sample {(2 * fp + other) / samples:.2f}")
    print("   " + ", ".join(f"{k} {n}" for k, n in sorted(h.items(), key=lambda kv: (-kv[1], kv[0]))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("object", nargs="?", default=str(ROOT / "build/obj/vs_render.o"))
    ap.add_argument("--kernel", default=BENCH)
    a = ap.parse_args()
    ins = sass(a.object, a.kernel)
    f_loops, g_loops = [], []
    for s, e in loops(ins):
        body = ins[s:e + 1]
        ops = collections.Counter(op.split(".")[0] for _, op, _ in body)
        if ops["DFMA"] >= 22 * 24:
            f_loops.append(body)
        elif ops["DMUL"] and ops["DMUL"] % 8 == 0 and ops["LDS"] >= ops["DMUL"]:
            g_loops.append(body)
    print(f"{a.kernel}: {len(ins)} instructions")
    for i, body in enumerate(f_loops[:1]):
        report(f"F, one 24-sample block ({len(f_loops)} copies, sizes {sorted(set(len(b) for b in f_loops))})", body, 24)
    for body in g_loops[:1]:
        n = sum(op == "DMUL" for _, op, _ in body)
        report(f"G, {n // 8} 8-sample group(s) ({len(g_loops)} copies)", body, n)


if __name__ == "__main__":
    main()
