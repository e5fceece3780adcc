"""Registers, spills and the steady-loop instruction mix of kernel C (pdps_tblock.cuh), from the compiler alone.

  python tools/sass_tblock.py                      # the bench kernel: fp64, T = 4, VEC = 2, scalar λ, strict
  python tools/sass_tblock.py --all                # every RING instantiation of every tblock_f{64,32}_t{2,3,4}.cu
  python tools/sass_tblock.py --unit tblock_f32_t2 --fast --map

Each unit is compiled with the Makefile's flags into a temporary directory (nothing in the tree changes), ptxas -v gives
registers and spills, and `cuobjdump -sass` the code.  The steady march loop is the innermost backward branch of the
kernel body that spans the most fp64 instructions (the two-step trip of pdps_tblock_kernel).  Its static instruction
count is divided by the pixel-iterations one trip covers (2 steps × T stages × VEC rows per thread); the never-taken
IEEE fallback of the projection (the forward-branched block around the ball_scale_ieee calls) is left out.  Needs nvcc
and cuobjdump, no GPU.
"""
import argparse
import collections
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "bpldenoising_b200", "csrc")
CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")
NVCC = os.path.join(CUDA, "bin", "nvcc")
CUOBJDUMP = os.path.join(CUDA, "bin", "cuobjdump")
# the Makefile's NVCCFLAGS
FLAGS = ["-O3", "-std=c++17", "-lineinfo", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler",
         "-fPIC,-Wall,-Wno-unused-function", "-Xptxas", "-v", "--expt-relaxed-constexpr"]

FP64 = {"DADD", "DMUL", "DFMA", "DSETP", "DMNMX"}
SELECT = {"FSEL", "SEL"}
COPY = {"MOV", "IMAD.MOV"}            # register copies (IMAD.MOV.U32 Rd, RZ, RZ, Rs is how ptxas spells most of them)


def mangled(real, vec, t, map_, strict, ring=True, batch=False, maxt=256, minb=None):
    minb = minb if minb is not None else (2 if t <= 2 else 1)
    b = lambda v: "Lb%dE" % int(v)  # noqa: E731
    return ("_ZN5bpltv18pdps_tblock_kernelI%sLi%dELi%dE%s%s%s%sLi%dELi%dEEEvNS_10TBlockArgsIT_XT1_EEE" %
            (real, vec, t, b(map_), b(strict), b(ring), b(batch), maxt, minb))


def compile_unit(unit, out_dir):
    obj = os.path.join(out_dir, unit + ".o")
    r = subprocess.run([NVCC] + FLAGS + ["-c", "-o", obj, os.path.join(CSRC, unit + ".cu")], cwd=CSRC,
                       capture_output=True, text=True)
    if r.returncode != 0:
        sys.exit(r.stderr)
    return obj, r.stderr


def ptxas_info(log, name):
    # "Compiling entry function 'NAME'" … "N bytes stack frame, S bytes spill stores, L bytes spill loads" … "Used R registers"
    i = log.find("Function properties for " + name)
    if i < 0:
        return None
    chunk = log[i:i + 600]
    m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", chunk)
    r = re.search(r"Used (\d+) registers", chunk)
    return {"regs": int(r.group(1)), "stack": int(m.group(1)), "spill_st": int(m.group(2)), "spill_ld": int(m.group(3))}


def parse_sass(text):
    ins = []
    for line in text.splitlines():
        m = re.match(r"\s*/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;", line)
        if m:
            ins.append((int(m.group(1), 16), m.group(2)))
    return ins


def opcode(txt):
    t = re.sub(r"^@!?U?P\w+\s+", "", txt)
    op = t.split()[0]
    if op.startswith("IMAD.MOV"):
        return "IMAD.MOV"
    return op


def branch_target(txt):
    m = re.search(r"\bBRA(?:\.[\w.]+)?\s+(?:!?U?P\w+,\s*)?0x([0-9a-f]+)", txt)
    return int(m.group(1), 16) if m else None


def steady_loop(ins):
    exits = [a for a, t in ins if opcode(t) == "EXIT"]
    end = max(exits) if exits else ins[-1][0]
    loops = []
    for a, t in ins:
        tgt = branch_target(t)
        if tgt is not None and tgt < a <= end and (a - tgt) // 16 >= 64:
            loops.append((tgt, a))
    inner = [l for l in loops if not any(o != l and l[0] <= o[0] and o[1] <= l[1] for o in loops)]
    if not inner:
        return None

    def fp64(l):
        return sum(1 for a, t in ins if l[0] <= a <= l[1] and opcode(t).split(".")[0] in FP64)
    return max(inner, key=fp64)


def fallback_ranges(body):
    # the smallest forward-branched block around each CALL of the loop body
    fwd = [(a, branch_target(t)) for a, t in body if branch_target(t) is not None and branch_target(t) > a]
    out = set()
    for a, t in body:
        if opcode(t).startswith("CALL"):
            c = [(s, e) for s, e in fwd if s < a < e]
            if c:
                out.add(min(c, key=lambda r: r[1] - r[0]))
    return sorted(out)


def analyse(sass, per_trip):
    ins = parse_sass(sass)
    loop = steady_loop(ins)
    if loop is None:
        return None
    body = [(a, t) for a, t in ins if loop[0] <= a <= loop[1]]
    fb = fallback_ranges(body)
    kept = [(a, t) for a, t in body if not any(s < a < e for s, e in fb)]
    hist = collections.Counter(opcode(t) for a, t in kept)
    cat = collections.Counter()
    for op, n in hist.items():
        base = op.split(".")[0]
        cat["fp64" if base in FP64 else "select" if base in SELECT else "copy" if op in COPY else "rest"] += n
    return {"loop": loop, "body": len(body), "fallback": len(body) - len(kept), "kept": len(kept), "hist": hist,
            "cat": cat, "per_trip": per_trip}


def report(unit, real, vec, t, map_, strict, log, obj):
    name = mangled(real, vec, t, map_, strict)
    info = ptxas_info(log, name)
    if info is None:
        print("%s: %s not built" % (unit, name))
        return
    sass = subprocess.run([CUOBJDUMP, "-sass", "-fun", name, obj], capture_output=True, text=True).stdout
    per_trip = 2 * t * vec
    a = analyse(sass, per_trip)
    tag = "%s VEC=%d T=%d %s %s" % ("fp64" if real == "d" else "fp32", vec, t, "map" if map_ else "scalar",
                                    "strict" if strict else "fast")
    print("== %s  (%s)" % (tag, unit))
    print("   registers %d, stack %d B, spill stores %d B, spill loads %d B" %
          (info["regs"], info["stack"], info["spill_st"], info["spill_ld"]))
    if a is None:
        print("   no steady loop found")
        return
    pt = float(per_trip)
    print("   steady loop 0x%x-0x%x: %d instructions, %d in the IEEE fallback, %d counted; %d pixel-iterations per trip" %
          (a["loop"][0], a["loop"][1], a["body"], a["fallback"], a["kept"], per_trip))
    c = a["cat"]
    print("   per pixel-iteration: total %.1f = fp64 %.1f + selects %.1f + copies %.1f (%d per trip) + rest %.1f" %
          (a["kept"] / pt, c["fp64"] / pt, c["select"] / pt, c["copy"] / pt, c["copy"], c["rest"] / pt))
    top = ", ".join("%s %.2f" % (op, n / pt) for op, n in a["hist"].most_common(24))
    print("   by opcode: " + top)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--unit", default="tblock_f64_t4", help="translation unit (tblock_f64_t4, tblock_f32_t2, ...)")
    ap.add_argument("--fast", action="store_true", help="fast arithmetic instead of strict")
    ap.add_argument("--map", action="store_true", help="the λ-map instantiation")
    ap.add_argument("--all", action="store_true", help="every RING instantiation of every unit")
    args = ap.parse_args()
    units = ["tblock_f64_t2", "tblock_f64_t3", "tblock_f64_t4", "tblock_f32_t2", "tblock_f32_t3", "tblock_f32_t4"] \
        if args.all else [args.unit]
    with tempfile.TemporaryDirectory() as tmp:
        for unit in units:
            m = re.match(r"tblock_f(64|32)_t(\d)$", unit)
            if not m:
                sys.exit("unknown unit " + unit)
            real, vec, t = ("d", 2, int(m.group(2))) if m.group(1) == "64" else ("f", 4, int(m.group(2)))
            obj, log = compile_unit(unit, tmp)
            combos = [(mp, st) for mp in (False, True) for st in (True, False)] if args.all else [(args.map, not args.fast)]
            for mp, st in combos:
                report(unit, real, vec, t, mp, st, log, obj)


if __name__ == "__main__":
    main()
