"""What the compiler made of the FP32 sweep's packed static-object loop, for the working tree and a git revision side by side
(no GPU needed). Compiles csrc/hmp_kernels.cu for sm_100a with -Xptxas -v twice and prints:
  - instructions per iteration of the packed static-object loop (one pair of objects) of sweep_tpc_kernel<2, true, float>,
    by opcode class;
  - registers, spill stores / loads and stack frame of every sweep_tpc_kernel instance.
usage: python tools/static_loop_sass.py [revision, default HEAD] [-- extra nvcc flags]"""
import collections
import os
import re
import subprocess
import sys
import tempfile
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KERNEL = "_ZN3hmp16sweep_tpc_kernelILi2ELb1EfEEv10KernelArgs"
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "--expt-relaxed-constexpr", "-cubin", "-Xptxas", "-v"]
CLASSES = [("FFMA2/FMUL2/FADD2", {"FFMA2", "FMUL2", "FADD2"}), ("FFMA/FMUL/FADD", {"FFMA", "FMUL", "FADD"}), ("MUFU", {"MUFU"}),
           ("FSETP/FSEL/FMNMX", {"FSETP", "FSEL", "FMNMX", "FMNMX3"}), ("LOP3/SHF/IMNMX", {"LOP3", "SHF", "IMNMX", "VIMNMX"}),
           ("LDS", {"LDS"})]


def compile_tree(src_root, extra):
    out = tempfile.mkdtemp()
    cubin = os.path.join(out, "k.cubin")
    r = subprocess.run(["nvcc"] + FLAGS + extra + ["-o", cubin, "hmp_kernels.cu"], cwd=os.path.join(src_root, "humap_local_planner_b200", "csrc"),
                       capture_output=True, text=True)
    if r.returncode != 0:
        sys.exit(r.stderr)
    sass = subprocess.run(["cuobjdump", "-sass", cubin], capture_output=True, text=True, check=True).stdout
    return r.stderr, sass


def resources(ptxas):
    """{kernel: (registers, spill stores, spill loads, stack)} of every sweep_tpc_kernel instance."""
    res, name, frame = {}, None, None
    for ln in ptxas.splitlines():
        m = re.search(r"Function properties for (\S+)", ln)
        if m:
            name = m.group(1)
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", ln)
        if m and name:
            frame = tuple(int(v) for v in m.groups())
        m = re.search(r"Used (\d+) registers", ln)
        if m and name and "sweep_tpc_kernel" in name:
            res[name] = (int(m.group(1)), frame[1], frame[2], frame[0])
    return res


def static_loop(sass):
    """Opcode counts of the packed static-object loop: the backward branch whose body has the densest run of FP32x2 opcodes."""
    body = sass.split(f"Function : {KERNEL}", 1)[1].split("Function :", 1)[0]
    ins = []   # (address, opcode, branch target or None)
    for ln in body.splitlines():
        m = re.match(r"\s+/\*([0-9a-f]{4,})\*/\s+(?:@!?U?P[T\d]+\s+)?([A-Z0-9_]+)(?:\.[A-Z0-9_.]+)?\s*([^;]*)", ln)
        if m:
            t = re.match(r"`?\(?\.?L?_?x?_?(0x[0-9a-f]+)", m.group(3).strip()) if m.group(2) == "BRA" else None
            ins.append((int(m.group(1), 16), m.group(2), int(t.group(1), 16) if t else None))
    addr = {a: i for i, (a, _, _) in enumerate(ins)}
    best = None
    for i, (a, op, tgt) in enumerate(ins):
        if op == "BRA" and tgt is not None and tgt < a and tgt in addr:
            ops = [o for _, o, _ in ins[addr[tgt]: i + 1]]
            packed = sum(o in CLASSES[0][1] for o in ops)
            if packed >= 16 and (best is None or packed / len(ops) > best[0]):
                best = (packed / len(ops), ops)
    if best is None:
        sys.exit("packed static-object loop not found")
    return collections.Counter(best[1])


def report(label, ptxas, sass):
    loop = static_loop(sass)
    classes = {}
    rest = collections.Counter(loop)
    for cname, ops in CLASSES:
        classes[cname] = sum(loop[o] for o in ops)
        for o in ops:
            rest.pop(o, None)
    classes["other"] = sum(rest.values())
    return {"label": label, "total": sum(loop.values()), "classes": classes, "other": dict(rest.most_common()), "res": resources(ptxas)}


def main():
    args = sys.argv[1:]
    extra = args[args.index("--") + 1:] if "--" in args else []
    args = args[: args.index("--")] if "--" in args else args
    rev = args[0] if args else "HEAD"
    tmp = tempfile.mkdtemp()
    arch = subprocess.run(["git", "-C", ROOT, "archive", rev, "humap_local_planner_b200/csrc", "include"], capture_output=True, check=True).stdout
    subprocess.run(["tar", "-x", "-C", tmp], input=arch, check=True)
    with ThreadPoolExecutor(2) as ex:
        fut_rev, fut_tree = ex.submit(compile_tree, tmp, extra), ex.submit(compile_tree, ROOT, extra)
        a, b = report(rev, *fut_rev.result()), report("working tree", *fut_tree.result())
    w = 26
    print(f"packed static-object loop of {KERNEL}, instructions per iteration (one pair of objects)")
    print(f"{'':{w}}{a['label']:>14}{b['label']:>14}")
    print(f"{'all':{w}}{a['total']:>14}{b['total']:>14}")
    for cname in [c for c, _ in CLASSES] + ["other"]:
        print(f"{cname:{w}}{a['classes'][cname]:>14}{b['classes'][cname]:>14}")
    for lab, r in ((a["label"], a), (b["label"], b)):
        print(f"  other opcodes, {lab}: " + ", ".join(f"{k} {v}" for k, v in r["other"].items()))
    print("\nsweep_tpc_kernel instances: registers / spill stores / spill loads / stack frame (bytes)")
    for k in sorted(set(a["res"]) | set(b["res"])):
        fa, fb = a["res"].get(k), b["res"].get(k)
        fmt = lambda f: "-" if f is None else "{} / {} / {} / {}".format(*f)
        print(f"  {k:52}{fmt(fa):>24}{fmt(fb):>24}")


if __name__ == "__main__":
    main()
