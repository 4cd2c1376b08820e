"""Static SASS report of the step kernel's control loop (no GPU needed).

    python tools/sass_loop_count.py [object or library ...] [--kernel SUBSTRING]

Default input: taco_b200/build/fpv_step_strict.o.  For every fpv_step_kernel variant it prints registers and stack (cuobjdump
-res-usage), and for each control loop found in its SASS (nvdisasm -gi) the static instruction count, the spills (STL / LDL) and
the opcode mix of the loop body.  The control loop is the `for (int k = 0; k < p.cfi; ++k)` loop of fpv_step_kernel.cuh: a loop
body is the span of a backward branch most of whose instructions come from that loop's source lines (attributed, like
tools/ncu_source_lines.py, through the inlining chain to the innermost line of fpv_step_kernel.cuh).  `philox` counts the
instructions of the rotor-noise Philox block (philox.cuh), which the default configuration skips; `out of line` counts loop-source
instructions placed outside the span (rarely taken blocks the compiler moved away)."""
import argparse
import collections
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KERNEL_SRC = os.path.join(ROOT, "taco_b200", "csrc", "fpv_step_kernel.cuh")
CUDA_BIN = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin")


def _tool(name):
    p = os.path.join(CUDA_BIN, name)
    return p if os.path.exists(p) else name


def loop_lines(path):
    """1-based source line range of the control loop in fpv_step_kernel.cuh (the for line to its closing brace)."""
    src = open(path).read().splitlines()
    start = next(i for i, l in enumerate(src) if "for (int k = 0; k < p.cfi; ++k)" in l)
    depth = 0
    for i in range(start, len(src)):
        code = src[i].split("//")[0]
        depth += code.count("{") - code.count("}")
        if depth == 0 and i > start:
            return start + 1, i + 1
    raise RuntimeError("unbalanced braces after the control loop")


def res_usage(obj):
    out = subprocess.run([_tool("cuobjdump"), "-res-usage", obj], capture_output=True, text=True, check=True).stdout
    res, name = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function (\S+):", line)
        if m:
            name = m.group(1)
            continue
        m = re.search(r"REG:(\d+) STACK:(\d+)", line)
        if m and name:
            res[name] = (int(m.group(1)), int(m.group(2)))
    return res


def functions(cubin):
    out = subprocess.run(["readelf", "-sW", cubin], capture_output=True, text=True).stdout
    fun = {}
    for line in out.splitlines():
        t = line.split()
        if len(t) > 7 and "FUNC" in t and t[0].rstrip(":").isdigit():
            fun[t[-1]] = int(t[0].rstrip(":"))
    return fun


_ANN = re.compile(r'File "([^"]+)", line (\d+)')
_INS = re.compile(r"/\*([0-9a-f]{4,})\*/\s+(.*?);")
_LBL = re.compile(r"^(\.L_x_\d+):")
_TGT = re.compile(r"`\((\.L_x_\d+)\)")


def parse(sass_text):
    """[(addr, opcode, text, innermost file, innermost fpv_step_kernel.cuh line or None)], {label: addr}"""
    ins, labels, pending_lbl, chain = [], {}, [], []
    for line in sass_text.splitlines():
        s = line.strip()
        if s.startswith("//##"):
            chain.append(_ANN.findall(s))
            continue
        m = _LBL.match(s)
        if m:
            pending_lbl.append(m.group(1))
            continue
        m = _INS.search(s)
        if not m:
            continue
        addr, text = int(m.group(1), 16), m.group(2).strip()
        for l in pending_lbl:
            labels[l] = addr
        pending_lbl = []
        frames = chain[0] if chain else []
        inner_file = os.path.basename(frames[0][0]) if frames else ""
        kline = next((int(ln) for f, ln in frames if f.endswith("fpv_step_kernel.cuh")), None)
        if chain:
            chain = []
            ins.append((addr, _opcode(text), text, inner_file, kline))
            last = ins[-1]
        else:                                  # no annotation: same source position as the previous instruction
            ins.append((addr, _opcode(text), text, last[3], last[4]) if ins else (addr, _opcode(text), text, "", None))
    return ins, labels


def _opcode(text):
    t = text.split()
    if t and t[0].startswith("@"):
        t = t[1:]
    return t[0] if t else ""


def loops(ins, labels, lo, hi):
    idx = {a: k for k, (a, *_) in enumerate(ins)}
    cands = []
    for k, (addr, op, text, _, _) in enumerate(ins):
        if not op.startswith("BRA"):
            continue
        m = _TGT.search(text)
        if not m or m.group(1) not in labels or labels[m.group(1)] >= addr:
            continue
        a = idx[labels[m.group(1)]]
        span = ins[a:k + 1]
        inside = sum(1 for x in span if x[4] is not None and lo <= x[4] <= hi)
        if len(span) >= 100 and inside >= 0.5 * len(span):
            cands.append((a, k))
    outer = [c for c in cands if not any(o != c and o[0] <= c[0] and c[1] <= o[1] for o in cands)]
    return sorted(set(outer))


def report(obj, kernel_filter):
    res = res_usage(obj)
    with tempfile.TemporaryDirectory() as tmp:
        subprocess.run([_tool("cuobjdump"), "-xelf", "all", os.path.abspath(obj)], cwd=tmp, capture_output=True, check=True)
        cubins = [os.path.join(tmp, f) for f in sorted(os.listdir(tmp)) if f.endswith(".cubin")]
        for cubin in cubins:
            for name, sym in sorted(functions(cubin).items()):
                if "fpv_step_kernel" not in name or (kernel_filter and kernel_filter not in name):
                    continue
                sass = subprocess.run([_tool("nvdisasm"), "-gi", "-c", "-fun", str(sym), cubin], capture_output=True, text=True, check=True).stdout
                ins, labels = parse(sass)
                # the source the object was built from (its line info names it), else this checkout's
                m = re.search(r'File "([^"]*fpv_step_kernel\.cuh)"', sass)
                src = m.group(1) if m and os.path.exists(m.group(1)) else KERNEL_SRC
                lo, hi = loop_lines(src)
                reg, stack = res.get(name, (None, None))
                spans = loops(ins, labels, lo, hi)
                in_span = set()
                for a, b in spans:
                    in_span.update(range(a, b + 1))
                ool = sum(1 for k, x in enumerate(ins) if k not in in_span and x[4] is not None and lo <= x[4] <= hi)
                print(f"{name}: regs {reg} stack {stack} total {len(ins)} loops {len(spans)} out-of-line loop-source {ool} "
                      f"(control loop: fpv_step_kernel.cuh lines {lo}-{hi})")
                for a, b in spans:
                    body = ins[a:b + 1]
                    mix = collections.Counter(x[1].split(".")[0] for x in body)
                    philox = sum(1 for x in body if x[3] == "philox.cuh")
                    spill = sum(1 for x in body if x[1].startswith(("STL", "LDL")))
                    top = " ".join(f"{o}:{n}" for o, n in mix.most_common(14))
                    print(f"    loop @{body[0][0]:05x}-{body[-1][0]:05x}: {len(body)} instructions, philox {philox}, "
                          f"without philox {len(body) - philox}, STL/LDL {spill}")
                    print(f"        {top}")


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("objects", nargs="*", default=[os.path.join(ROOT, "taco_b200", "build", "fpv_step_strict.o")])
    ap.add_argument("--kernel", default="", help="only the variants whose mangled name contains this")
    a = ap.parse_args()
    for obj in a.objects:
        report(obj, a.kernel)


if __name__ == "__main__":
    sys.exit(main())
