#!/usr/bin/env python
"""Writes profiles/r02_sass_*.txt: opcode histograms and the inner loops of the hot kernels, from cuobjdump -sass of the
built library (run after build())."""
import collections, os, re, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "cuda-sfm_b200", "libsfmb200.so")
sass = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True).stdout
funcs = {}
cur = None
for line in sass.splitlines():
    m = re.match(r"\s*Function : (\S+)", line)
    if m:
        cur = m.group(1)
        funcs[cur] = []
    elif cur and re.match(r"\s*/\*[0-9a-f]{4}\*/", line):
        funcs[cur].append(line)
demangle = lambda n: subprocess.run(["c++filt", n], capture_output=True, text=True).stdout.strip()
def opcode(line):
    m = re.match(r"\s*/\*[0-9a-f]{4}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", line)
    return m.group(1) if m else None
def hist(lines):
    c = collections.Counter()
    for l in lines:
        o = opcode(l)
        if o:
            c[o.split(".")[0]] += 1
    return c
def clean(l):
    return re.sub(r"\s*/\* 0x[0-9a-f]+ \*/\s*$", "", l).rstrip()
def longest_loop(lines):
    """the backward branch spanning the most FFMA/FFMA2 instructions = the inner loop"""
    addr = lambda l: int(re.match(r"\s*/\*([0-9a-f]{4})\*/", l).group(1), 16)
    best = None
    for i, l in enumerate(lines):
        m = re.search(r"BRA(?:\.U)?(?:\.\w+)* (?:!?U?P\d+, )?0x([0-9a-f]+)", l)
        if m and int(m.group(1), 16) < addr(l):
            tgt = int(m.group(1), 16)
            j = next(k for k, x in enumerate(lines) if addr(x) == tgt)
            body = lines[j:i + 1]
            fp = sum(1 for x in body if "FFMA" in x or "FMUL" in x)
            if fp < 0.6 * len(body):
                continue                      # an outer loop: mostly bookkeeping
            if best is None or fp > best[0]:
                best = (fp, body)
    return best[1] if best else []
targets = [("score", "score_kernelILi8ELb1ELi256ELi1ELi0ELb0E", "score_kernel<8, true, 256, 1, 0>: Sampson scoring, packed FFMA2, TMA-staged points (the config-2 / 3 / 4 kernel)"),
           ("triangulate", "triangulate_kernelILi2ELb0ELb0E", "triangulate_kernel<2, false>: two points per thread in packed f32x2"),
           ("hypgen", "hypgen_kernelILi128ELi4ELi0ELi1E", "hypgen_kernel<128, 4, 0, 1>: 8x8 Cholesky projector hypothesis solver"),
           ("small", "small_path_kernel", "small_path_kernel: fused single-launch path, one thread-block cluster per pair")]
for tag, key, title in targets:
    name = next((n for n in funcs if key in n), None)
    if not name:
        continue
    lines = funcs[name]
    h = hist(lines)
    out = [f"# {title}", f"# {demangle(name)}", f"# {len(lines)} SASS instructions (cuobjdump -sass libsfmb200.so, sm_100a)", "", "## opcode histogram (top 24)"]
    out += [f"{v:6d}  {k}" for k, v in h.most_common(24)]
    marks = {"UBLKCP": "TMA bulk copy (cp.async.bulk)", "SYNCS": "mbarrier arrive / try_wait", "FFMA2": "packed fma.rn.f32x2", "FMUL2": "packed mul.rn.f32x2",
             "UCGABAR_ARV": "barrier.cluster.arrive", "UCGABAR_WAIT": "barrier.cluster.wait", "REDUX": "warp reduce", "LDCU": "uniform constant load", "ACQBULK": "bulk async acquire"}
    out += ["", "## evidence opcodes"] + [f"{h[k]:6d}  {k:14s} {v}" for k, v in marks.items() if h.get(k)]
    body = longest_loop(lines)
    out += ["", f"## inner loop ({len(body)} instructions; {sum(1 for x in body if 'FFMA2' in x or 'FMUL2' in x)} packed + "
            f"{sum(1 for x in body if re.search(r'F(FMA|MUL|ADD) ', x))} scalar FP32-pipe instructions)"] + [clean(l) for l in body[:330]] + ([f"... ({len(body) - 330} more)"] if len(body) > 330 else [])
    with open(os.path.join(ROOT, "profiles", f"r02_sass_{tag}.txt"), "w") as f:
        f.write("\n".join(out) + "\n")
    print(tag, len(lines), dict(h.most_common(6)))
