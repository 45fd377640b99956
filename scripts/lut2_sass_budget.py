"""Warp-instruction budget of the headline kernel (qtable_scan_lut2<float, true, false>, DESIGN.md 4.1) by phase, from its
SASS alone (CPU only; no profiler needed).

    python scripts/lut2_sass_budget.py [--lib th_rl_b200/libthrl.so] [--build] [--dirty 12,12] [--loops]

The kernel is disassembled with line info (`cuobjdump -xelf`, `nvdisasm -gi`).  Every instruction is attributed to the line
of thrl_scan_lut2.cuh it comes from (the call site, for inlined helpers), and the line to a phase by the markers in the
source (an instruction from a line of the kernel's prologue, a value re-derived inside a loop, goes with the one before it):
  A       draws (Philox)                       seq     rebuild of the state sequence (noisy instantiation only: 0 here)
  B       rollout                              C       snapshot (old values, visit counters, dirty masks)
  expand  D's per-chunk expansion + prologue   D       D's inner loop (one transition of each agent per iteration)
  E       greedy refresh, greedy-pair cache    stats   epsilon decay, logs, statistics
Loops are the backward branches.  A loop's trip count per entry comes from the source line of its `for` (loop_trips below)
at the C2 shape of bench.py: T = L = 100 steps, 16-transition chunks (7 per epoch), NR = 41 compact rows per agent, 21
actions, and `--dirty` written compact rows per agent and epoch (scripts/lut2_chain_stats.py: ~26 distinct states per episode
at epsilon = 0.11, 12 at 0.026, 7.5 at 0.01).  Each instruction counts (executions per epoch of its innermost loop) / (2 T)
warp instructions per agent-step; code outside the epoch loop (staging, write-back) is per run and is left out.

This is a static model: divergent paths count as if every branch were taken by some lane, and data-dependent branches
(`if (v > m)` in a scan is a select, not a branch) are counted as taken.  It steers and compares builds of the same source
tree; a profiler's count is the measurement.
"""
import argparse
import math
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = "thrl_scan_lut2.cuh"
KERNEL = "_ZN4thrl16qtable_scan_lut2IfLb1ELb0EEEvNS_10Lut2ParamsE"
CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")

# phase markers: the first source line containing the text opens the phase (in source order)
MARKERS = [
    ("run", "// ---- this warp's slot"),
    ("A", "// ---- A: draws"),
    ("B", "// ---- B: the episode"),
    ("Bmap", "// ---- B.map"),
    ("Bfill", "// ---- B.fill"),
    ("Blog", "// ---- B.log"),
    ("Bser", "} else if (!kNoise) {"),
    ("seq", "// states before every step"),
    ("trace", "// optional per-step traces"),
    ("C", "// ---- C: snapshot pass"),
    ("expand", "// chunk expansion, lane-parallel"),
    ("D", "// ---- D: the sequential pass"),
    ("expand", "for (int c0 = 0; c0 < L0; c0 += kLut2Chunk)"),
    ("D", "#pragma unroll 2\n          for (int j = n; j > 0; --j, --cd)"),
    ("Dsplit", "} else {\n        for (int ag = 0; ag < 2; ++ag)"),
    ("E", "// ---- E: refresh"),
    ("stats", "// epsilon decay"),
    ("run", "// ---- write the run back"),
]
PHASES = ["A", "B", "Bmap", "Bfill", "Blog", "seq", "C", "expand", "D", "E", "stats"]


def shape(dirty, events):
    T, L, chunk, NR, A = 100, 100, 16, 41, 21
    return dict(T=T, L=L, chunk=chunk, chunks=math.ceil(L / chunk), NR=NR, A=A, dirty=dirty, events=events)


# loop trip counts per entry, by the text of the loop's `for` line (first match wins); the unroll factor of the source
# pragma divides the count of the unrolled body
def loop_trips(text, s):
    T, L, A = s["T"], s["L"], s["A"]
    nd = sum(s["dirty"])
    table = [
        (r"for \(int e = 0; e < E; \+\+e\)", None),                            # the epoch loop: counts are per epoch
        (r"for \(int t = lane; t < T; t \+= 32\)", math.ceil(T / 32)),          # A (and traces)
        (r"for \(int n2 = T >> 1", T / 2 / 2),                                  # B step by step (Bser), pairs, unroll 2
        (r"for \(int c0 = 0; c0 < T; c0 \+= 32\)", math.ceil(T / 32)),         # B.fill, 32 steps per pass
        (r"for \(unsigned mw = m; mw != 0u", s["events"] / math.ceil(T / 32)),  # B.fill, the events of 32 steps
        (r"for \(; t \+ 32 <= T; t \+= 32\)", T // 32),                        # B.log, 32 steps per iteration
        (r"for \(; t \+ 8 <= T; t \+= 8\)", T % 32 // 8),                       # B.log, 8 steps
        (r"for \(; t < T; \+\+t\)", T % 8),                                      # B.log, single steps
        (r"for \(int t = lane; t <= T; t \+= 32\)", math.ceil((T + 1) / 32)),   # seq
        (r"for \(int j = T - L1 \+ lane; j < T; j \+= 32\) reinterpret_cast", 0),  # C, unequal batches only (none at C2)
        (r"for \(int j = T - L0 \+ lane|for \(int j = T - L1 \+ lane", math.ceil(L / 32)),  # C, one agent per loop
        (r"for \(int j = T - \(L0 > L1", math.ceil(L / 32)),                   # C, both agents per step
        (r"for \(int c0 = 0; c0 < L0; c0 \+= kLut2Chunk\)", s["chunks"]),      # D chunks
        (r"for \(int j = n; j > 0; --j, --cd\)", L / s["chunks"] / 2),          # D inner, unroll 2
        (r"for \(int c = 64 \+ lane", 0),                                     # E, rows from 64 on (none at C2)
        (r"for \(int i = lane; i < nd; i \+= 32\)", max(1, math.ceil(nd / 32))),  # E, lane per written row
        (r"for \(int k = 1; k < A; \+\+k\)", (A - 1) / 4),                     # E, row scan, unroll 4
        (r"for \(int s = lane; s <= NS; s \+= 32\)", math.ceil((s["NR"] + 2) / 32)),  # E, greedy pairs (NS = 41 states)
    ]
    for pat, n in table:
        if re.search(pat, text):
            return n
    return None


# loops inside lambdas carry the line of the lambda's call site only: trip counts by that line, and whether the loop has
# another loop inside it
def lambda_trips(text, nested, s):
    if re.search(r"for \(int c = 64 \+ lane", text):
        return 0
    if re.search(r"\brefresh\(", text):
        return math.ceil((s["NR"] + 2) / 32) if nested else (s["A"] - 1) / 4  # lane per compact row; its row scan (unroll 4)
    if re.search(r"\bscan_row\(", text) and not nested:
        return (s["A"] - 1) / 4
    return None


def disassemble(lib):
    with tempfile.TemporaryDirectory() as tmp:
        subprocess.run([os.path.join(CUDA, "bin", "cuobjdump"), "-xelf", "all", os.path.abspath(lib)], cwd=tmp, check=True,
                       stdout=subprocess.DEVNULL)
        out = []
        for f in sorted(os.listdir(tmp)):
            if f.endswith(".cubin"):
                r = subprocess.run([os.path.join(CUDA, "bin", "nvdisasm"), "-gi", "-c", os.path.join(tmp, f)], check=True,
                                   stdout=subprocess.PIPE, text=True)
                out.append(r.stdout)
    text = "\n".join(out)
    i = text.find(".text.%s:" % KERNEL)
    if i < 0:
        sys.exit("%s not found in %s" % (KERNEL, lib))
    j = text.find("\t.section", i)
    return text[i:j if j > 0 else len(text)]


LINE_RE = re.compile(r'//## File "([^"]+)", line (\d+)(.*)')
INSTR_RE = re.compile(r"/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;")
LABEL_RE = re.compile(r"^(\.L_x_\d+):")


def parse(sass):
    """-> [(addr, instr, (innermost, outermost) line of thrl_scan_lut2.cuh, (0, 0) if none)], {label: instruction index}"""
    instrs, labels = [], {}
    cur = (0, 0)
    for raw in sass.splitlines():
        m = LINE_RE.search(raw)
        if m:
            chain = [(m.group(1), int(m.group(2)))] + [(f, int(n)) for f, n in re.findall(r'inlined at "([^"]+)", line (\d+)', m.group(3))]
            own = [n for f, n in chain if f.endswith(SRC)]
            cur = (own[0], own[-1]) if own else (0, 0)
            continue
        m = LABEL_RE.match(raw.strip())
        if m:
            labels[m.group(1)] = len(instrs)
            continue
        m = INSTR_RE.search(raw)
        if m:
            instrs.append((int(m.group(1), 16), m.group(2), cur))
    return instrs, labels


def phase_of_lines(src_lines):
    text = "\n".join(src_lines)
    starts = []
    for ph, marker in MARKERS:
        k = text.find(marker)
        if k < 0:
            continue
        line = text.count("\n", 0, k) + 1 + marker.count("\n")
        starts.append((line, ph))
    starts.sort()

    def phase(line):
        ph = "setup"
        for l0, p in starts:
            if line >= l0:
                ph = p
        return ph
    return phase


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--lib", default=os.path.join(ROOT, "th_rl_b200", "libthrl.so"))
    ap.add_argument("--src", default=None, help="thrl_scan_lut2.cuh the library was built from (default: next to --lib)")
    ap.add_argument("--build", action="store_true", help="build the library first (th_rl_b200.build)")
    ap.add_argument("--dirty", default="12,12", help="written compact rows per agent and epoch")
    ap.add_argument("--events", type=float, default=8.0,
                    help="exploration steps (events) per episode: the lane-parallel rollout's event loop trips")
    ap.add_argument("--loops", action="store_true", help="also list every loop with its static size and trip count")
    a = ap.parse_args()
    if a.build:
        sys.path.insert(0, ROOT)
        from th_rl_b200 import build as b
        a.lib = b.build()
    src = a.src or os.path.join(os.path.dirname(os.path.abspath(a.lib)), "csrc", SRC)
    with open(src) as f:
        src_lines = f.read().splitlines()
    phase = phase_of_lines(src_lines)
    s = shape([int(x) for x in a.dirty.split(",")], a.events)
    instrs, labels = parse(disassemble(a.lib))

    # loops: backward branches (target index <= branch index), innermost first.  A loop's `for` is one of the `for` lines
    # its body's instructions come from (innermost source line) that no loop nested in it has taken.
    loops = []
    for i, (_, ins, _) in enumerate(instrs):
        m = re.search(r"\bBRA\b.*?(\.L_x_\d+)", ins)
        if m and labels.get(m.group(1)) is not None and labels[m.group(1)] <= i:
            loops.append(dict(lo=labels[m.group(1)], hi=i))
    loops.sort(key=lambda L: L["hi"] - L["lo"])
    for L in loops:
        taken = {M["for_line"] for M in loops if "for_line" in M and L["lo"] <= M["lo"] and M["hi"] <= L["hi"]}
        cand = sorted({ln[0] for _, _, ln in instrs[L["lo"]:L["hi"] + 1]
                       if ln[0] and "for (" in src_lines[ln[0] - 1] and ln[0] not in taken})
        bl = instrs[L["hi"]][2][0]
        L["for_line"] = bl if bl in cand else (cand[0] if cand else None)
    epoch = [L for L in loops if L["for_line"] and re.search(r"for \(int e = 0; e < E;", src_lines[L["for_line"] - 1])]
    if not epoch:
        sys.exit("epoch loop not found")
    ep = max(epoch, key=lambda L: L["hi"] - L["lo"])
    inner = [L for L in loops if ep["lo"] <= L["lo"] and L["hi"] <= ep["hi"] and L is not ep]
    for L in inner:
        if L["for_line"]:
            L["text"] = src_lines[L["for_line"] - 1].strip()
            L["trips"] = loop_trips(L["text"], s)
        else:
            body = [ln[0] for _, _, ln in instrs[L["lo"]:L["hi"] + 1] if ln[0]]
            dom = max(set(body), key=body.count)
            nested = any(M is not L and L["lo"] <= M["lo"] and M["hi"] <= L["hi"] for M in inner)
            L["text"] = "(call at %d) %s" % (dom, src_lines[dom - 1].strip())
            L["trips"] = lambda_trips(src_lines[dom - 1], nested, s)
    unknown = [L for L in inner if L["trips"] is None and phase(instrs[L["lo"]][2][1]) in PHASES]

    # executions per epoch of instruction i = product of the trip counts of the loops around it (inside the epoch loop)
    per_phase = {p: 0.0 for p in PHASES}
    other = {}
    static = {p: 0 for p in PHASES}
    prev = "A"
    for i in range(ep["lo"], ep["hi"] + 1):
        n = 1.0
        for L in inner:
            if L["lo"] <= i <= L["hi"] and L["trips"] is not None:
                n *= L["trips"]
        ph = phase(instrs[i][2][1]) if instrs[i][2][1] else "?"
        if ph in ("setup", "run", "?"):  # values from the kernel's prologue re-derived in a loop: the phase it runs in
            ph = prev
        prev = ph
        if ph in per_phase:
            per_phase[ph] += n
            static[ph] += 1
        else:
            other[ph] = other.get(ph, 0.0) + n
    steps = 2 * s["T"]
    print("qtable_scan_lut2<float, true, false>  %s" % a.lib)
    print("shape: T = L = %d, %d chunks, NR = %d, A = %d, written rows per epoch %s, events per episode %g" %
          (s["T"], s["chunks"], s["NR"], s["A"], "+".join(map(str, s["dirty"])), s["events"]))
    print("%-8s %8s %14s" % ("phase", "static", "instr/ag-step"))
    for p in PHASES:
        print("%-8s %8d %14.2f" % (p, static[p], per_phase[p] / steps))
    for p, n in sorted(other.items()):
        print("%-8s %8s %14.2f   (not on the C2 path: left out of the total)" % (p, "", n / steps))
    off = sum(per_phase[p] for p in PHASES if p not in ("B", "D")) / steps
    print("total %.2f   off-chain (all but B and D) %.2f" % (sum(per_phase.values()) / steps, off))
    if unknown:
        print("loops without a trip count (counted once):", "; ".join(L["text"] for L in unknown))
    if a.loops:
        for L in sorted(inner, key=lambda L: L["lo"]):
            print("  loop %5d-%5d  %4d instr  x%s  line %s: %s" % (L["lo"], L["hi"], L["hi"] - L["lo"] + 1, L["trips"],
                                                                  L["for_line"], L["text"]))


if __name__ == "__main__":
    main()
