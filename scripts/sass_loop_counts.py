"""Static SASS instruction counts of K2q's per-step streams (rollout_cartpole_ws6_kernel), read from cuobjdump -sass:
usage: python scripts/sass_loop_counts.py [relearn_b200/librelearn_b200.so | build/rollout.o]

  dynamics loop      the dynamics warp's loop (the backward branch whose body holds BAR.SYNC 0x2 and BAR.ARV 0x1)
  dynamics b2 -> b1  BAR.SYNC 0x2 .. BAR.ARV 0x1, both counted: the select / convert / publish segment on the step cycle
  aux noise step     the aux warp's loop over one step of noise (the innermost loop holding a Philox multiply by
                     0xD2511F53 that sits inside another loop: the steady-state fill, not the two prologue fills)
  policy b1 -> b2    BAR.SYNC 0x1 .. BAR.ARV 0x2 of the policy loop, both counted, along the loop's fall-through path
                     (through the backward branch when ptxas rotated the loop so that the barrier sits at its end)
Each row also lists its most frequent opcodes."""
import collections
import re
import subprocess
import sys

lib = sys.argv[1] if len(sys.argv) > 1 else "relearn_b200/librelearn_b200.so"
out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
body = re.split(r"\n\s*Function : ", out)
text = next((b for b in body if "rollout_cartpole_ws6_kernel" in b.split("\n", 1)[0]), None)
if text is None:
    sys.exit(f"{lib}: no rollout_cartpole_ws6_kernel")

ins = []  # (address, opcode, full text)
for line in text.splitlines():
    m = re.match(r"\s+/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;", line)
    if m:
        txt = m.group(2)
        op = re.sub(r"^@!?U?P[T0-9]+\s+", "", txt).split()[0]
        ins.append((int(m.group(1), 16), op, txt))
index = {a: i for i, (a, _, _) in enumerate(ins)}


def find(lo, hi, pred):
    return [i for i in range(lo, hi + 1) if pred(ins[i][2])]


loops = []  # (head index, backedge index)
for i, (a, op, txt) in enumerate(ins):
    m = re.search(r"\bBRA(?:\.U)?\s+(?:!?U?P\d+,\s*)?0x([0-9a-f]+)", txt)
    if op.startswith("BRA") and m and int(m.group(1), 16) < a and int(m.group(1), 16) in index:
        loops.append((index[int(m.group(1), 16)], i))


def is_bar(txt, kind, bid):
    return re.search(rf"\bBAR\.{kind}\S*\s+0x{bid}\b", txt) is not None


def row(name, idx):
    c = collections.Counter(ins[i][1] for i in idx)
    top = ", ".join(f"{k} {v}" for k, v in c.most_common(8))
    print(f"{name:20s} {len(idx):5d}   {top}")


print(f"# {lib}: rollout_cartpole_ws6_kernel, static SASS instructions per loop iteration (sm_100a)")
dyn = [(h, b) for h, b in loops if find(h, b, lambda t: is_bar(t, "SYNC", 2)) and find(h, b, lambda t: is_bar(t, "ARV", 1))]
h, b = min(dyn, key=lambda l: l[1] - l[0])
row("dynamics loop", range(h, b + 1))
s = find(h, b, lambda t: is_bar(t, "SYNC", 2))[0]
e = next(i for i in range(s, b + 1) if is_bar(ins[i][2], "ARV", 1))
row("dynamics b2 -> b1", range(s, e + 1))

philox = [(h, b) for h, b in loops if find(h, b, lambda t: "-0x2daee0ad" in t.lower() or "0xd2511f53" in t.lower())
       and any(h2 < h and b <= b2 for h2, b2 in loops)]
h, b = min(philox, key=lambda l: l[1] - l[0])
row("aux noise step", range(h, b + 1))

pol = [(h, b) for h, b in loops if find(h, b, lambda t: is_bar(t, "ARV", 2)) and find(h, b, lambda t: is_bar(t, "SYNC", 1))
       and not find(h, b, lambda t: is_bar(t, "SYNC", 2))]
h, b = min(pol, key=lambda l: l[1] - l[0])
a2 = find(h, b, lambda t: is_bar(t, "ARV", 2))[0]
s1 = find(h, b, lambda t: is_bar(t, "SYNC", 1))
s = max(i for i in s1 if i < a2) if any(i < a2 for i in s1) else s1[-1]
row("policy b1 -> b2", range(s, a2 + 1) if s < a2 else list(range(s, b + 1)) + list(range(h, a2 + 1)))
