"""Static SASS inspection of lib/libfsr1_b200.so (no GPU needed).

  python tools/sass_tools.py hist [substring]      opcode histogram per kernel (largest basic blocks with --blocks)
  python tools/sass_tools.py snapshot FILE         save the instruction streams of every kernel
  python tools/sass_tools.py loops BINARY          opcode histogram of each kernel's largest loop (the timed loop of
                                                   tools/ubench_pipes.cu: one iteration)
  python tools/sass_tools.py diff FILE             compare the current library against a snapshot: lists kernels whose
                                                   instruction stream changed (used to prove that adding an opt-in
                                                   variant leaves every production kernel byte-for-byte the same)
"""
import collections
import json
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "fidelityfx-fsr_b200", "lib", "libfsr1_b200.so")


def kernels(path=LIB):
    out = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True).stdout
    d, cur = {}, None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            d[cur] = []
            continue
        m = re.match(r"\s+/\*([0-9a-f]{4,})\*/\s+(.*?);", line)
        if m and cur:
            d[cur].append((int(m.group(1), 16), m.group(2).strip()))
    return d


def demangle(name):
    try:
        return subprocess.run(["c++filt", name], capture_output=True, text=True).stdout.strip().split("(")[0]
    except OSError:
        return name


def opcode(text):
    t = text.split()
    return (t[1] if t[0].startswith("@") else t[0]).split(".")[0]


def blocks(ins):
    targets = set()
    for _, t in ins:
        m = re.search(r"\bBRA\b.*?0x([0-9a-f]+)", t)
        if m:
            targets.add(int(m.group(1), 16))
    out, cur = [], []
    for a, t in ins:
        if a in targets and cur:
            out.append(cur)
            cur = []
        cur.append((a, t))
        if re.search(r"\b(BRA|EXIT|RET|BSYNC)\b", t):
            out.append(cur)
            cur = []
    if cur:
        out.append(cur)
    return out


def main():
    cmd = sys.argv[1] if len(sys.argv) > 1 else "hist"
    if cmd == "loops":
        for name, ins in kernels(sys.argv[2]).items():
            body = []
            for a, t in ins:  # the largest loop: from the target of a backward branch up to that branch
                m = re.search(r"\bBRA\b.*?0x([0-9a-f]+)", t)
                if m and int(m.group(1), 16) < a:
                    loop = [(b, u) for b, u in ins if int(m.group(1), 16) <= b <= a]
                    body = loop if len(loop) > len(body) else body
            print("%-28s %4d SASS per iteration: %s" % (demangle(name), len(body),
                                                         dict(collections.Counter(opcode(t) for _, t in body).most_common(6))))
        return
    ks = kernels()
    if cmd == "hist":
        sub = [a for a in sys.argv[2:] if not a.startswith("--")]
        for name, ins in ks.items():
            dn = demangle(name)
            if sub and sub[0] not in dn:
                continue
            h = collections.Counter(opcode(t) for _, t in ins)
            print("%s: %d instructions" % (dn, len(ins)))
            print("   ", dict(h.most_common(18)))
            if "--blocks" in sys.argv:
                for b in sorted(blocks(ins), key=len, reverse=True)[:4]:
                    hb = collections.Counter(opcode(t) for _, t in b)
                    print("    block @%#x, %d instructions: %s" % (b[0][0], len(b), dict(hb.most_common(10))))
    elif cmd == "snapshot":
        json.dump({demangle(k): [t for _, t in v] for k, v in ks.items()}, open(sys.argv[2], "w"))
        print("saved", len(ks), "kernels")
    elif cmd == "diff":
        old = json.load(open(sys.argv[2]))
        new = {demangle(k): [t for _, t in v] for k, v in ks.items()}
        changed = [k for k in old if k in new and old[k] != new[k]]
        print("changed:", changed)
        print("removed:", [k for k in old if k not in new])
        print("added:", [k for k in new if k not in old])
        sys.exit(1 if changed else 0)


if __name__ == "__main__":
    main()
