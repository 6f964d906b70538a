"""Per-kernel counts of the SASS mnemonics that prove tcgen05 / TMEM / TMA / bulk-async use (B200_PROFILING.md), and of the
fp32 arithmetic (scalar FFMA / FADD / FMUL against packed FFMA2 / FADD2 / FMUL2, and MOV), from `cuobjdump -sass`.
Usage: python tools/sass_summary.py [LIB] > profiles/r2_sass_summary.md
       python tools/sass_summary.py LIB --before OLD_LIB     # + static fp32 census of the tensor-core MLP kernels, before / after"""
import argparse
import collections
import re
import subprocess

MN = ["UTCHMMA", "UTCQMMA", "LDTM", "STTM", "UTMALDG", "UTMASTG", "UBLKCP", "SYNCS", "UTCBAR", "HMMA", "FFMA2", "DFMA", "RED", "ATOM"]
FP = ["FFMA", "FADD", "FMUL", "FFMA2", "FADD2", "FMUL2", "MOV", "MUFU", "F2FP", "STL", "LDL"]
TC_MLP = ("ppo_grad_tc_kernel", "rollout_tc_kernel", "critic_values_tc_kernel")


def census(lib):
    out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True).stdout
    counts = collections.OrderedDict()
    cur = None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = subprocess.run(["c++filt", m.group(1)], capture_output=True, text=True).stdout.strip()
            cur = re.sub(r"\(.*", "", cur)
            counts[cur] = collections.Counter()
            continue
        if cur is None:
            continue
        m = re.search(r"/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\w+\s+)?([A-Z0-9_.]+)", line)
        if m:
            op = m.group(1).split(".")[0]
            counts[cur]["_total"] += 1
            counts[cur][op] += 1
            for k in ("RED", "ATOM"):
                if op.startswith(k) and op != k:
                    counts[cur][k] += 1
    return counts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("lib", nargs="?", default="aur_ppo_b200/libaurppo.so")
    ap.add_argument("--before", metavar="OLD_LIB", default=None)
    a = ap.parse_args()
    counts = census(a.lib)
    tc_like = lambda c: any(c[m] for m in ("UTCHMMA", "LDTM", "STTM", "UTMALDG", "UBLKCP"))
    print("# SASS evidence per kernel\n")
    print(f"`cuobjdump -sass {a.lib}` (sm_100a), instruction counts per kernel.  UTCHMMA = tcgen05.mma (kind::f16), LDTM / STTM = tcgen05.ld / st")
    print("(TMEM), UTMALDG = TMA tensor load, UBLKCP = cp.async.bulk, SYNCS = mbarrier ops, UTCBAR = tcgen05.commit.\n")
    cols = MN + [f for f in FP if f not in MN]
    print("| kernel | SASS instr | " + " | ".join(cols) + " |")
    print("|---|---:|" + "---:|" * len(cols))
    tot = collections.Counter()
    for k, c in counts.items():
        if not tc_like(c):
            continue
        print(f"| `{k[:90]}` | {c['_total']} | " + " | ".join(str(c[m]) if c[m] else "" for m in cols) + " |")
        tot.update(c)
    print(f"| **all kernels with tensor-core / TMA / bulk-copy instructions** | {tot['_total']} | " + " | ".join(str(tot[m]) if tot[m] else "" for m in cols) + " |")
    others = [k for k, c in counts.items() if not tc_like(c)]
    print(f"\n{len(others)} further kernels are plain SIMT (env reset, shuffle, moments, reductions, Adam, elementwise helpers, the SIMT cross-check kernels).")
    if a.before:
        before = census(a.before)
        print(f"\n## fp32 arithmetic of the tensor-core MLP kernels: `{a.before}` -> `{a.lib}`\n")
        print("Static counts over the whole kernel (actor and critic paths).  scalar = FFMA + FADD + FMUL.  A kernel that gained a")
        print("template argument (the actor's head width) is set against the one it replaces.\n")
        print("| kernel | SASS instr | scalar | " + " | ".join(FP) + " |")
        print("|---|---:|---:|" + "---:|" * len(FP))
        for k, c in counts.items():
            if not any(t in k for t in TC_MLP):
                continue
            b = before.get(k) or before.get(re.sub(r", \d+>$", ">", k))
            cell = lambda m: f"{b[m]} -> {c[m]}" if b is not None else str(c[m])
            sc = lambda x: x["FFMA"] + x["FADD"] + x["FMUL"]
            print(f"| `{k[:70]}` | {cell('_total')} | " + (f"{sc(b)} -> {sc(c)}" if b is not None else str(sc(c))) + " | " +
                  " | ".join(cell(m) for m in FP) + " |")


if __name__ == "__main__":
    main()
