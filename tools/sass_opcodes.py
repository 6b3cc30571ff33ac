#!/usr/bin/env python
"""Per-kernel histogram of the Blackwell-specific SASS opcodes in the shipped library (cuobjdump -sass):

    python tools/sass_opcodes.py [jittor-clip-fewshot_b200/libjclip_b200.so] > profiles/sass_opcodes.md

UTCHMMA = tcgen05.mma (.2CTA = cta_group::2), LDTM / STTM = tcgen05.ld / st (TMEM), UTMALDG / UTMASTG / UTMAREDG = TMA
tensor load / store / reduce-add (cp.async.bulk.tensor, cp.reduce.async.bulk.tensor), UTCBAR = tcgen05.commit,
HMMA = legacy mma.sync, SYNCS = mbarrier operations, ACQBULK / PREEXIT =
griddepcontrol.wait / launch_dependents (programmatic dependent launch), UCGABAR = barrier.cluster (thread-block clusters).
"""
import collections
import re
import subprocess
import sys

LIB = sys.argv[1] if len(sys.argv) > 1 else "jittor-clip-fewshot_b200/libjclip_b200.so"
OPS = ["UTCHMMA", "UTCHMMA.2CTA", "LDTM", "STTM", "UTMALDG", "UTMASTG", "UTMAREDG", "UTCBAR", "HMMA", "SYNCS", "MUFU.TANH", "MUFU.EX2", "ACQBULK", "PREEXIT", "UCGABAR"]


def demangle(names):
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.splitlines()
    return dict(zip(names, out))


def short(sig):
    sig = re.sub(r"\(anonymous namespace\)::", "", sig)
    sig = re.sub(r"^void ", "", sig)
    sig = re.sub(r"jcb::", "", sig)
    m = re.match(r"([\w:]+(<.*?>)?)\(", sig)
    return m.group(1) if m else sig[:80]


def main():
    sass = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True, check=True).stdout
    counts, cur, arch = collections.OrderedDict(), None, set()
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            counts[cur] = collections.Counter()
            continue
        a = re.match(r"\s*arch = (sm_\w+)", line)
        if a:
            arch.add(a.group(1))
        if cur is None:
            continue
        m = re.search(r"^\s*/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_.]+)", line)
        if not m:
            continue
        op = m.group(1)
        c = counts[cur]
        c["_total"] += 1
        if op.startswith("UTCHMMA"):
            c["UTCHMMA"] += 1
            if ".2CTA" in op:
                c["UTCHMMA.2CTA"] += 1
        elif op.startswith("LDTM"):
            c["LDTM"] += 1
        elif op.startswith("STTM"):
            c["STTM"] += 1
        elif op.startswith("UTMALDG"):
            c["UTMALDG"] += 1
        elif op.startswith("UTMASTG"):
            c["UTMASTG"] += 1
        elif op.startswith("UTMAREDG"):
            c["UTMAREDG"] += 1
        elif op.startswith("UTCBAR"):
            c["UTCBAR"] += 1
        elif op.startswith("HMMA"):
            c["HMMA"] += 1
        elif op.startswith("SYNCS"):
            c["SYNCS"] += 1
        elif op.startswith("MUFU.TANH"):
            c["MUFU.TANH"] += 1
        elif op.startswith("MUFU.EX2"):
            c["MUFU.EX2"] += 1
        elif op.startswith("ACQBULK"):
            c["ACQBULK"] += 1
        elif op.startswith("PREEXIT"):
            c["PREEXIT"] += 1
        elif op.startswith("UCGABAR"):
            c["UCGABAR"] += 1
    names = demangle(list(counts))
    print(f"# SASS opcode histogram of `{LIB}` (cuobjdump -sass; architectures: {', '.join(sorted(arch))})\n")
    print("Static instruction counts per kernel; kernels without any of the listed opcodes are summarised at the end.  "
          "`gemm_tcgen05[_2cta]_kernel<BN, EPI, F16>`: EPI 0 bias, 1 bias + QuickGELU, 2 bias + fp32 residual reduce-add, "
          "4 fp32 out, 5 LayerNorm-folded, 6 LayerNorm-folded + QuickGELU, 7 / 8 residual + LayerNorm preparation (out_proj / "
          "c_proj); F16 = fp16 (true) or bf16 (false) 16-bit outputs.  `attention_tcgen05_kernel<T, F16, MODE>`: MODE 0 two heads "
          "per 128-row tile (image tower), 1 one head per tile with optional causal mask (text tower).\n")
    print("| kernel | SASS instrs | " + " | ".join(OPS) + " |")
    print("|---|---:|" + "---:|" * len(OPS))
    tot = collections.Counter()
    plain = []
    for k, c in counts.items():
        for o in OPS:
            tot[o] += c[o]
        if not any(c[o] for o in OPS):
            plain.append(short(names[k]))
            continue
        print(f"| `{short(names[k])}` | {c['_total']} | " + " | ".join(str(c[o]) if c[o] else "" for o in OPS) + " |")
    print("| **total** | | " + " | ".join(str(tot[o]) for o in OPS) + " |")
    print(f"\n{len(plain)} kernels with none of these opcodes (SIMT kernels: row-wise, MTA, head, TTA, weight packing): "
          + ", ".join(f"`{p}`" for p in sorted(set(plain))))


if __name__ == "__main__":
    main()
