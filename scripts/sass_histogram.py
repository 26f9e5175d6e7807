#!/usr/bin/env python
"""SASS mnemonic histogram of the shipped sweep kernels (no GPU needed: cuobjdump reads the .so).

    python scripts/sass_histogram.py [--lib stencilstream_b200/libstst_workloads.so] [--match Jacobi5Rule]

For every `fused_sweep_kernel` instantiation whose mangled name contains `--match`: instruction count,
the mnemonic histogram grouped by pipe (FP32 / FP64 / integer / shared-memory / global-memory / TMA +
barrier / control), and the Blackwell evidence lines (UTMALDG = cp.async.bulk.tensor loads, SYNCS =
mbarrier, STG.E.128 = 128-bit stores, LDGSTS = cp.async). Used for the profiles/r0*_sass_*.txt files.

With --loops, also the body of every loop (a backward branch and what lies between its target and it)
that holds at least 20 FFMA: what one iteration of a sweep's row loop issues, which the kernel totals
hide when a kernel carries several loop variants.
"""
import argparse
import collections
import re
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
GROUPS = [
    ("fp32", r"^(FFMA|FADD|FMUL|FMNMX|FSEL|FSETP|FSET|MUFU|FCHK|F2F|FFMA2|FADD2|FMUL2)"),
    ("fp64", r"^(DFMA|DADD|DMUL|DSETP|DMNMX|F2F\.F64|DFMA2)"),
    ("shared-memory", r"^(LDS|STS|LDSM|STSM)"),
    ("global-memory", r"^(LDG|STG|LDGSTS|LD\.|ST\.|ATOM|RED|LDGDEPBAR|DEPBAR|CCTL|MEMBAR|ERRBAR|FENCE)"),
    ("tma+mbarrier", r"^(UTMALDG|UTMASTG|UBLKCP|SYNCS|UTMACCTL|UTMAPF)"),
    ("control", r"^(BRA|BSSY|BSYNC|EXIT|RET|CALL|BAR|WARPSYNC|NOP|BMOV|BREAK|YIELD|NANOSLEEP|JMP|BRX)"),
    ("integer/logic", r"^(IADD|IMAD|IMNMX|ISETP|LOP|SHF|LEA|MOV|SEL|PRMT|POPC|FLO|I2F|F2I|I2I|PLOP|P2R|R2P|S2R|CS2R|S2UR|"
                      r"UMOV|UIADD|UIMAD|ULOP|USHF|ULEA|UISETP|USEL|R2UR|UFLO|UPOPC|VOTE|SHFL|REDUX|LDC|ULDC|IABS|UPLOP|"
                      r"UP2UR|UR2UP|I2FP|F2FP|VIADD|VIMNMX|UIADD3|IADD3|LOP3|UPRMT|BREV|SGXT|USGXT|UF2FP|HADD|HFMA|HMUL|IDP)"),
]


def kernels(lib: Path):
    text = subprocess.run(["cuobjdump", "-sass", str(lib)], capture_output=True, text=True).stdout
    name, body = None, []
    for line in text.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            if name:
                yield name, body
            name, body = m.group(1), []
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_.]*)", line)
        if m and name:
            body.append(m.group(1))
    if name:
        yield name, body


def loops(lib: Path, match: str):
    """(kernel, [(first address, instruction count, Counter of base mnemonics)]) per sweep kernel."""
    text = subprocess.run(["cuobjdump", "-sass", str(lib)], capture_output=True, text=True).stdout
    for part in re.split(r"\n\s*Function : ", text)[1:]:
        name = part.split("\n", 1)[0].strip()
        if "fused_sweep_kernel" not in name or match not in name:
            continue
        ins = []
        for line in part.splitlines():
            m = re.match(r"\s*/\*([0-9a-f]{4,})\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9_.]*)(.*);", line)
            if m:
                ins.append((int(m.group(1), 16), m.group(2), m.group(3)))
        index = {a: i for i, (a, _, _) in enumerate(ins)}
        found = []
        for i, (a, op, rest) in enumerate(ins):
            t = re.search(r"0x([0-9a-f]+)", rest) if op.startswith("BRA") else None
            if t and int(t.group(1), 16) < a and int(t.group(1), 16) in index:
                body = ins[index[int(t.group(1), 16)]:i + 1]
                ops = collections.Counter(o.split(".")[0] for _, o, _ in body)
                if ops["FFMA"] >= 20:
                    found.append((body[0][0], len(body), ops))
        yield name, found


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", type=Path, default=ROOT / "stencilstream_b200" / "libstst_workloads.so")
    ap.add_argument("--match", default="")
    ap.add_argument("--loops", action="store_true", help="also the instruction counts of the row loops")
    args = ap.parse_args()
    for name, body in kernels(args.lib):
        if "fused_sweep_kernel" not in name or args.match not in name:
            continue
        demangled = subprocess.run(["c++filt", name], capture_output=True, text=True).stdout.strip()
        print(f"kernel: {demangled[:150]}")
        print(f"  instructions: {len(body)}")
        grouped = collections.Counter()
        detail = collections.defaultdict(collections.Counter)
        for op in body:
            base = op
            for group, pattern in GROUPS:
                if re.match(pattern, base):
                    grouped[group] += 1
                    detail[group][base.split(".")[0]] += 1
                    break
            else:
                grouped["other"] += 1
                detail["other"][base.split(".")[0]] += 1
        for group, count in grouped.most_common():
            top = ", ".join(f"{k} {v}" for k, v in detail[group].most_common(6))
            print(f"  {group:15s} {count:6d} ({100.0 * count / max(len(body), 1):4.1f} %)  {top}")
        ops = collections.Counter(body)
        evidence = {k: v for k, v in ops.items()
                    if k.startswith(("UTMALDG", "UTMASTG", "SYNCS", "LDGSTS", "STG.E.128", "LDS.128", "STS.128",
                                     "UBLKCP", "MEMBAR", "ATOM", "FFMA2"))}
        print("  evidence: " + ", ".join(f"{k} x{v}" for k, v in sorted(evidence.items())))
        print()
    if args.loops:
        for name, found in loops(args.lib, args.match):
            demangled = subprocess.run(["c++filt", name], capture_output=True, text=True).stdout.strip()
            print(f"loops of: {demangled[:150]}")
            for start, n, ops in found:
                counts = " ".join(f"{k} {ops[k]}" for k in ("FFMA", "FMUL", "LDS", "STS", "STG", "BAR"))
                print(f"  loop at {start:#07x}: {n:5d} instructions, {counts}")


if __name__ == "__main__":
    sys.exit(main())
