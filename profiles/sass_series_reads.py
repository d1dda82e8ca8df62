#!/usr/bin/env python
"""Static register-read count of the unrolled series block of a kernel, from its SASS (no GPU needed):
    python profiles/sass_series_reads.py [LIB] [--kernel REGEX] [--rows-per-thread N] [--json]
LIB defaults to the in-tree libso3d.so; the kernel defaults to the two-row `series` kernel
(rowwise_kernel_w2<LogpScore2Op<0>>).  The unrolled block is the basic block with the most MUFU.EX2.  Per term of N rows
(N = 2 for the packed form: two MUFU.EX2 per term, N = 1 for the one-row form) it reports the instructions by opcode, the
MUFU count, the vector-register words the instructions read (a register pair of an F32x2 operand is two words; uniform
registers, RZ and immediates are none), the words ptxas serves from the operand reuse cache (operands flagged `.reuse`:
the next instruction's read of that operand slot hits the cache) and the floors they set per warp and SMSP:
    read floor = words / 2 clocks (about 2 register words per clock per SMSP: profiles/microbench/pipes.cu measures a
                 3-register FFMA at 85 and a 2-register one at 117 lanes/clk/SM),
    XU floor   = 8 clocks per MUFU (16 lanes/clk/SM).
"""
import argparse
import collections
import json
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORDS_PER_CLK = 2.0
XU_CLK_PER_MUFU = 8.0
INS = re.compile(r"/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;")
REG = re.compile(r"^-?\|?(R\d+)((?:\.\w+)*)\|?$")


def cuobjdump():
    from diffusion_extensions_b200 import build
    return os.path.join(os.path.dirname(build.find_nvcc()), "cuobjdump")


def functions(sass):
    """{mangled name: [(address, text)]} of every function in a cuobjdump -sass listing."""
    out, cur = {}, None
    for line in sass.splitlines():
        if "Function :" in line:
            cur = out.setdefault(line.split("Function :")[1].strip(), [])
            continue
        m = INS.search(line)
        if cur is not None and m:
            cur.append((int(m.group(1), 16), m.group(2)))
    return out


def parse(text):
    """(opcode, [source operands]) of one instruction; the predicate guard is dropped."""
    t = re.sub(r"^@!?U?P\w+\s+", "", text)
    op, _, rest = t.partition(" ")
    ops = [o.strip() for o in rest.split(",")] if rest else []
    has_dst = not (op.startswith(("BRA", "EXIT", "RET", "BAR", "ST", "RED", "NOP", "WARPSYNC", "BSYNC", "CALL")))
    return op, ops[1:] if has_dst and ops else ops


def reads(src):
    """[(slot, words, reused)] of the vector-register operands of an instruction."""
    r = []
    for slot, o in enumerate(src):
        m = REG.match(o)
        if not m:
            continue
        mods = m.group(2)
        r.append((slot, 2 if ".F32x2" in mods else 1, ".reuse" in mods))
    return r


def basic_blocks(ins):
    targets = {int(t, 16) for _, x in ins for t in re.findall(r"\bBRA(?:\.\w+)*\s+(?:!?U?P\w+,\s*)?(0x[0-9a-f]+)", x)}
    blocks, cur = [], []
    for addr, x in ins:
        if addr in targets and cur:
            blocks.append(cur)
            cur = []
        cur.append((addr, x))
        if re.search(r"\b(BRA|EXIT|RET|CALL)\b", x):
            blocks.append(cur)
            cur = []
    if cur:
        blocks.append(cur)
    return blocks


def count(block, rows):
    ops = collections.Counter()
    words = reused = mufu = 0
    for _, x in block:
        op, src = parse(x)
        ops[op] += 1
        if op.startswith("MUFU"):
            mufu += 1
        for _, w, ru in reads(src):
            words += w
            reused += w if ru else 0
    if not mufu:
        sys.exit("the block has no MUFU: not a series block")
    terms = mufu / rows
    per = lambda v: round(v / terms, 3)
    return {
        "terms_in_block": terms,
        "instructions_per_term": per(sum(ops.values())),
        "opcodes_per_term": {k: per(v) for k, v in sorted(ops.items(), key=lambda kv: -kv[1])},
        "mufu_per_term": per(mufu),
        "register_words_per_term": per(words),
        "reuse_words_per_term": per(reused),
        "read_floor_clk": per(words / WORDS_PER_CLK),
        "read_floor_clk_after_reuse": per((words - reused) / WORDS_PER_CLK),
        "xu_floor_clk": per(mufu * XU_CLK_PER_MUFU),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("lib", nargs="?", default=os.path.join(ROOT, "diffusion_extensions_b200", "libso3d.so"))
    ap.add_argument("--kernel", default=r"rowwise_kernel_w2INS_12LogpScore2OpILi0EEEE")
    ap.add_argument("--rows-per-thread", type=int, default=2)
    ap.add_argument("--json", action="store_true", help="one JSON line per kernel instead of the table")
    a = ap.parse_args()
    sass = subprocess.run([cuobjdump(), "-sass", a.lib], capture_output=True, text=True, check=True).stdout
    found = [(n, i) for n, i in functions(sass).items() if re.search(a.kernel, n)]
    if not found:
        sys.exit(f"no kernel matches {a.kernel!r} in {a.lib}")
    for name, ins in found:
        blk = max(basic_blocks(ins), key=lambda b: sum(1 for _, x in b if "MUFU.EX2" in x))
        r = {"lib": os.path.basename(a.lib), "kernel": name, "rows_per_term": a.rows_per_thread, **count(blk, a.rows_per_thread)}
        if a.json:
            print(json.dumps(r))
            continue
        print(f"{name}  ({r['lib']}, unrolled block of {r['terms_in_block']:g} terms of {a.rows_per_thread} rows)")
        print("  per term: " + ", ".join(f"{v:g} {k}" for k, v in r["opcodes_per_term"].items()))
        print(f"  register words {r['register_words_per_term']:g}, of which .reuse {r['reuse_words_per_term']:g};  "
              f"read floor {r['read_floor_clk']:g} clk ({r['read_floor_clk_after_reuse']:g} after reuse), XU floor {r['xu_floor_clk']:g} clk")


if __name__ == "__main__":
    main()
