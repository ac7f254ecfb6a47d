"""Static SASS budget of k_playout: instruction counts by opcode of the round body and of the prologue.

Compiles csrc/hz_engine.cu with the library's flags (build.NVCC_FLAGS) to a cubin in a temporary directory, disassembles
k_playout<false> and k_playout<true> and splits each into basic blocks.  The round body is the largest basic block (the
round is one straight line of several hundred instructions; the next largest block is a quarter of it or less), the
prologue is everything ahead of the first BAR.SYNC (the block's tables are ready there).  Opcodes on the integer ALU pipe
(LOP3, SEL, SHF, ISETP, IADD3, LEA, PRMT, ...) are summed apart from IMAD, which issues to the FMA pipe.  Local-memory
accesses (STL, LDL: register spills) are counted in the round body, the prologue and the rest of the kernel.  No GPU
needed.

    python profiles/sass_mix.py [--src DIR]     # DIR: another checkout's harmonies_alphazero_b200/csrc (A/B)
"""
import argparse
import collections
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from harmonies_alphazero_b200 import build  # noqa: E402

KERNELS = {"k_playout<false>": "_ZN2hz9k_playoutILb0EEEvPvliPjPyPKmmmS2_",
           "k_playout<true>": "_ZN2hz9k_playoutILb1EEEvPvliPjPyPKmmmS2_"}
ALU = ("LOP3", "SEL", "SHF", "ISETP", "IADD3", "LEA", "PRMT", "VIADD", "IABS", "VIMNMX", "FLO", "BREV", "PLOP3", "SGXT",
       "BMSK", "ICMP", "IMNMX")
ENDS_BLOCK = ("BRA", "EXIT", "RET", "BRX", "CALL", "BSSY", "BSYNC", "WARPSYNC", "BAR")


def opcode(ins):
    return re.sub(r"^@!?U?P\w+\s+", "", ins).split()[0].split(".")[0]


def cubin_sass(csrc):
    nvcc = build._nvcc()
    cuda_bin = os.path.dirname(nvcc) if os.path.isabs(nvcc) else ""
    with tempfile.TemporaryDirectory() as tmp:
        cubin = os.path.join(tmp, "hz_engine.cubin")
        subprocess.run([nvcc] + build.NVCC_FLAGS + ["-cubin", "-o", cubin, os.path.join(csrc, "hz_engine.cu")], check=True)
        text = subprocess.run([os.path.join(cuda_bin, "nvdisasm"), cubin], check=True, capture_output=True, text=True).stdout
    return text


def kernel_sass(text, mangled):
    return text.split("//--------------------- .text." + mangled)[1].split("//---------------------")[0]


def blocks_of(sass):
    """Instructions of the kernel in order and its basic blocks (split at labels and after control flow)."""
    ins, blocks, cur = [], [], []
    for line in sass.splitlines():
        if re.match(r"\s*\.L_x_\d+:", line):
            if cur:
                blocks.append(cur)
            cur = []
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;", line)
        if not m:
            continue
        op = opcode(m.group(1))
        ins.append(op)
        cur.append(op)
        if op in ENDS_BLOCK:
            blocks.append(cur)
            cur = []
    if cur:
        blocks.append(cur)
    return ins, blocks


def report(name, ops):
    c = collections.Counter(ops)
    alu = sum(v for k, v in c.items() if k in ALU)
    print(f"{name}: {len(ops)} instructions, ALU pipe {alu}, IMAD {c.get('IMAD', 0)}, POPC {c.get('POPC', 0)}, "
          f"STL {c.get('STL', 0)}, LDL {c.get('LDL', 0)}")
    print("   " + "  ".join(f"{k} {v}" for k, v in c.most_common()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--src", default=build.CSRC, help="csrc directory to compile (default: this tree's)")
    a = ap.parse_args()
    text = cubin_sass(a.src)
    for name, mangled in KERNELS.items():
        ins, blocks = blocks_of(kernel_sass(text, mangled))
        sizes = sorted((len(b) for b in blocks), reverse=True)
        print(f"{a.src}: {name} {len(ins)} instructions, largest basic blocks {sizes[:4]}")
        body = max(blocks, key=len)
        report("round body (largest basic block)", body)
        report("prologue (ahead of the first BAR.SYNC)", ins[:ins.index("BAR")])
        rest = collections.Counter(ins) - collections.Counter(body) - collections.Counter(ins[:ins.index("BAR")])
        print(f"rest of the kernel: STL {rest.get('STL', 0)}, LDL {rest.get('LDL', 0)}")


if __name__ == "__main__":
    main()
