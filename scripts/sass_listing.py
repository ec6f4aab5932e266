"""SASS of the hot kernels of librpsf_b200.so (sm_100a), per kernel: opcode histogram with the Blackwell / TMA markers
counted, then the instruction listing (encodings stripped).  Needs cuobjdump; no GPU.

    python scripts/sass_listing.py [P] > profiles/<round>_sass_k1_k2_k3_p256.txt
"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "regularizepsf_b200", "librpsf_b200.so")
P = sys.argv[1] if len(sys.argv) > 1 else "256"
WANTED = [rf"k1_streamILi{P}Ef", rf"k2_pipelinedILi{P}Ef", rf"k3_streamILi{P}EfLb0"]
MARKERS = ["UBLKCP", "SYNCS", "UTMALDG", "UTMASTG", "LDGSTS", "FFMA2", "FADD2", "FMUL2", "FFMA", "FADD", "FMUL", "LDS", "STS",
           "LDG", "STG", "SHFL", "BAR", "MEMBAR", "ATOMG", "REDG", "HMMA", "UTC", "ACQBULK", "PREEXIT"]


def main():
    names = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True).stdout
    blocks = re.split(r"\n\s*Function : ", names)
    print(f"# cuobjdump -sass {os.path.relpath(LIB, ROOT)} (sm_100a), kernels of patch size {P}, float32")
    for want in WANTED:
        for block in blocks[1:]:
            head, _, body = block.partition("\n")
            if not re.search(want, head):
                continue
            demangled = subprocess.run(["c++filt", head.strip()], capture_output=True, text=True).stdout.strip()[:160]
            ops = []
            lines = []
            for line in body.splitlines():
                m = re.match(r"\s*/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;", line)
                if not m:
                    continue
                text = re.sub(r"\s+", " ", m.group(2))
                lines.append(f"  /*{m.group(1)}*/ {text}")
                op = text.split()[1] if text.startswith("@") and len(text.split()) > 1 else text.split()[0]
                ops.append(op.split(".")[0])
            hist = collections.Counter(ops)
            print(f"\n================ {demangled}\n# {len(lines)} instructions")
            print("# markers: " + ", ".join(f"{k} {sum(v for o, v in hist.items() if o == k)}" for k in MARKERS
                                           if any(o == k for o in hist)))
            print("# top opcodes: " + ", ".join(f"{o} {c}" for o, c in hist.most_common(16)))
            print("\n".join(lines))
            break


if __name__ == "__main__":
    main()
