"""Static SASS instruction counts of a kernel per code section (cut at barriers, votes, calls and exits), by pipe.

    python tools/phase_count.py "k_inverse4<3, 256, 0>"          # from himg_b200/_lib/libhimgcu.so
    python tools/phase_count.py "k_inverse4<3, 256, 0>" --file=x.cubin

Used to balance the ALU and FMA pipes of K-inv (DESIGN.md 7); compile the kernel with -DHIMG_FORCE_PRE3 to
count the quality <= 60 path alone."""
import collections
import os
import re
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
FMA = ("IMAD", "IDP", "IMUL")
LSU = ("LDS", "STS", "LDG", "STG", "LDGSTS")
CTRL = ("BRA", "NOP", "BSSY", "BSYNC", "VOTE", "CALL", "EXIT", "BAR", "WARPSYNC", "RET")


def main():
    out = subprocess.run([sys.executable, os.path.join(HERE, "sass_stats.py"), sys.argv[1], "--dump"] + sys.argv[2:],
                         capture_output=True, text=True).stdout
    body = [l.strip() for l in out.splitlines()][1:]
    marks = [i for i, l in enumerate(body) if re.search(r"BAR.SYNC|VOTE|CALL|EXIT|RET", l)]
    cuts = [0] + marks + [len(body)]
    print("%d instructions, sections end at %s" % (len(body), [(i, re.sub(r"^@!?U?P\d+\s+", "", body[i]).split()[0]) for i in marks]))
    for k in range(len(cuts) - 1):
        a, b = cuts[k], cuts[k + 1]
        ops = collections.Counter(re.sub(r"^@!?U?P\d+\s+", "", l).split()[0].split(".")[0] for l in body[a:b])
        fma = sum(v for o, v in ops.items() if o in FMA)
        lsu = sum(v for o, v in ops.items() if o in LSU)
        ctrl = sum(v for o, v in ops.items() if o in CTRL)
        print("section %d: %5d instr | fma %4d  lsu %4d  alu+other %4d | %s" % (k, b - a, fma, lsu, b - a - fma - lsu - ctrl, dict(ops.most_common(10))))


if __name__ == "__main__":
    main()
