"""Counts the SASS instructions one path through a kernel issues (no GPU needed), for profiles/r3_sass_step_hot_path.txt.

    cuobjdump -sass libsoccer2d.so | awk '/Function : /{f = ($3 == K)} f' K=<mangled kernel name> > k.sass
    python profiles/sass_hot_path.py k.sass START STOP [TAKEN,TAKEN,...]

Walks from address START to address STOP (hex, both counted): unconditional branches are followed, a conditional one
(`@P BRA`, `BRA P`, `BRA.U`) only when its address is listed in TAKEN, calls are counted as one instruction and not
entered (the cold paths are out-of-line functions)."""
import re
import sys


def walk(path, start, stop, taken):
    ins = {}
    for line in open(path):
        m = re.match(r"\s*/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;", line)
        if m:
            ins[int(m.group(1), 16)] = m.group(2)
    pc, n = start, 0
    while n < 100000:
        text = ins[pc]
        n += 1
        if pc == stop:
            return n
        m = re.search(r"\bBRA(?:\.U)?\s+(?:!?U?P\d, )?0x([0-9a-f]+)", text)
        if m:
            conditional = text.startswith("@") or "BRA.U" in text or re.search(r"BRA\s+!?P\d,", text)
            if not conditional or pc in taken:
                pc = int(m.group(1), 16)
                continue
        pc += 16
    raise RuntimeError("STOP is not on the path")


if __name__ == "__main__":
    taken = {int(a, 16) for a in sys.argv[4].split(",")} if len(sys.argv) > 4 and sys.argv[4] else set()
    print(walk(sys.argv[1], int(sys.argv[2], 16), int(sys.argv[3], 16), taken))
