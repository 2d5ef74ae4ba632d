"""Function-by-function comparison of two builds' device code.

    python tools/sass_compare.py BASE.sass NEW.sass [BASE_ptxas.log NEW_ptxas.log]

BASE.sass / NEW.sass: `cuobjdump -sass build/rt_device.o` of the two builds.  Each kernel's instructions are compared
with the addresses stripped (encodings kept): "same" means byte-identical machine code, hence the same memory traffic.
With the two `-Xptxas -v` logs (EXTRA_NVCCFLAGS="-Xptxas -v" make) it also prints registers, stack and spills per kernel.
"""
import re
import sys


def functions(path):
    out, name, body = {}, None, []
    for line in open(path):
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            if name:
                out[name] = body
            name, body = m.group(1), []
        elif name:
            body.append(re.sub(r"/\*[0-9a-f]{4,}\*/", "", line).rstrip())
    if name:
        out[name] = body
    return out


def ptxas(path):
    out, name = {}, None
    for line in open(path):
        m = re.search(r"Function properties for (\S+)", line)
        if m:
            name = m.group(1)
            out[name] = {}
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and name:
            out[name].update(stack=int(m.group(1)), spill_st=int(m.group(2)), spill_ld=int(m.group(3)))
        m = re.search(r"Used (\d+) registers", line)
        if m and name:
            out[name]["regs"] = int(m.group(1))
    return out


def main():
    a, b = functions(sys.argv[1]), functions(sys.argv[2])
    pa = ptxas(sys.argv[3]) if len(sys.argv) > 4 else {}
    pb = ptxas(sys.argv[4]) if len(sys.argv) > 4 else {}
    fmt = lambda p: "%3d regs %4d B stack %3d/%3d B spill st/ld" % (p["regs"], p["stack"], p["spill_st"], p["spill_ld"]) if p else "-"
    for k in sorted(set(a) | set(b)):
        state = "new " if k not in a else "gone" if k not in b else "same" if a[k] == b[k] else "DIFF"
        extra = "   base: %s   new: %s" % (fmt(pa.get(k)), fmt(pb.get(k))) if pa else ""
        print("%s %s%s" % (state, k, extra))


if __name__ == "__main__":
    main()
