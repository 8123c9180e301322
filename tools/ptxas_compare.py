"""Compare two `nvcc -Xptxas -v` logs of the library, kernel by kernel.

    python tools/ptxas_compare.py BEFORE.txt AFTER.txt

For every entry function: registers and cumulative stack (the "Used ..." line of its compilation) and its own stack frame and
spill bytes (the "Function properties for <entry>" line).  Out-of-line device functions (__noinline__) get their own properties
line, which ptxas prints among the entries; they are listed as functions of their own.  Names are demangled with c++filt.
"""
import re
import subprocess
import sys


def parse(path):
    entries, props, cur, props_for = {}, {}, None, None
    for line in open(path):
        m = re.search(r"Compiling entry function '(\w+)'", line)
        if m:
            cur = m.group(1)
            entries.setdefault(cur, {})
            continue
        m = re.search(r"Function properties for (\w+)", line)
        if m:
            props_for = m.group(1)
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and props_for:
            props[props_for] = "stack %s, spill stores %s, spill loads %s" % m.groups()
            props_for = None
            continue
        m = re.search(r"Used (\d+) registers", line)
        if m and cur:
            c = re.search(r"(\d+) bytes cumulative stack size", line)
            entries[cur]["regs"] = "%s registers, cumulative stack %s" % (m.group(1), c.group(1) if c else "0")
    out = {}
    for k, v in entries.items():
        out[k] = "%s; %s" % (v.get("regs", "?"), props.get(k, "?"))
    for k, v in props.items():
        if k not in entries:
            out[k] = "(device function) " + v
    return out


def demangle(name):
    try:
        return re.sub(r"\(.*", "", subprocess.run(["c++filt", name], capture_output=True, text=True).stdout.strip()) or name
    except OSError:
        return name


def main():
    a, b = parse(sys.argv[1]), parse(sys.argv[2])
    for k in sorted(set(a) | set(b), key=demangle):
        sa, sb = a.get(k), b.get(k)
        tag = "same" if sa == sb else "NEW" if sa is None else "GONE" if sb is None else "CHANGED"
        print(f"{tag:8s} {demangle(k)}\n         before: {sa}\n         after:  {sb}")


if __name__ == "__main__":
    main()
