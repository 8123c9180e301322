"""SASS of the step's kernels in two builds of the library: instruction counts, the grid-dependency instructions, and the
instructions of each kernel that one build has and the other has not, as multisets with branch and reconvergence targets
masked (so that an inserted instruction, and the rescheduling around it, shows as that instruction alone).

    python tools/sass_chain.py BEFORE.so AFTER.so > profiles/r06_sass_chain.txt

ACQBULK = griddepcontrol.wait (a kernel's reads of the previous kernel's results come after it), PREEXIT =
griddepcontrol.launch_dependents (the next kernel's CTAs may start).
"""
import collections
import re
import subprocess
import sys

CHAIN = ("bv_count_kernel", "bv_scalar_kernel", "bv_bound_kernel", "bv_hist_kernel", "bv_em_iter_kernel", "bv_em_task_kernel",
         "bv_fisher_kernel")


def kernels(lib):
    txt = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    out, name = {}, None
    for line in txt.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            name = subprocess.run(["c++filt", m.group(1)], capture_output=True, text=True).stdout.strip()
            out[name] = []
            continue
        m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(.*?)\s*;", line)
        if m and name:
            ins = re.sub(r"\s+", " ", m.group(1))
            if re.search(r"\b(BRA|BSSY|CALL|JMP|BRX|WARPSYNC)\b", ins):
                ins = re.sub(r"0x[0-9a-f]+$", "<target>", ins)
            out[name].append(ins)
    return {k: v for k, v in out.items() if any(c in k for c in CHAIN)}


before, after = kernels(sys.argv[1]), kernels(sys.argv[2])
for k in sorted(after):
    a, b = before.get(k, []), after[k]
    op = lambda L, o: sum(1 for x in L if o in x.split(" ")[0:2])
    print(f"{k}: {len(a)} -> {len(b)} instructions; ACQBULK {op(a, 'ACQBULK')} -> {op(b, 'ACQBULK')}, "
          f"PREEXIT {op(a, 'PREEXIT')} -> {op(b, 'PREEXIT')}")
    ca, cb = collections.Counter(a), collections.Counter(b)
    diff = ["- " + x for x in sorted((ca - cb).elements())] + ["+ " + x for x in sorted((cb - ca).elements())]
    if len(diff) <= 12:
        for d in diff:
            print("    " + d)
    else:
        print(f"    ({len(diff)} instructions differ)")
