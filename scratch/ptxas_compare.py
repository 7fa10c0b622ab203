"""ptxas -v resource lines (registers, spills, stack, static shared memory) of two builds, kernel by kernel: every kernel
of the first build must be unchanged in the second.

    make -C rpsmf_b200/csrc OBJDIR=/tmp/obj_parent ...   (at the parent commit), then at this one:
    make -C rpsmf_b200/csrc OBJDIR=/tmp/obj_new ...
    python scratch/ptxas_compare.py /tmp/obj_parent /tmp/obj_new

Prints every kernel that differs or is missing, then the counts."""
import glob, os, re, sys

def parse(d):
    out = {}
    for f in sorted(glob.glob(os.path.join(d, "*.ptxas.log"))):
        cur = None
        for line in open(f):
            m = re.search(r"Compiling entry function '([^']+)'", line)
            if m:
                cur = m.group(1); out[cur] = []; continue
            if cur and ("Used" in line or "spill" in line or "stack frame" in line):
                out[cur].append(re.sub(r"^ptxas info\s*:\s*", "", line.strip()))
    return out

a, b = parse(sys.argv[1]), parse(sys.argv[2])
# the new trailing template parameter (bool LL = false) of the three kernels is part of the mangled name
b = {re.sub(r"Lb0E(EEvNS_7KParamsE)$", r"\1", k) if "psmf_" in k and "_kernelI" in k else k: v for k, v in b.items()}
diff = [k for k in a if a[k] != b.get(k)]
for k in diff:
    print(k, a[k], b.get(k))
print("parent kernels: %d, new tree kernels: %d, added: %d, changed or missing: %d" % (len(a), len(b), len(set(b) - set(a)), len(diff)))
