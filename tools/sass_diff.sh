#!/bin/bash
# Do two builds of the library carry the same machine code for the kernels matching $3 (mangled-name regex)?
#   tools/sass_diff.sh build/librtrace_b200_r01.so rust-tracer_b200/librtrace_b200.so 'phase_.*ILi4ELi1ELi1ELi2ELi2E'
# Prints per kernel: instruction counts and whether the opcode+operand streams are identical (addresses and
# line-info stripped).  A change that is meant to leave existing kernels alone can be checked here on the CPU
# before GPU time is spent on an A/B.  Kernels in an anonymous namespace are matched without the namespace's name,
# whose hashes change with the source file's contents.
A=$1; B=$2; RE=${3:-phase_}
for lib in "$A" "$B"; do
  cuobjdump -sass "$lib" 2>/dev/null | awk -v re="$RE" '
    /Function :/ { name=$3; keep = (name ~ re); next }
    keep && /^[ \t]+\/\*[0-9a-f]+\*\// { line=$0; sub(/^[ \t]+\/\*[0-9a-f]+\*\/[ \t]+/, "", line); sub(/[ \t]*\/\*.*$/, "", line); print name "\t" line }
  ' > /tmp/sass_$(basename "$lib").txt
done
python3 - "$A" "$B" <<'PY'
import sys, collections, os, re
a, b = ["/tmp/sass_%s.txt" % os.path.basename(x) for x in sys.argv[1:3]]
def strip_ns(name):  # <len>_GLOBAL__N__<hash>_<file>_<hash>: drop the <len> characters of the namespace's name
    m = re.search(r"(\d+)_GLOBAL__N__", name)
    return name if not m else name[:m.start()] + "_GLOBAL__N__" + name[m.end(1) + int(m.group(1)):]
def load(p):
    d = collections.OrderedDict()
    for ln in open(p):
        k, _, ins = ln.rstrip("\n").partition("\t")
        d.setdefault(strip_ns(k), []).append(ins)
    return d
da, db = load(a), load(b)
for k in da:
    if k not in db:
        print("only in A:", k); continue
    same = da[k] == db[k]
    print("%s  A %d  B %d instr  %s" % (k[:70], len(da[k]), len(db[k]), "IDENTICAL" if same else "DIFFERENT"))
for k in db:
    if k not in da: print("only in B:", k[:70], len(db[k]))
PY
