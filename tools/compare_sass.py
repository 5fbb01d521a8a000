"""Compare the SASS of two builds of libqcoh.so kernel by kernel.

    python tools/compare_sass.py OLD.so NEW.so [--ptxas OLD.log NEW.log]

The kernels are split at cuobjdump's "Function :" lines and matched by demangled name.  Names of the predict kernels
from before the walk policies (predict_tiles_kernel<ILP, MINB, TEX, HM, PL>, predict_tiles_nodes8_kernel<ILP, HM, PL,
MINB, TEX, CTOP> and predict_soa_kernel<TEX, CTOP, DUO>) are mapped to their DuoWalk / NodesWalk form first.  Constant
bank operands c[0x0][0x...] are masked, because a change of the argument structs moves the parameter offsets, and
the encoding comments, which hold those offsets too, are dropped.  With --ptxas, the register and spill lines of the
two ptxas logs (quickchem_b200/csrc/kernels.ptxas.log) are compared as well.  Exits 1 on any difference.
"""
import argparse
import re
import subprocess
import sys

CUDA_BIN = "/usr/local/cuda/bin"


def demangle(names):
    out = subprocess.run([f"{CUDA_BIN}/cu++filt"], input="\n".join(names), capture_output=True, text=True, check=True)
    return out.stdout.splitlines()


def current_name(name):
    """The policy form of a kernel name of either build."""
    m = re.search(r"predict_tiles_kernel<\(int\)(\d+), \(int\)(\d+), \(int\)(\d+), (\(bool\)\d), (\(bool\)\d)>", name)
    if m:
        ilp, minb, tex, hm, pl = m.groups()
        return name.replace(m.group(0), f"predict_tiles_kernel<qcoh::DuoWalk<(int){ilp}, (int){tex}, (int){minb}>, {hm}, {pl}>")
    m = re.search(r"predict_tiles_nodes8_kernel<\(int\)(\d+), (\(bool\)\d), (\(bool\)\d), \(int\)(\d+), \(int\)(\d+), \(int\)(\d+)>", name)
    if m:
        ilp, hm, pl, minb, tex, ctop = m.groups()
        walk = f"qcoh::NodesWalk<(int){ilp}, (int){tex}, (int){ctop}, (int){minb}>"
        return name.replace(m.group(0), f"predict_tiles_kernel<{walk}, {hm}, {pl}>")
    m = re.search(r"predict_soa_kernel<\(int\)(\d+), \(int\)(\d+), \(bool\)(\d)>", name)
    if m:
        tex, ctop, duo = m.groups()
        nodes = f"qcoh::NodesWalk<(int)4, (int){tex}, (int){ctop}, (int)6>"
        walk = "qcoh::DuoWalk<(int)6, (int)54, (int)5>" if duo == "1" else nodes
        return name.replace(m.group(0), f"predict_soa_kernel<{walk}, {nodes}>")
    return name


def sass(lib):
    text = subprocess.run([f"{CUDA_BIN}/cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    mangled, bodies = [], []
    for line in text.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            mangled.append(m.group(1))
            bodies.append([])
            continue
        if not bodies:
            continue
        line = re.sub(r"/\* 0x[0-9a-f]{16} \*/", "", line)  # encoding
        line = re.sub(r"c\[0x0\]\[0x[0-9a-f]+\]", "c[0x0][PARAM]", line).strip()
        if line:
            bodies[-1].append(line)
    return {current_name(n): b for n, b in zip(demangle(mangled), bodies)}


def ptxas(log):
    """{kernel: [register / spill lines]} of a ptxas -v log."""
    out, cur = {}, None
    for line in open(log):
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            cur = m.group(1)
            out[cur] = []
        elif cur and ("Used" in line or "spill" in line):
            out[cur].append(line.split(":", 1)[-1].strip())
    return {current_name(n): v for n, v in zip(demangle(list(out)), out.values())}


def compare(what, old, new):
    bad = sorted(set(old) ^ set(new))
    for k in bad:
        print(f"{what}: only in {'old' if k in old else 'new'}: {k}")
    same = 0
    for k in sorted(set(old) & set(new)):
        if old[k] == new[k]:
            same += 1
        else:
            bad.append(k)
            print(f"{what}: differs: {k}")
    print(f"{what}: {same} of {len(old)} old / {len(new)} new kernels identical")
    return not bad


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("old")
    ap.add_argument("new")
    ap.add_argument("--ptxas", nargs=2, metavar=("OLD_LOG", "NEW_LOG"))
    a = ap.parse_args()
    ok = compare("sass", sass(a.old), sass(a.new))
    if a.ptxas:
        ok = compare("ptxas", ptxas(a.ptxas[0]), ptxas(a.ptxas[1])) and ok
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
