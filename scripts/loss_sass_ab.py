"""Instruction-level A/B of the compiled loss kernels of two objects (no GPU needed).

    nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC --expt-relaxed-constexpr \\
         -c gcn-string_b200/csrc/loss.cu -o new_loss.o        # and the same for the other revision's loss.cu
    python scripts/loss_sass_ab.py base_loss.o new_loss.o

Every kernel of the first object is matched with the kernel of the same demangled name in the second, after dropping
the default template flag of the weighted policies (`Xent<1024, 1, false>` is `Xent<1024, 1>`) and the parameter list.
It prints `same` or `DIFF` with the instruction counts, compares the instruction text without addresses or encodings,
and exits 1 if a kernel differs or is missing.
"""
import re
import subprocess
import sys


def kernels(path):
    out = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    found, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            cur = found.setdefault(m.group(1), [])
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(.*?);", line)
        if m and cur is not None:
            cur.append(m.group(1).strip())
    return found


def key(mangled):
    name = subprocess.run(["c++filt", mangled], capture_output=True, text=True, check=True).stdout.strip()
    name = name.replace(", false>", ">").replace(">>", "> >")
    return re.sub(r"\(.*\)$", "", name)


def main(a_path, b_path):
    a = {key(k): v for k, v in kernels(a_path).items()}
    b = {key(k): v for k, v in kernels(b_path).items()}
    bad = 0
    for name in sorted(a):
        if name not in b:
            print("MISSING", name)
            bad += 1
            continue
        same = a[name] == b[name]
        bad += not same
        print("same " if same else "DIFF ", len(a[name]), len(b[name]), name)
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1], sys.argv[2]))
