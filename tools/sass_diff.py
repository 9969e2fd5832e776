"""Per-kernel SASS comparison of two builds of libptap.so (runs on the CPU: cuobjdump needs no GPU).

    python tools/sass_diff.py OLD/libptap.so NEW/libptap.so

Instructions are compared without their encodings' address comments and blank lines.  Names are normalised for what does not change
code: the hash of anonymous namespaces (it depends on the build directory), the ANY = false parameter that k_trace_bvh gained with the
any-hit mode (`k_trace_bvh<UV, COUNT>` before, `<UV, COUNT, false>` after), and the INST = false parameter and trailing `leaf_model`
argument that k_lbvh_collapse and k_lbvh_single gained with the device TLAS (compared by their demangled names without either).  Exit
status 1 when a kernel of OLD is missing or differs."""
import re
import subprocess
import sys


def kernels(lib):
    out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    d, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1); d[cur] = []
            continue
        if line.startswith("Fatbin"):
            cur = None
        if cur and line.strip():
            d[cur].append(re.sub(r"/\*[0-9a-f]{4,}\*/", "", line).rstrip())
    return d


def norm(name):
    if re.search(r"k_lbvh_(collapse|single)(ILb0EEEv|E)", name):            # the triangle-leaf instantiation, before and after
        d = subprocess.run(["c++filt", name], capture_output=True, text=True, check=True).stdout.strip()
        return re.sub(r", int const\*\)$", ")", re.sub(r"^void ", "", d).replace("<false>", ""))
    name = re.sub(r"_GLOBAL__N__[0-9a-f]+_", "_GLOBAL__N__", name)
    return re.sub(r"(k_trace_bvhILb[01]ELb[01]E)Lb0EE", r"\1E", name)


def main():
    old = {norm(k): v for k, v in kernels(sys.argv[1]).items()}
    new = {norm(k): v for k, v in kernels(sys.argv[2]).items()}
    bad = 0
    for k, v in sorted(old.items()):
        if k not in new:
            print("missing in new:", k); bad += 1
        elif v != new[k]:
            print(f"differs: {k} ({len(v)} -> {len(new[k])} lines)"); bad += 1
    for k in sorted(set(new) - set(old)):
        print("new kernel:", k)
    print(f"{len(old) - bad} of {len(old)} kernels identical")
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
