"""Function-by-function comparison of the SASS of two builds of libtfglacier.so (no GPU needed).

    python scripts/sass_compare.py OLD.so NEW.so

Every kernel of OLD must appear in NEW with identical instructions.  Names are demangled (cu++filt) and normalised:
the per-build hash of anonymous namespaces is dropped, and a trailing `false` template argument that NEW's
`run_kernel` has beyond OLD's (a new template flag whose default keeps the old kernels) is removed, so that
`run_kernel<P, ..., PAR, false>` of NEW is compared with `run_kernel<P, ..., PAR>` of OLD.  Addresses inside the
listing (/*0a30*/ comments, branch targets) are compared as they are: an identical kernel has identical offsets.
Prints one line per kernel of OLD and the kernels only NEW has; exit code 1 if any kernel of OLD differs or is missing.
"""
import re
import subprocess
import sys
from pathlib import Path

CUDA_BIN = Path("/usr/local/cuda/bin")


def tool(name):
    p = CUDA_BIN / name
    return str(p) if p.exists() else name


def functions(so):
    text = subprocess.run([tool("cuobjdump"), "-sass", str(so)], capture_output=True, text=True, check=True).stdout
    out, name, body = {}, None, []
    for line in text.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            if name:
                out[name] = body
            name, body = m.group(1), []
        elif name and line.strip().startswith("/*"):   # instructions and their encodings, not the fatbin headers
            body.append(line.strip())
    if name:
        out[name] = body
    names = list(out)
    dem = subprocess.run([tool("cu++filt")], input="\n".join(names), capture_output=True, text=True, check=True).stdout.split("\n")
    return {re.sub(r"\(anonymous namespace\)::|_GLOBAL__N__\w+::", "", d): out[n] for n, d in zip(names, dem)}


def n_args(name):
    m = re.search(r"run_kernel<(.*?)>\(", name)
    return len(m.group(1).split(",")) if m else 0


def main(old_so, new_so):
    old, new = functions(old_so), functions(new_so)
    k_old = max((n_args(n) for n in old), default=0)
    norm = {}
    for n, body in new.items():
        key = n
        if n_args(n) == k_old + 1:
            key = re.sub(r"run_kernel<(.*), (?:false|\(bool\)0)>\(", r"run_kernel<\1>(", n)
        norm[key] = (n, body)
    bad = 0
    for n, body in old.items():
        if n not in norm:
            print(f"MISSING   {n}")
            bad += 1
        elif norm[n][1] != body:
            print(f"DIFFERENT {n}")
            bad += 1
        else:
            print(f"identical {n}  ({len(body)} lines)")
    matched = {v[0] for k, v in norm.items() if k in old}
    for n in new:
        if n not in matched:
            print(f"new       {n}  ({len(new[n])} lines)")
    print(f"{len(old) - bad} of {len(old)} kernels of {old_so} identical in {new_so}")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1], sys.argv[2]))
