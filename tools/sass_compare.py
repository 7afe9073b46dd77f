"""Compare the SASS of two builds of the library, kernel by kernel (needs cuobjdump / cu++filt, no GPU).

    python tools/sass_compare.py OLD.so NEW.so

Kernels are matched by demangled name.  Trailing template arguments that newer builds added to a kernel, at their
values for the existing instantiations, are dropped first (the exclusion flag `false` of score_topk_kernel /
topk_rows_kernel, then the epilogue `0` of score_topk_kernel), so an existing instantiation is compared with its own
successor.  Only instruction lines are compared.  Prints one line per kernel; exits 1 when a kernel of OLD
is missing from NEW or compiles differently."""
import os
import re
import subprocess
import sys

CUDA_BIN = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin")


def kernel_name(mangled):
    d = subprocess.run([os.path.join(CUDA_BIN, "cu++filt"), mangled], capture_output=True, text=True, check=True).stdout
    d = re.sub(r"\((int|bool)\)", "", d.strip())
    d = re.match(r"(?:void )?([\w:]+(<[^>]*>)?)", d).group(1).replace(" ", "")
    d = re.sub(r"^(mr::st::score_topk_kernel<\d+,\d+,\d+,\d+,\d+),0>$", r"\1>", d)
    d = re.sub(r"^(mr::st::score_topk_kernel<\d+,\d+,\d+,\d+),0>$", r"\1>", d)
    return d.replace("topk_rows_kernel<0>", "topk_rows_kernel")


def kernels(path):
    out = subprocess.run([os.path.join(CUDA_BIN, "cuobjdump"), "-sass", path], capture_output=True, text=True, check=True).stdout
    res, cur = {}, None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = kernel_name(m.group(1))
            res[cur] = []
        elif cur and re.match(r"\s+/\*[0-9a-f]{4,}\*/", line):
            res[cur].append(line.strip())
    return res


def main():
    old, new = kernels(sys.argv[1]), kernels(sys.argv[2])
    bad = 0
    for name in sorted(old):
        state = "missing" if name not in new else "same" if new[name] == old[name] else "DIFFERS"
        bad += state != "same"
        print(f"{state:8s} {name}")
    for name in sorted(set(new) - set(old)):
        print(f"{'new':8s} {name}")
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
