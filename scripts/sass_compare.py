"""Compares the SASS of the CPU-mode solver kernels in two builds of tvl1_engine.cu, instruction by instruction
(symbol names aside: the cv::cuda-semantics instantiations add a `false` template argument).  No GPU needed:

    nvcc <the flags of csrc/build.py> -cubin -o old.cubin tvl1_engine.cu     (in each tree)
    python scripts/sass_compare.py old.cubin new.cubin
"""
import re
import subprocess
import sys

KERNELS = ("k_outer", "k_iterate", "k_warp", "k_median5")


def functions(cubin):
    out = subprocess.check_output(["cuobjdump", "-sass", cubin], text=True)
    fs, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = subprocess.check_output(["c++filt", m.group(1)], text=True).strip()
            fs[cur] = []
        elif cur and re.search(r"/\*[0-9a-f]{4}\*/", line):
            ins = re.sub(r"/\*[0-9a-f]{4}\*/", "", line).split(";")[0].strip()
            fs[cur].append(re.sub(r"_Z\w+", "SYM", ins))
    return fs


def main():
    old, new = functions(sys.argv[1]), functions(sys.argv[2])
    bad = 0
    for name in sorted(old):
        if not any(k in name for k in KERNELS) or "_cuda" in name:
            continue
        match = [n for n in new if "true" not in n and (n == name or n.replace(", false>", ">") == name)]
        if not match:
            print("MISSING", name)
            bad += 1
            continue
        same = old[name] == new[match[0]]
        bad += not same
        print("%s %5d %5d  %s" % ("same" if same else "DIFF", len(old[name]), len(new[match[0]]), name))
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
