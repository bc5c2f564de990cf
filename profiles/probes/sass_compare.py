"""Compare the SASS of two builds of libbcg_b200.so kernel by kernel.

    python profiles/probes/sass_compare.py OLD.so NEW.so

Kernels are matched by demangled name, with trailing `false` template arguments (the per-env rows and episode-ends flags:
`move_kernel<8, false, false>`) and the trailing BcgEnvRows / episode-ends parameters dropped, so that the instantiations
without rows or ends line up with the kernels of a build that had neither.  Branch-target addresses are ignored.  Prints
`same` or `DIFFERENT` (with the count of changed instructions) per kernel; instantiations without a counterpart are
listed as new.
"""
import difflib
import re
import subprocess
import sys

CUDA = "/usr/local/cuda/bin/"


def kernels(so):
    out = subprocess.run([CUDA + "cuobjdump", "-sass", so], capture_output=True, text=True, check=True).stdout
    res, name = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = m.group(1)
            res[name] = []
            continue
        if name is None:
            continue
        ins = re.sub(r"/\*\s*(0x)?[0-9a-f]+\s*\*/", "", line).strip()
        if not ins or ins.startswith("..."):
            continue
        if re.match(r"(@!?U?P\w+ )?(BRA|CALL|BSSY|JMP|BREAK|WARPSYNC|BMOV)", ins):
            ins = re.sub(r"0x[0-9a-f]+ ;$", "ADDR ;", ins)
        res[name].append(ins)
    return res


def key(name):
    d = subprocess.run([CUDA + "cu++filt", name], capture_output=True, text=True).stdout.strip()
    d = re.sub(r"^void ", "", d.replace("(anonymous namespace)::", ""))
    d = d.replace(", BcgEpisodeEnds)", ")").replace(", BcgEnvRows, int *)", ")").replace(", BcgEnvRows)", ")")
    while True:
        k = d.replace("<(bool)0>", "").replace(", (bool)0>", ">")
        if k == d:
            return d
        d = k


def main(old, new):
    a = {key(n): v for n, v in kernels(old).items()}
    b = {key(n): v for n, v in kernels(new).items()}
    for k in sorted(set(a) | set(b)):
        if k not in a:
            print("new        %s" % k)
        elif k not in b:
            print("GONE       %s" % k)
        elif a[k] == b[k]:
            print("same %5d  %s" % (len(a[k]), k))
        else:
            sm = difflib.SequenceMatcher(None, a[k], b[k], autojunk=False)
            changed = sum(max(i2 - i1, j2 - j1) for t, i1, i2, j1, j2 in sm.get_opcodes() if t != "equal")
            print("DIFFERENT %5d -> %5d, %d changed  %s" % (len(a[k]), len(b[k]), changed, k))


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2])
