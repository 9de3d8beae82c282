"""Compares two builds of libv5ela.so kernel by kernel: the cuobjdump -sass instruction text (addresses, encodings and symbol names
stripped) and the -Xptxas -v resources (registers, barriers, shared memory, stack, spills). A change that only moves host code or
renames the namespace of a kernel's parameter type must leave both identical.

usage: python profiles/sass_compare.py OLD.so OLD_BUILD.log NEW.so NEW_BUILD.log
where a build log is the output of `make -C fake-video-detection-engine_b200/csrc -B` (the Makefile passes -Xptxas -v) and the
library is the libv5ela.so that build wrote. Kernels are matched by their demangled name without the parameter list, so that
`v5::ela_fused_kernel<true, false, false>` of both builds meet whatever namespace KParams lives in. Exit status 1 on any difference."""
import collections
import re
import subprocess
import sys


def demangle(names):
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True, check=True).stdout.splitlines()
    return {n: re.sub(r"\(.*\)$", "", d) for n, d in zip(names, out)}


def sass_by_kernel(so):
    text = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True, check=True).stdout
    funcs, cur = collections.OrderedDict(), None
    for ln in text.splitlines():
        m = re.search(r"Function : (\S+)", ln)
        if m:
            cur = m.group(1)
            funcs[cur] = []
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;", ln)
        if m and cur:
            funcs[cur].append(re.sub(r"_Z\w+", "<sym>", m.group(1)))
    names = demangle(list(funcs))
    return {names[k]: v for k, v in funcs.items()}


def ptxas_by_function(log):
    res, cur = collections.defaultdict(list), None
    for ln in open(log):
        m = re.search(r"Function properties for (\S+)", ln) or re.search(r"Compiling entry function '(\S+)'", ln)
        if m:
            cur = m.group(1)
            continue
        if cur and ("bytes stack frame" in ln or ln.startswith("ptxas info    : Used")):
            res[cur].append(re.sub(r"^ptxas info\s+:\s+", "", ln.strip()))
    names = demangle(list(res))
    return {names[k]: v for k, v in res.items()}


def main(old_so, old_log, new_so, new_log):
    bad = 0
    old, new = sass_by_kernel(old_so), sass_by_kernel(new_so)
    print(f"# SASS: {len(old)} kernels in {old_so}, {len(new)} in {new_so}")
    for k in sorted(set(old) | set(new)):
        if k not in old or k not in new:
            print(f"only in {'new' if k in new else 'old'}: {k}")
            bad += 1
            continue
        same = old[k] == new[k]
        bad += not same
        print(f"{'identical' if same else 'DIFFERS  '} {len(old[k]):6d} / {len(new[k]):6d} instructions  {k}")
    old, new = ptxas_by_function(old_log), ptxas_by_function(new_log)
    print(f"# -Xptxas -v: {len(old)} functions in {old_log}, {len(new)} in {new_log}")
    for k in sorted(set(old) | set(new)):
        same = old.get(k) == new.get(k)
        bad += not same
        if not same:
            print(f"DIFFERS {k}\n  old: {old.get(k)}\n  new: {new.get(k)}")
    print(f"# {'no differences' if bad == 0 else f'{bad} differences'}"
          f" ({sum(1 for k in new if 'ela_fused_kernel' in k)} ela_fused_kernel entries in the resource report)")
    return 1 if bad else 0


if __name__ == "__main__":
    if len(sys.argv) != 5:
        sys.exit(__doc__)
    sys.exit(main(*sys.argv[1:]))
