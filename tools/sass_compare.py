"""Compares the SASS of every kernel of two builds of wfa_kernels.o, function by function.

usage: cuobjdump -sass <parent>/wfa-gpu_b200/build/csrc/wfa_kernels.o > parent.sass
       cuobjdump -sass wfa-gpu_b200/build/csrc/wfa_kernels.o > branch.sass
       python tools/sass_compare.py parent.sass branch.sass

A branch kernel `wfa_exact_kernel<..., false>` with one template argument more than the parent's instantiations is
compared with the parent's kernel of the same arguments without that trailing `false`; with a trailing `true` it is
listed as new.  Exit code 1 if any pre-existing kernel differs or is missing."""
import re
import subprocess
import sys


def blocks(path):
    out, name, buf = {}, None, []
    for line in open(path):
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            if name:
                out[name] = buf
            name, buf = m.group(1), []
        elif name is not None:
            buf.append(line.rstrip())
    if name:
        out[name] = buf
    return out


def demangle(names):
    r = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True, check=True)
    return dict(zip(names, r.stdout.split("\n")))


def key(sig, n_parent_args):
    m = re.match(r"void wfagpu::wfa_exact_kernel<(.*)>\(", sig)
    if not m:
        return sig
    args = m.group(1).split(", ")
    if len(args) > n_parent_args:
        if args[-1] == "true":
            return None
        args = args[:-1]
    return "wfa_exact_kernel<" + ", ".join(args) + ">"


def main():
    old, new = blocks(sys.argv[1]), blocks(sys.argv[2])
    do, dn = demangle(list(old)), demangle(list(new))
    n_args = min(len(re.match(r"void wfagpu::wfa_exact_kernel<(.*)>\(", s).group(1).split(", "))
                 for s in do.values() if s.startswith("void wfagpu::wfa_exact_kernel<"))
    ref = {key(do[k], n_args): v for k, v in old.items()}
    same, bad, fresh, seen = 0, [], [], set()
    for k, v in new.items():
        kk = key(dn[k], n_args)
        if kk is None:
            fresh.append(dn[k])
            continue
        seen.add(kk)
        if ref.get(kk) == v:
            same += 1
        else:
            bad.append(kk)
    missing = sorted(set(ref) - seen)
    print(f"identical={same} differing={len(bad)} missing={len(missing)} new={len(fresh)}")
    for k in bad:
        print("  differs:", k)
    for k in missing:
        print("  missing:", k)
    for k in fresh:
        print("  new:", k)
    return 1 if bad or missing else 0


if __name__ == "__main__":
    sys.exit(main())
