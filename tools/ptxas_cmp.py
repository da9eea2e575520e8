"""Compare the `ptxas -v` report of every kernel entry of two builds (mh-ppo_b200/build/ptxas.log, written by build.py).

  python tools/ptxas_cmp.py PARENT/mh-ppo_b200/build/ptxas.log mh-ppo_b200/build/ptxas.log > profiles/<name>_ptxas_cmp.txt

Per entry: registers, stack frame / spill stores / spill loads (bytes).  A template parameter appended with a default keeps the
old instance under a longer name (`k_ppo_grad<16, 0, false>` is now `k_ppo_grad<16, 0, false, false>`): a parent entry that is
missing by name is matched to the new entry whose name is the parent's with `, (bool)0` (false) added to its template arguments,
and, failing that, to the one such entry whose parameter list starts with the parent's and goes on (a defaulted trailing kernel
parameter that only the new instance reads: `k_adam2_clip<false>(..., double *)` is now `k_adam2_clip<false, false>(..., double *,
mhppo::AdaptArgs)`)."""
import re
import subprocess
import sys

CUFILT = "/usr/local/cuda/bin/cu++filt"


def entries(path):
    out, cur, frame = {}, None, None
    for line in open(path):
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            cur, frame = m.group(1), None
            continue
        m = re.search(r"Function properties for (\S+)", line)
        if m:
            frame = m.group(1)
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur is not None and frame == cur:
            out.setdefault(cur, {})["stack"] = tuple(int(v) for v in m.groups())
            continue
        m = re.search(r"Used (\d+) registers", line)
        if m and cur is not None:
            out.setdefault(cur, {})["regs"] = int(m.group(1))
            cur = None
    return out


def demangle(names):
    r = subprocess.run([CUFILT], input="\n".join(names), capture_output=True, text=True, check=True)
    return dict(zip(names, r.stdout.splitlines()))


def fmt(e):
    return "%4d  %d/%d/%d" % ((e["regs"],) + e.get("stack", (0, 0, 0)))


def main(old_log, new_log):
    old, new = entries(old_log), entries(new_log)
    dn = demangle(sorted(set(old) | set(new)))
    by_name_new = {dn[k]: k for k in new}
    matched, changed, missing = {}, [], []
    for k in sorted(old, key=lambda k: dn[k]):
        name = dn[k]
        alt = name.replace(">(", ", (bool)0>(", 1)
        nk = by_name_new.get(name) or by_name_new.get(alt)
        if nk is None and alt.endswith(")"):
            longer = [k2 for n2, k2 in by_name_new.items() if n2.startswith(alt[:-1] + ", ")]
            nk = longer[0] if len(longer) == 1 else None
        if nk is None:
            missing.append(name)
            continue
        matched[nk] = k
        if new[nk] != old[k]:
            changed.append((name, fmt(old[k]), fmt(new[nk])))
    print("ptxas -v of every sm_100a kernel (nvcc, -gencode arch=compute_100a,code=sm_100a), parent commit vs this change.")
    print("Columns: registers, stack frame / spill stores / spill loads (bytes).\n")
    for k in sorted(set(new) - set(matched), key=lambda k: dn[k]):
        print("new        %-90s %s" % (dn[k], fmt(new[k])))
    for name, a, b in changed:
        print("changed    %-90s %s -> %s" % (name, a, b))
    for name in missing:
        print("missing    %s" % name)
    renamed = sum(1 for nk, k in matched.items() if dn[nk] != dn[k])
    print("\n%d kernel entries of the parent build found in this build (%d of them under a name with the new defaulted template "
          "parameter or trailing kernel parameter); %d with different registers, stack frame or spills; %d missing"
          % (len(matched), renamed, len(changed), len(missing)))


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2])
