"""Compare the SASS of every kernel between two builds, function by function (instruction text only: addresses, encodings
and comments stripped).  Usage: python profiles/scripts/sass_compare.py OLD_BUILD_DIR NEW_BUILD_DIR stream fcnet ...
(the directories hold the <name>.o objects ddrl_b200/build.py writes to ddrl_b200/csrc/_build/).  A function whose mangled
name changed is paired through RENAMED."""
import re
import subprocess
import sys

RENAMED = {  # graphnet_fwd_warp_kernel became a template on SAMPLE; <false> is the former kernel
    "_ZN4ddrl24graphnet_fwd_warp_kernelEPKfPKiS1_S1_liPfS4_":
        "_ZN4ddrl24graphnet_fwd_warp_kernelILb0EEEvPKfPKiS2_S2_liPfS5_S2_S5_S5_",
    # fcnet_forward_kernel became a template on CUP (leg coupling); <false> is the former kernel
    "_ZN4ddrl20fcnet_forward_kernelEPKfS1_S1_PKdfliiPfS4_S4_S1_S4_S4_":
        "_ZN4ddrl20fcnet_forward_kernelILb0EEEvPKfS2_S2_PKdfliiPfS5_S5_S2_S5_S5_PKiS2_Pi"}


def functions(obj):
    out = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True, check=True).stdout
    res, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            cur = m.group(1)
            res[cur] = []
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4}\*/\s*(.*?)\s*;?\s*(/\*.*\*/)?\s*$", line)
        if cur and m:
            res[cur].append(re.sub(r"\s+", " ", m.group(1)))
    return res


def main():
    old_dir, new_dir, *srcs = sys.argv[1:]
    for src in srcs:
        old, new = functions(f"{old_dir}/{src}.o"), functions(f"{new_dir}/{src}.o")
        same = 0
        for f, body in old.items():
            g = RENAMED.get(f, f)
            if new.get(g) == body:
                same += 1
            else:
                print(f"{src}: {f} {'missing' if g not in new else 'differs'}")
        added = sorted(set(new) - {RENAMED.get(f, f) for f in old})
        print(f"{src}.cu: {same} of {len(old)} functions identical SASS; added: {added}")


if __name__ == "__main__":
    main()
