"""Compare the SASS of every kernel of one build of the attention library with the same instantiation in another:
instruction text and encoding, kernel by kernel.  The fused-prologue kernels gained a trailing `bool MASK = false`
template argument with the padding mask; it is stripped from the new names to match, and the MASK = true kernels are
listed as new.

    nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 --expt-relaxed-constexpr -cubin \
         -o new.cubin devis_b200/csrc/msda_capi.cu          (and base.cubin from the parent commit's tree)
    python benchmarks/sass_compare.py base.cubin new.cubin report.txt
"""
import re
import subprocess
import sys

CUOBJ = "/usr/local/cuda/bin/cuobjdump"


def functions(cubin):
    txt = subprocess.run([CUOBJ, "-sass", cubin], capture_output=True, text=True, check=True).stdout
    funcs, name, body = {}, None, []
    for line in txt.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            if name:
                funcs[name] = body
            name, body = m.group(1), []
        elif name and re.match(r"\s*/\*[0-9a-f]{4,}\*/", line):
            body.append(re.sub(r"\s+", " ", line.strip()))
        elif name and re.match(r"\s*/\* 0x[0-9a-f]+ \*/", line):
            body.append(line.strip())
    if name:
        funcs[name] = body
    names = list(funcs)
    dem = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.splitlines()
    return {d: funcs[n] for n, d in zip(names, dem)}


def main(base, new, out):
    b, n = functions(base), functions(new)
    norm = {}
    for name, body in n.items():
        if "tmsda_fused_" in name:
            if re.search(r", true>\(devis::FusedArgs\)", name):
                continue                      # MASK = true: new kernels
            name = re.sub(r", false>\(devis::FusedArgs\)", ">(devis::FusedArgs)", name)
        norm[name] = body
    lines, same, diff, missing = [], 0, 0, 0
    for name in sorted(b):
        if name not in norm:
            missing += 1
            lines.append(f"MISSING  {name}")
        elif norm[name] == b[name]:
            same += 1
            lines.append(f"same     {len(b[name]) // 2:6d} instr  {name}")
        else:
            diff += 1
            lines.append(f"DIFFERS  {name}")
    new_only = [x for x in n if "tmsda_fused_" in x and ", true>(devis::FusedArgs)" in x]
    head = (f"kernels in the parent's library: {len(b)}; identical SASS (instructions and encodings): {same}; "
            f"different: {diff}; missing: {missing}\nnew MASK = true instantiations: {len(new_only)}\n")
    open(out, "w").write(head + "\n".join(lines) + "\n\nnew:\n" + "\n".join(sorted(new_only)) + "\n")
    print(head)
    return 0 if diff == 0 and missing == 0 else 1


if __name__ == "__main__":
    sys.exit(main(*sys.argv[1:4]))
