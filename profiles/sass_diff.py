"""Compare the SASS instruction text of two builds of a translation unit, kernel by kernel (no GPU needed):

    nvcc -cubin -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -o old.cubin so3d_kernels.cu   # parent tree
    nvcc -cubin ... -o new.cubin so3d_kernels.cu                                                              # this tree
    python profiles/sass_diff.py old.cubin new.cubin

Addresses and encodings are dropped; kernel names are demangled and the by-value SE(3) ops, which became templates with a
`false` device-seed argument, are mapped back to their old names.  Prints every pre-existing kernel whose instructions
differ and the kernels only the new build has.
"""
import re, subprocess, sys
def dump(cubin):
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-sass", cubin], capture_output=True, text=True, check=True).stdout
    funcs, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1); funcs[cur] = []; continue
        if cur is None: continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?);", line)
        if m: funcs[cur].append(m.group(1).strip())
    names = list(funcs)
    dem = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.splitlines()
    return {d: funcs[n] for n, d in zip(names, dem)}
def norm(name):
    for a, b in [("SE3QSample2Op<false>", "SE3QSample2Op"), ("SE3QSampleOp<false>", "SE3QSampleOp"),
                 ("SE3PStepOp<true, false>", "SE3PStepOp<true>"), ("SE3PStepOp<false, false>", "SE3PStepOp<false>"),
                 ("SE3PStep2Op<false>", "SE3PStep2Op")]:
        name = name.replace(a, b)
    return re.sub(r"\s+>", ">", name)
old, new = dump(sys.argv[1]), dump(sys.argv[2])
newn = {norm(k): v for k, v in new.items()}
same = diff = 0
old = {norm(k): v for k, v in old.items()}
for k, v in old.items():
    if k not in newn: print("MISSING", k); diff += 1; continue
    if v == newn[k]: same += 1
    else: diff += 1; print("DIFF", k, len(v), len(newn[k]))
extra = [k for k in newn if k not in old]
print(f"pre-existing kernels: {len(old)}, identical instruction text: {same}, differing/missing: {diff}")
print("new kernels:"); [print("  ", k) for k in extra]
