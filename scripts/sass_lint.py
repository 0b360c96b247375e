"""SASS lint for the streaming kernels: in the main row-batch loop all U data loads and their weight records
must be issued before the first FFMA2 that consumes them (ptxas sometimes sinks loads below the first row's
arithmetic when registers get tight, which serialises the HBM requests -- measured -15 % on cfg2).
usage: python scripts/sass_lint.py [lib.so]   -> prints, per aa_stream_kernel instantiation, the longest run of
128/64-bit LDGs that precedes an FFMA2 and flags the ones where that run is shorter than U."""
import re, shutil, subprocess, sys, os
lib = sys.argv[1] if len(sys.argv) > 1 else os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "interpolate_antialiasing_b200", "_build", "libaa_resize_b200.so")
cuobjdump = shutil.which("cuobjdump") or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")
out = subprocess.run([cuobjdump, "-sass", lib], capture_output=True, text=True, check=True).stdout
cur, funcs = None, {}
for line in out.splitlines():
    m = re.search(r"Function : (\S+)", line)
    if m:
        cur = m.group(1); funcs[cur] = []; continue
    if cur and re.match(r"\s+/\*[0-9a-f]{4}\*/", line):
        funcs[cur].append(line.split("*/", 1)[1].strip())
bad = 0
for name, ins in funcs.items():
    k = re.search(r"aa_stream_kernelILi(\d+)ELi(\d+)E(\w)Li(\d+)ELi(\d+)ELi(\d+)ELb(\d)ELb(\d)ELb(\d)", name)
    if not k: continue
    A, VEC, ty, NT, U, MINB, GEN, PAD, PF = k.groups()
    U = int(U)
    # runs of wide data loads (the .NA = no-allocate data rows) between FFMA2s
    best, run = 0, 0
    for i in ins:
        if i.startswith("LDG") and ".NA" in i: run += 1
        elif "FFMA" in i:
            best = max(best, run); run = 0
    flag = "" if best >= U else "   <-- loads not hoisted"
    bad += best < U
    print(f"A={A} VEC={VEC} {ty} NT={NT} U={U} GEN={GEN} PAD={PAD} PF={PF}: {best} data loads before the first FMA{flag}")
print("flagged:", bad)
