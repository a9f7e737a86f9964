"""Instruction counts per kernel from `cuobjdump -sass` of the built library -> profiles/sass_<tag>.txt (run here, no GPU)."""
import collections, os, re, subprocess, sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "discontinuum_b200", "libdgp.so")
COLS = ["DMMA", "UTMALDG", "SYNCS", "USETMAXREG", "DFMA", "MUFU", "LDS", "STL", "LDL"]
HEAD = """# cuobjdump -sass discontinuum_b200/libdgp.so, instruction counts per kernel (tools/sass_profile.py)
# build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -shared -Xcompiler -fPIC -o libdgp.so dgp_api.cu (CUDA 12.9)
# DMMA = FP64 tensor-core MMA (mma.sync.m8n8k4.f64; tcgen05 has no f64 kind), UTMALDG = TMA tensor load (cp.async.bulk.tensor),
# SYNCS = mbarrier ops, USETMAXREG = warpgroup register reallocation (setmaxnreg), STL / LDL = local-memory spills (none inside
# the DMMA main loops).  UTCIMMA (tcgen05.mma kind::i8) appears in k_l8_gemm only: the INT8 modular LAUUM of dgp_lauum8.cuh."""


def main(tag):
    sass = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True, check=True).stdout
    names = subprocess.run(["c++filt"], input="\n".join(re.findall(r"Function : (\S+)", sass)), capture_output=True, text=True).stdout.split("\n")
    counts, order, cur, k = {}, [], None, 0
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = re.sub(r"\(int\)", "", names[k].split("(")[0]).replace("void ", "") if "<" not in names[k] else re.sub(r"\(int\)", "", names[k][:names[k].index(">") + 1]).replace("void ", "")
            k += 1
            counts[cur] = collections.Counter(); order.append(cur)
            continue
        m = re.search(r"^\s+/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_]+)", line)
        if m and cur:
            counts[cur][m.group(1).split(".")[0]] += 1
    out = [HEAD, f"{'kernel':70s}" + "".join(f"{c:>11s}" for c in COLS)]
    for name in order:
        out.append(f"{name:70s}" + "".join(f"{counts[name][c]:11d}" for c in COLS))
    tot = collections.Counter()
    for c in counts.values():
        tot.update(c)
    out.append(f"{'all kernels':70s}" + "".join(f"{tot[c]:11d}" for c in COLS))
    out.append("tcgen05 (UTC*MMA) instructions: %d" % sum(v for k_, v in tot.items() if k_.startswith("UTC") and "MMA" in k_))
    path = os.path.join(ROOT, "profiles", f"sass_{tag}.txt")
    open(path, "w").write("\n".join(out) + "\n")
    print(path, len(order), "kernels")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else "rXX")
