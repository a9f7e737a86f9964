"""LAUUM (K^-1 = U U', lower tiles) on the FP64 DMMA tile engine against the INT8 modular emulation of dgp_lauum8.cuh.

Builds lauum_emul_probe.cu into a temporary directory, runs it at n = 1024 ... 32768 and prints, per size, each kernel's
time (CUDA events), the INT8 GEMM's achieved rate against the data-sheet 4 500 dense INT8 TOPS of a B200, the number of
sampled entries that differ from the exact product rounded once (must be 0), the crossover size, the card and its power
limit.   usage: python tools/lauum_emul_probe.py [n ...]
"""
import json
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
DATASHEET_INT8_TOPS = 4500.0


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
        return out
    except (OSError, subprocess.CalledProcessError, IndexError):
        return "unknown"


def main(sizes):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "lauum_emul_probe")
        subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-o", exe,
                        os.path.join(HERE, "lauum_emul_probe.cu"), "-lcuda"], check=True)
        out = subprocess.run([exe] + [str(n) for n in sizes], capture_output=True, text=True)
        sys.stderr.write(out.stderr)
        if out.returncode != 0:
            raise SystemExit("probe failed (%d)" % out.returncode)
    rows = [json.loads(l) for l in out.stdout.splitlines() if l.startswith("{")]
    print("card: %s" % card())
    print("%7s %4s %10s %10s %10s %10s %10s %8s %7s %9s" % ("n", "b", "dmma_ms", "conv_ms", "i8gemm_ms", "recon_ms",
                                                           "emul_ms", "i8_TOPS", "of_4500", "mismatch"))
    for r in rows:
        print("%7d %4d %10.3f %10.3f %10.3f %10.3f %10.3f %8.0f %7.3f %4d/%d" % (
            r["n"], r["b"], r["dmma_lauum_ms"], r["convert_ms"], r["i8_gemm_ms"], r["recon_ms"], r["emulated_ms"],
            r["i8_tops"], r["i8_tops"] / DATASHEET_INT8_TOPS, r["mismatches"], r["checked"]))
    faster = [r["n"] for r in rows if r["emulated_ms"] < r["dmma_lauum_ms"]]
    slower = [r["n"] for r in rows if r["emulated_ms"] >= r["dmma_lauum_ms"]]
    cross = min((n for n in faster if all(m < n for m in slower)), default=None)
    print("crossover: emulated faster from n = %s on" % cross)
    print(json.dumps({"card": card(), "sizes": rows, "crossover_n": cross}))
    if any(r["mismatches"] for r in rows):
        raise SystemExit("emulated LAUUM differs from the exact rounded product")


if __name__ == "__main__":
    main([int(a) for a in sys.argv[1:]] or [1024, 2048, 4096, 8192, 12288, 16384, 32768])
