"""The lower-right quadrant update of a split Cholesky factorisation (A22 -= L21 L21', K = 128 hs) on the FP64 DMMA tile
engine, as the rank-512 trailing updates of the panels left of hs, against the INT8 modular emulation of dgp_lauum8.cuh,
as syrk_i8 of dgp_api.cu launches it.

Builds syrk_emul_probe.cu into a temporary directory, runs it for the cases npad:hs (default n = 16384 and 32768 at
hs = nb/3, 3nb/8 and nb/2 rounded to 8, and n = 12288 at 3nb/8) and prints, per case, the DMMA time and rate, the emulated
time split into conversion, INT8 GEMM and reconstruction, the INT8 GEMM's rate against the data-sheet 4 500 dense INT8
TOPS of a B200, the number of sampled entries (at least 500) that differ from the exact product rounded once and then
subtracted (must be 0), the card and its power limit.
   usage: python tools/syrk_emul_probe.py [npad:hs ...]
"""
import json
import os
import subprocess
import sys
import tempfile

from lauum_emul_probe import DATASHEET_INT8_TOPS, HERE, card


def main(cases):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "syrk_emul_probe")
        subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-o", exe,
                        os.path.join(HERE, "syrk_emul_probe.cu"), "-lcuda"], check=True)
        out = subprocess.run([exe] + cases, capture_output=True, text=True)
        sys.stderr.write(out.stderr)
        if out.returncode != 0:
            raise SystemExit("probe failed (%d)" % out.returncode)
    rows = [json.loads(l) for l in out.stdout.splitlines() if l.startswith("{")]
    print("card: %s" % card())
    print("%6s %4s %9s %7s | %8s %8s %8s %9s | %7s %7s %9s %9s" % (
        "npad", "hs", "dmma_ms", "TF", "convert", "i8gemm", "recon", "emul_ms", "i8TOPS", "of4500", "mismatch", "dmma_rel"))
    for r in rows:
        print("%6d %4d %9.3f %7.1f | %8.3f %8.3f %8.3f %9.3f | %7.0f %7.3f %4d/%d %9.2e" % (
            r["npad"], r["hs"], r["dmma_ms"], r["dmma_tflops"], r["convert_ms"], r["i8_gemm_ms"], r["recon_ms"],
            r["emulated_ms"], r["i8_tops"], r["i8_tops"] / DATASHEET_INT8_TOPS, r["mismatches"], r["checked"],
            r["dmma_max_rel_diff"]))
    print(json.dumps({"card": card(), "cases": rows}))
    if any(r["mismatches"] for r in rows):
        raise SystemExit("emulated quadrant update differs from the exact rounded product")


if __name__ == "__main__":
    main(sys.argv[1:] or ["16384:40", "16384:48", "16384:64", "32768:88", "32768:96", "32768:128", "12288:32"])
