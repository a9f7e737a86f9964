"""One merge of the recursive triangular inverse (M' = U11 L21', U12 = -M' T22') on the FP64 DMMA tile engine against the
INT8 modular emulation of dgp_lauum8.cuh, as inv_merge_i8 of dgp_api.cu launches it.

Builds inv_emul_probe.cu into a temporary directory, runs it for merges hb | w2 (default 16|16, 32|32, 64|64, 128|128 and the
ragged 64|33, 64|16) and prints, per merge, the DMMA time of both products and the emulated time per product (conversion of
both operands, INT8 GEMM, reconstruction), the INT8 GEMMs' rate against the data-sheet 4 500 dense INT8 TOPS of a B200,
the number of sampled entries that differ from the exact product rounded once (must be 0), the card and its power limit.
   usage: python tools/inv_emul_probe.py [hb:w2 ...]
"""
import json
import os
import subprocess
import sys
import tempfile

from lauum_emul_probe import DATASHEET_INT8_TOPS, HERE, card


def main(merges):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "inv_emul_probe")
        subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-o", exe,
                        os.path.join(HERE, "inv_emul_probe.cu"), "-lcuda"], check=True)
        out = subprocess.run([exe] + merges, capture_output=True, text=True)
        sys.stderr.write(out.stderr)
        if out.returncode != 0:
            raise SystemExit("probe failed (%d)" % out.returncode)
    rows = [json.loads(l) for l in out.stdout.splitlines() if l.startswith("{")]
    print("card: %s" % card())
    print("%4s %4s %9s | %8s %8s %8s | %8s %8s %8s | %9s %7s %7s %9s" % (
        "hb", "w2", "dmma_ms", "M'conv", "M'gemm", "M'recon", "U conv", "U gemm", "U recon", "emul_ms", "i8TOPS", "of4500",
        "mismatch"))
    for r in rows:
        print("%4d %4d %9.3f | %8.3f %8.3f %8.3f | %8.3f %8.3f %8.3f | %9.3f %7.0f %7.3f %4d/%d" % (
            r["hb"], r["w2"], r["dmma_ms"], r["m_convert_ms"], r["m_i8_gemm_ms"], r["m_recon_ms"], r["u_convert_ms"],
            r["u_i8_gemm_ms"], r["u_recon_ms"], r["emulated_ms"], r["i8_tops"], r["i8_tops"] / DATASHEET_INT8_TOPS,
            r["mismatches"], r["checked"]))
    print(json.dumps({"card": card(), "merges": rows}))
    if any(r["mismatches"] for r in rows):
        raise SystemExit("emulated merge differs from the exact rounded product")


if __name__ == "__main__":
    main(sys.argv[1:] or ["16:16", "32:32", "64:64", "128:128", "64:33", "64:16"])
