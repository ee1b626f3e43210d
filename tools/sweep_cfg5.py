"""BASELINE.json configs[4]: nhidden in {50,100,200,400,800} x T in {128,512,2048}, 128 lines per GPU, one bench line per
cell (bench.py is run as a subprocess per cell, so every cell gets a fresh handle and its own clock samples).

    python tools/sweep_cfg5.py [--gpus N] [--steps K] [--out profiles/r2_cfg5_n1.jsonl] [--cells 50x128,800x2048]

With --gpus N > 1 every cell is launched through torch.distributed.run (128 lines per rank, weak scaling).
Prints a markdown table at the end: ms/step, Mpx/s, recurrent kernel variant, TFLOP/s of the recurrence and its share of the
step, HBM GB/s of the CTC and update kernels."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=128)
    ap.add_argument("--out", default=None)
    ap.add_argument("--cells", default=None, help="comma list of NHxT, default: the whole grid")
    a = ap.parse_args()
    cells = [(nh, T) for nh in (50, 100, 200, 400, 800) for T in (128, 512, 2048)]
    if a.cells:
        cells = [tuple(int(v) for v in c.split("x")) for c in a.cells.split(",")]
    rows = []
    out = open(a.out, "w") if a.out else None
    for nh, T in cells:
        cmd = [sys.executable]
        if a.gpus > 1:
            cmd += ["-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(a.gpus), "--master-addr", "127.0.0.1",
                    "--master-port", str(29500 + (nh + T) % 400)]
        cmd += [os.path.join(ROOT, "bench.py"), "--gpus", str(a.gpus), "--steps", str(a.steps), "--warmup", str(a.warmup),
                "--nhidden", str(nh), "--batch", str(a.batch), "--T", str(T), "--Tmax", "0", "--no-extras",
                "--no-cpu-baseline"]
        r = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT)
        line = [ln for ln in r.stdout.split("\n") if ln.startswith("{")]
        if r.returncode != 0 or not line:
            print("cell %dx%d failed: %s" % (nh, T, r.stderr[-400:]), file=sys.stderr)
            continue
        j = json.loads(line[-1])
        j["cell"] = {"nhidden": nh, "T": T, "batch": a.batch}
        rows.append(j)
        if out:
            out.write(json.dumps(j) + "\n")
            out.flush()
    print("| nhidden | T | GPUs | ms/step | Mpx/s | e2e Mpx/s | recurrence | fwd+bwd ms (share) | recurrence TFLOP/s (frac of peak) | ctc GB/s | update GB/s | clocks MHz |")
    print("|---|---|---|---|---|---|---|---|---|---|---|---|")
    for j in rows:
        k = j["kernels"]
        rec_ms = k.get("lstm_fwd", {}).get("ms_per_step", 0.0) + k.get("lstm_bwd", {}).get("ms_per_step", 0.0)
        nh, T = j["cell"]["nhidden"], j["cell"]["T"]
        fl = 2 * 2.0 * 2 * j["config"]["columns_per_gpu"] * 4 * nh * nh
        tf = fl / (rec_ms / 1e3) / 1e12 if rec_ms > 0 else 0.0
        print("| %d | %d | %d | %.3f | %.1f | %.1f | %s | %.3f (%.0f%%) | %.1f (%.4f) | %.0f | %.0f | %s |" % (
            nh, T, j["n_gpus"], j["ms_per_step"], j["value"] / 1e6, j["e2e"]["value"] / 1e6, j["config"]["lstm_kernel"], rec_ms,
            100.0 * rec_ms / max(j["ms_per_step"], 1e-9), tf, tf / k["lstm_fwd"]["peak"] if "lstm_fwd" in k else 0.0,
            k.get("ctc_align", {}).get("achieved", 0.0), k.get("sgd_update", {}).get("achieved", 0.0),
            (j.get("clocks") or {}).get("sm_mhz")))


if __name__ == "__main__":
    main()
