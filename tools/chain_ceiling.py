"""Compile and run the ceiling probe of the cfg2 chain (tools/chain_ceiling.cu) and print its JSON
line with the card's name, power limit and SM clocks (read-only nvidia-smi queries) beside it.

    python tools/chain_ceiling.py [--edge 16384] [--blocks-per-sm N] [--launches 1000]
                                  [--skeleton single|pinned|pipelined] [--work W] [--k K] [--sweep]

``--blocks-per-sm N`` caps the grid at N blocks per SM that stride over the chunks; the default (0)
launches one block per K chunks.  ``--work W`` adds W dependent multiply-adds per pixel that leave the
output unchanged.  ``--sweep`` runs every skeleton at W in {0, 8, 16, 24}, the pipelined one at
K in {1, 2, 4, 8}, and prints one line per run."""
import argparse
import json
import os
import subprocess
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
SKELETONS = ("single", "pinned", "pipelined")   # the order of enum Skeleton in chain_ceiling.cu
NVCC = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")


def card():
    fields = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        line = subprocess.run(["nvidia-smi", "--query-gpu=" + fields, "--format=csv,noheader", "-i", "0"],
                              check=True, capture_output=True, text=True).stdout.strip()
    except (OSError, subprocess.CalledProcessError) as e:
        return {"nvidia_smi": "unavailable: {}".format(e)}
    return dict(zip(fields.split(","), (x.strip() for x in line.split(","))))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--edge", type=int, default=16384)
    ap.add_argument("--blocks-per-sm", type=int, default=0)
    ap.add_argument("--launches", type=int, default=1000)
    ap.add_argument("--skeleton", choices=SKELETONS, default="single")
    ap.add_argument("--work", type=int, choices=(0, 8, 16, 24), default=0)
    ap.add_argument("--k", type=int, default=1)
    ap.add_argument("--sweep", action="store_true")
    args = ap.parse_args()
    if args.sweep:
        runs = [(s, w, k) for w in (0, 8, 16, 24) for s in SKELETONS
                for k in ((1, 2, 4, 8) if s == "pipelined" else (1,))]
    else:
        runs = [(args.skeleton, args.work, args.k)]
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "chain_ceiling")
        subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-o", exe,
                        os.path.join(HERE, "chain_ceiling.cu")], check=True)
        for skeleton, work, k in runs:
            out = subprocess.run([exe, str(args.edge), str(args.blocks_per_sm), str(args.launches),
                                  str(SKELETONS.index(skeleton)), str(work), str(k)],
                                 check=True, capture_output=True, text=True).stdout
            result = json.loads(out.strip().splitlines()[-1])
            result["card"] = card()
            print(json.dumps(result), flush=True)


if __name__ == "__main__":
    main()
