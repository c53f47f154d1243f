"""Compile and run the ceiling probe of the cfg2 chain (tools/chain_ceiling.cu) and print its JSON
line with the card's name, power limit and SM clocks (read-only nvidia-smi queries) beside it.

    python tools/chain_ceiling.py [--edge 16384] [--blocks-per-sm N] [--launches 1000]

``--blocks-per-sm N`` caps the grid at N blocks per SM that stride over the chunks; the default (0)
launches one block per chunk, as the specialised kernel does for programs without shared-memory
tables."""
import argparse
import json
import os
import subprocess
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
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
    args = ap.parse_args()
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "chain_ceiling")
        subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-o", exe,
                        os.path.join(HERE, "chain_ceiling.cu")], check=True)
        out = subprocess.run([exe, str(args.edge), str(args.blocks_per_sm), str(args.launches)],
                             check=True, capture_output=True, text=True).stdout
    result = json.loads(out.strip().splitlines()[-1])
    result["card"] = card()
    print(json.dumps(result))


if __name__ == "__main__":
    main()
