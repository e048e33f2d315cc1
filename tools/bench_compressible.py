"""Plain against compressible output planes, in one process on one GPU (StrategoEngine(compressible_outputs=)).

    python tools/bench_compressible.py [--out FILE] [--rounds 6] [--steps 50] [--workloads barrage,...]

Each workload is de-phased once as bench.py does it (render-free steps from a seeded reset); two engines, one with
``torch.empty`` planes (compressible_outputs=False) and one with the planes in one compressible allocation of the library,
step copies of that state, alternating round by round, CUDA events around each round of launches.  The outputs stay
byte-identical (tests/test_compressible_outputs_gpu.py); only where the bytes go changes.  `GB/s` is algorithmic bytes
(bench.py's count at the element size) over time: with compressed planes it can exceed what HBM can carry, because
fewer bytes reach DRAM, so it is no longer a bandwidth.  Prints the card name, power limit, clocks and the compression
type granted first."""
import argparse
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bench import WORKLOADS  # noqa: E402
from stratego_env_b200.config import VERSION_CONFIGS, as_version  # noqa: E402
from stratego_env_b200.engine import DeviceAllocation, StrategoEngine, load_setup_table  # noqa: E402

CASES = [("barrage", torch.float32), ("barrage", torch.bfloat16), ("standard", torch.float32),
         ("standard_both", torch.float32), ("micro", torch.float32)]
LOG = []


def say(line=""):
    print(line, flush=True)
    LOG.append(line)


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm,clocks.mem",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def bytes_per_step(lay, full, eb):
    """bench.py's algorithmic bytes (SURVEY.md 8(d)) with `eb` bytes per observation element"""
    obs = lay.cells * 67 * eb + (lay.cells * 79 * eb if full else 0)
    state = lay.cells + 4 * lay.pieces_per_side + 16
    return obs + lay.cells * lay.spatial_channels + 2 * state + 13


def measure(name, dtype, rounds, steps):
    w = WORKLOADS[name]
    B, full = w["envs"], w["full"]
    cfg = VERSION_CONFIGS[as_version(w["version"])]
    table = load_setup_table(w["table"]) if w["table"] else None
    engines = {k: StrategoEngine(cfg, device="cuda:0", p2_rot180=table is None, obs_dtype=dtype, compressible_outputs=v)
               for k, v in (("plain", False), ("compressible", True))}
    eng0 = engines["plain"]
    setups = eng0.upload_setups(table) if table is not None else None
    kw = dict(auto_reset=True, sample_next=True, setups=setups, shuffle=setups is None, seed=1)
    st0 = eng0.alloc_state(B)
    eng0.reset(st0, seed=1, setups=setups, shuffle=setups is None)
    lean = eng0.alloc_outputs(B, partial=False, full=False, mask=False, sample=True)
    acts0 = eng0.sample_valid(eng0.valid_mask(st0), seed=1)
    for _ in range(w["dephase"]):
        eng0.step_all(st0, acts0, lean, **kw)
        acts0, lean["next_action"] = lean["next_action"], acts0
    del lean
    runs = {}
    for k, eng in engines.items():
        st, acts = st0.clone(), acts0.clone()
        out = eng.alloc_outputs(B, partial=True, full=full, mask=True, sample=True)
        assert eng.outputs_compressed == (k == "compressible")

        def run(n, eng=eng, st=st, out=out, box=[acts]):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n):
                eng.step_all(st, box[0], out, **kw)
                box[0], out["next_action"] = out["next_action"], box[0]
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / n
        runs[k] = run
    times = {k: [] for k in runs}
    for k in runs:
        runs[k](5)
    for _ in range(rounds):
        for k in runs:
            runs[k](2)
            times[k].append(runs[k](steps))
    nb = bytes_per_step(eng0.layout, full, 4 if dtype == torch.float32 else 2)
    info = eng0.launch_info(partial=True, full=full, mask=True)
    res = {}
    for k, v in times.items():
        med = statistics.median(v)
        res[k] = med
        say("%-14s %-5s %-12s B=%-8d median %7.4f ms  %8.1f M env-steps/s  %6.0f GB/s algorithmic  spread %.2f %%  "
            "%s  (rounds %s)" % (name, str(dtype)[6:], k, B, med, B / med / 1e3, B * nb / med / 1e6,
                                 100 * (max(v) - min(v)) / med, "toy" if info["thread_per_game"] else
                                 "warp x%d" % info["warps_per_block"], " ".join("%.4f" % t for t in v)))
    say("%-14s %-5s compressible / plain throughput: %.3f" % (name, str(dtype)[6:], res["plain"] / res["compressible"]))
    engines.clear()
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the report to this file")
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--steps", type=int, default=50, help="launches per round")
    ap.add_argument("--workloads", default=None, help="comma list of name[:bf16] (default: the five cases)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_compressible.py measures on a GPU; none found")
    cases = CASES
    if args.workloads:
        cases = [(c.split(":")[0], torch.bfloat16 if c.endswith(":bf16") else torch.float32)
                 for c in args.workloads.split(",")]
    say("card: %s" % card())
    probe = DeviceAllocation("cuda:0", 2 << 20, compressible=True)
    say("compressible memory granted: %s (CU_MEM_ALLOCATION_COMP_GENERIC through sx_device_alloc)"
        % ("GENERIC" if probe.compressed else "no: plain memory"))
    if not probe.compressed:
        sys.exit("no compressible memory on this device: nothing to compare")
    del probe
    say("== fused step, plain vs compressible planes (alternating, %d rounds x %d launches, median ms per launch)"
        % (args.rounds, args.steps))
    for name, dtype in cases:
        measure(name, dtype, args.rounds, args.steps)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(LOG) + "\n")


if __name__ == "__main__":
    main()
