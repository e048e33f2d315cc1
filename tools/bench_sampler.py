"""Time sx_sample_policy of two or more library builds, alternating, in one process on one GPU.

    python tools/bench_sampler.py --lib A.so --lib B.so [--games 131072] [--launches 300] [--rounds 6] [--out FILE]

The workload is the sampler leg of the Standard conv-policy rollout: 131 072 Standard games (human setups) played
40 uniformly sampled moves in, bf16 logits [games, 10 * 10 * 36], temperature 1, log-probability on.  Each build loads
through SX_LIB into an engine of its own; all engines read the same state and logits.  Per round every build gets 20
warm-up launches and then `--launches` launches between two CUDA events, in alternating order.  The logits (0.94 GB)
and the state exceed the 126 MB L2, so every launch reads them from HBM.  Prints the card name and power limit first,
one line per round and build, the median / min / max per build and the share of games whose action differs from the
first build's."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from stratego_env_b200 import _lib  # noqa: E402
from stratego_env_b200.config import STANDARD_STRATEGO_CONFIG  # noqa: E402
from stratego_env_b200.engine import StrategoEngine, load_setup_table  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def engine_for(lib_path):
    os.environ["SX_LIB"] = os.path.abspath(lib_path)
    _lib._lib = None  # the next engine loads (and keeps) this build
    return StrategoEngine(STANDARD_STRATEGO_CONFIG, device="cuda:0", p2_rot180=False)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", required=True, help="library build to time (repeat for each)")
    ap.add_argument("--games", type=int, default=131072)
    ap.add_argument("--launches", type=int, default=300)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    say("card: %s" % card())
    engines = [engine_for(p) for p in args.lib]
    e0, B = engines[0], args.games
    st = e0.alloc_state(B)
    e0.reset(st, seed=1, setups=e0.upload_setups(load_setup_table("standard")))
    out = e0.alloc_outputs(B, partial=False, full=False, mask=False, sample=True)
    actions = e0.sample_valid(e0.valid_mask(st), seed=1)
    for _ in range(40):
        e0.step_all(st, actions, out, sample_next=True, seed=1)
        actions = out["next_action"].clone()
    g = torch.Generator(device="cuda").manual_seed(0)
    logits = torch.randn(B, e0.layout.spatial_actions, generator=g, device="cuda").to(torch.bfloat16)

    first = engines[0].sample_policy(st, logits, seed=3, step=0)
    for path, e in zip(args.lib, engines):
        a = e.sample_policy(st, logits, seed=3, step=0)
        say("%s: actions differing from %s: %d of %d" % (path, args.lib[0], int((a != first).sum()), B))

    times = {p: [] for p in args.lib}
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for r in range(args.rounds):
        order = list(zip(args.lib, engines))
        if r % 2:
            order.reverse()
        for path, e in order:
            for i in range(20):
                e.sample_policy(st, logits, seed=3, step=i, return_logprob=True)
            start.record()
            for i in range(args.launches):
                e.sample_policy(st, logits, seed=3, step=i, return_logprob=True)
            end.record()
            end.synchronize()
            ms = start.elapsed_time(end) / args.launches
            times[path].append(ms)
            say(json.dumps({"round": r, "lib": path, "ms_per_launch": round(ms, 5)}))
    for path in args.lib:
        t = times[path]
        say("%s: median %.4f ms, min %.4f, max %.4f per %d games (%d rounds x %d launches)"
            % (path, statistics.median(t), min(t), max(t), B, args.rounds, args.launches))
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
