"""Time position keys (StrategoEngine.state_keys, sx_state_keys) on one GPU.

    python tools/bench_state_keys.py [--rounds 5] [--iters 50] [--out FILE]

(profiles/r7d_state_keys.txt is this tool's output.)  Workloads: 262 144 Barrage and 131 072 Standard games, de-phased
(game b first plays its own number of random moves in [1, 120)).  Per workload, four arms, each timed with CUDA events
around `--iters` back-to-back calls (after a warm-up), alternating for `--rounds` rounds, median reported:
- state keys (info_set=False);
- information-set keys of the player to move (info_set=True, viewer None);
- clone() of the three state tensors: a floor for reading the compact state (and writing it once more);
- one fused step (step_all with sample_next, auto-reset and the mask and partial observation, as bench.py).
The whole working set (a few tens of MB) sits in the 126 MB L2 after the first pass, so the key and clone times are
L2-resident times.  The kernel's feature count per game is printed too (from the exported states: the non-zero dense
entries of layers 0-1 and 3-33 plus the player), with the Philox blocks a lane computes, ceil(slots / 32) per game, to
read the times against: the kernel issues one Philox4x32-10 block per slot, occupied cells x 3 + 11 + capture entries.
The card name and power limit are printed first."""
import argparse
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from stratego_env_b200.config import VERSION_CONFIGS, as_version  # noqa: E402
from stratego_env_b200.engine import StrategoEngine  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def dephased(e, B, steps, seed=1):
    st = e.alloc_state(B)
    e.reset(st, seed=seed, shuffle=True)
    out = e.alloc_outputs(B, partial=False, full=False, mask=True, sample=True)
    e.observe(st, out=out, partial=False, full=False, mask=True)
    actions = e.sample_valid(out["valid_mask"], seed=seed)
    g = torch.Generator(device="cuda").manual_seed(seed)
    target = torch.randint(1, steps, (B,), generator=g, device="cuda")
    for s in range(steps):
        a = torch.where(target > s, actions, torch.full_like(actions, -1))
        e.step_all(st, a, out, auto_reset=False, sample_next=True, seed=seed, shuffle=True)
        actions = torch.where(target > s, out["next_action"], actions)
    return st


def features(e, st, chunk=16384):
    """(mean dense features per game, mean slots per game, mean Philox blocks per lane per game)"""
    feats = slots = blocks = 0
    for lo in range(0, st.num_envs, chunk):
        part = st.select(lo, min(lo + chunk, st.num_envs))
        dense, _ = e.export_ref_state(part)
        keyed = torch.cat([dense[:, :2], dense[:, 3:]], 1).reshape(part.num_envs, -1)
        feats += int((keyed != 0).sum().item()) + part.num_envs
        occupied = ((part.board[:, :e.cells] & 0x0F) != 0).sum(1)
        ncap = (part.aux[:, 2].long() >> 8) & 0xFF
        s = 3 * occupied + 11 + ncap
        slots += int(s.sum().item())
        blocks += int(((s + 31) // 32).sum().item())
    B = st.num_envs
    return feats / B, slots / B, blocks / B


def timed(fn, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    say("card: %s" % card())
    say("%-10s %7s %9s %7s %9s | %10s %10s %10s %10s | %8s %8s" % (
        "workload", "games", "features", "slots", "philox/l", "state ms", "infoset ms", "clone ms", "step ms",
        "Gkey/s", "GB/s cl"))
    for name, B in (("barrage", 262144), ("standard", 131072)):
        e = StrategoEngine(VERSION_CONFIGS[as_version(name)], device="cuda:0")
        st = dephased(e, B, 120)
        feats, slots, blocks = features(e, st)
        step_state = st.clone()
        outs = [e.alloc_outputs(B, partial=True, full=False, mask=True, sample=True) for _ in range(2)]
        e.step_all(step_state, torch.full((B,), -1, dtype=torch.int32, device="cuda"), outs[1], sample_next=True, seed=3)
        n_steps = [0]

        def step():  # each step plays the previous step's next_action (two buffers), auto-reset as in bench.py
            i = n_steps[0] & 1
            e.step_all(step_state, outs[i ^ 1]["next_action"], outs[i], auto_reset=True, sample_next=True, seed=3,
                       shuffle=True)
            n_steps[0] += 1

        arms = {
            "state": lambda: e.state_keys(st),
            "infoset": lambda: e.state_keys(st, info_set=True),
            "clone": lambda: st.clone(),
            "step": step,
        }
        for fn in arms.values():  # warm-up
            timed(fn, 3)
        times = {k: [] for k in arms}
        for _ in range(args.rounds):
            for k, fn in arms.items():
                times[k].append(timed(fn, args.iters))
        med = {k: statistics.median(v) for k, v in times.items()}
        state_bytes = sum(t.numel() * t.element_size() for t in (st.board, st.aux, st.captured))
        say("%-10s %7d %9.1f %7.1f %9.2f | %10.4f %10.4f %10.4f %10.4f | %8.2f %8.0f" % (
            name, B, feats, slots, blocks, med["state"], med["infoset"], med["clone"], med["step"],
            B / med["state"] / 1e6, 2 * state_bytes / med["clone"] / 1e6))
        say("           rounds ms: " + " | ".join("%s %s" % (k, " ".join("%.4f" % x for x in v)) for k, v in times.items()))
        say("           state bytes %.1f MB (board + aux + capture list)" % (state_bytes / 1e6))
        del e, st, step_state, outs
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
