"""Time the device tree search (StrategoEngine.search, sx_search) on one GPU against random playouts
(StrategoEngine.playout, sx_playout) of the same roots with the same ply cap.

    python tools/bench_search.py [--rounds 3] [--out FILE]

(profiles/r7e_search.txt is this tool's output.)  Workloads, 128 iterations per tree:
- the shape of examples/determinized_mcts.py: 256 de-phased Barrage games x 16 determinized worlds (4 096 trees),
  playouts of at most 100 plies;
- 32 768 de-phased Barrage trees, at most 100 plies;
- 4 096 de-phased Standard trees, at most 100 plies;
- 4 096 de-phased Micro trees, playouts to the end.
The baseline plays `iterations` playouts of every root in one `playout` call: a batch of B x iterations copies of the
roots (copied outside the timed window), so both arms run B x iterations playouts from about the same states.  The
search reports no ply count, so its playout plies per second are an estimate: its iterations per second times the
baseline's mean plies per playout (the search's leaves lie a few plies below the roots).  The gap between the two
plies-per-second figures is what the tree costs: descent, expansion and backup, and the shorter parallel work per warp.
The arms alternate for `--rounds` rounds, each timed with CUDA events around the whole call; the median is reported
with every round.  Node use is the mean and max of `used` against the pool (1 + 32 x iterations).  The card name and
power limit are printed first."""
import argparse
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from stratego_env_b200.config import VERSION_CONFIGS, as_version  # noqa: E402
from stratego_env_b200.engine import DeviceState, StrategoEngine  # noqa: E402

SEED = 17
ITERATIONS = 128
STATE = ("board", "aux", "captured")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def dephased(e, B, steps, seed=1):
    """B games, game b played for its own number of random moves in [1, steps)"""
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


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e-3


def workloads():
    e = StrategoEngine(VERSION_CONFIGS[as_version("barrage")], device="cuda:0")
    yield "pimc worlds", e, e.sample_hidden_states(dephased(e, 256, 60, seed=2), n_samples=16, seed=3), 100
    yield "barrage", e, dephased(e, 32768, 120), 100
    e = StrategoEngine(VERSION_CONFIGS[as_version("standard")], device="cuda:0")
    yield "standard", e, dephased(e, 4096, 120), 100
    e = StrategoEngine(VERSION_CONFIGS[as_version("micro")], device="cuda:0")
    yield "micro", e, dephased(e, 4096, 12), None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    say("card: %s" % card())
    say("%d iterations per tree; search plies/s = iterations/s x the baseline's mean plies per playout (estimate)"
        % ITERATIONS)
    say("%-12s %6s %4s %10s %10s %12s %11s %11s %9s %11s" % (
        "workload", "trees", "cap", "search ms", "iter/s", "search ply/s", "playout ms", "play ply/s", "ratio",
        "used mean/max"))
    for label, e, roots, cap in workloads():
        B = roots.num_envs
        copies = DeviceState(*(getattr(roots, n).repeat_interleave(ITERATIONS, 0) for n in STATE))
        work = copies.clone()
        tree = e.search(roots, ITERATIONS, max_plies=cap, seed=SEED)  # warm-up of both arms
        e.playout(work, max_plies=cap, seed=SEED)
        t_search, t_play, plies = [], [], None
        for _ in range(args.rounds):
            t_search.append(timed(lambda: e.search(roots, ITERATIONS, max_plies=cap, seed=SEED)))
            for n in STATE:
                getattr(work, n).copy_(getattr(copies, n))
            res = {}
            t_play.append(timed(lambda: res.setdefault("p", e.playout(work, max_plies=cap, seed=SEED))))
            plies = res["p"].plies
        ts, tp = statistics.median(t_search), statistics.median(t_play)
        n_playouts = B * ITERATIONS
        mean_plies = float(plies.double().mean())
        used = tree.used.double()
        say("%-12s %6d %4s %10.2f %10.3g %12.3g %11.2f %11.3g %8.2fx %6.0f/%d of %d" % (
            label, B, "-" if cap is None else cap, ts * 1e3, n_playouts / ts, n_playouts * mean_plies / ts, tp * 1e3,
            n_playouts * mean_plies / tp, ts / tp, float(used.mean()), int(used.max()), tree.visits.shape[1]))
        say("             baseline plies per playout: mean %.1f, max %d; rounds ms: search %s | playout %s" % (
            mean_plies, int(plies.max()), " ".join("%.2f" % (x * 1e3) for x in t_search),
            " ".join("%.2f" % (x * 1e3) for x in t_play)))
        del tree, copies, work, roots
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
