"""Time the guided tree search (StrategoEngine.guided_select / guided_backup) on one GPU, per round, with the
observation and the conv network of examples/guided_mcts.py on the same leaves for context.

    python tools/bench_guided_search.py [--rounds 3] [--out FILE]

Workloads, 64 simulations (rounds) per tree, pool 1 + 48 x 64 nodes, de-phased roots:
- 4 096 Barrage trees (the shape of examples/guided_mcts.py: 256 games x 16 worlds);
- 65 536 Barrage trees;
- 4 096 Standard trees.
Each round is guided_select, then guided_backup with one fixed, precomputed logits tensor (float32 [B, R, C, A], random
multiples of 1/8) and values tensor, so the tree grows as it would under a network without the network's cost.  Every
select and every backup is timed with its own pair of CUDA events; a workload's figure is the mean per round over the
64 rounds of a fresh tree.  The workloads alternate for `--rounds` passes and the median pass is reported with every
pass.  On the leaves of the last round, for context: observe (partial observation, float32) and the conv forward of
examples/guided_mcts.py's evaluator (bfloat16 trunk, policy and value heads), each the median of 10 timed calls after a
warm-up.  The card name and power limit are printed first."""
import argparse
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "examples"))
from guided_mcts import ConvEvaluator  # noqa: E402
from stratego_env_b200.config import VERSION_CONFIGS, as_version  # noqa: E402
from stratego_env_b200.engine import StrategoEngine  # noqa: E402

ROUNDS = 64
NODES = 1 + 48 * ROUNDS


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


def grow(e, roots, logits, values):
    """a fresh tree grown ROUNDS rounds: (mean select ms, mean backup ms, the tree, the last leaves)"""
    tree = e.guided_tree(roots, NODES)
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(ROUNDS)]
    torch.cuda.synchronize()
    leaves = None
    for r in range(ROUNDS):
        ev[r][0].record()
        leaves = e.guided_select(roots, tree)
        ev[r][1].record()
        e.guided_backup(tree, leaves, logits, values)
        ev[r][2].record()
    torch.cuda.synchronize()
    sel = sum(x[0].elapsed_time(x[1]) for x in ev) / ROUNDS
    back = sum(x[1].elapsed_time(x[2]) for x in ev) / ROUNDS
    return sel, back, tree, leaves


def median_ms(fn, n=10):
    fn()
    torch.cuda.synchronize()
    t = []
    for _ in range(n):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        t.append(a.elapsed_time(b))
    return statistics.median(t)


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
    say("%d rounds per tree, pool %d nodes; per round: guided_select, guided_backup (fixed logits and values); "
        "median of %d alternated passes" % (ROUNDS, NODES, args.rounds))
    engines = {v: StrategoEngine(VERSION_CONFIGS[as_version(v)], device="cuda:0") for v in ("barrage", "standard")}
    work = []
    for label, v, B in (("barrage 4k", "barrage", 4096), ("barrage 64k", "barrage", 65536),
                        ("standard 4k", "standard", 4096)):
        e = engines[v]
        roots = dephased(e, B, 120)
        g = torch.Generator(device="cuda").manual_seed(5)
        logits = (torch.randint(-16, 17, (B,) + tuple(e.spatial_action_size), generator=g, device="cuda") / 8).float()
        values = (torch.randint(-16, 17, (B,), generator=g, device="cuda") / 16).float()
        grow(e, roots, logits, values)  # warm-up
        work.append(dict(label=label, e=e, roots=roots, logits=logits, values=values, sel=[], back=[]))
    for _ in range(args.rounds):
        for w in work:
            sel, back, tree, leaves = grow(w["e"], w["roots"], w["logits"], w["values"])
            w["sel"].append(sel)
            w["back"].append(back)
            w["tree"], w["leaves"] = tree, leaves
    say("%-12s %6s %10s %10s %10s %12s %11s %10s %14s" % (
        "workload", "trees", "select ms", "backup ms", "engine ms", "sims/s", "observe ms", "conv ms",
        "used mean/max"))
    for w in work:
        e, leaves, tree = w["e"], w["leaves"], w["tree"]
        B = leaves.node.shape[0]
        sel, back = statistics.median(w["sel"]), statistics.median(w["back"])
        out = e.alloc_outputs(B, partial=True, full=False, mask=False)
        t_obs = median_ms(lambda: e.observe(leaves.states, out=out, partial=True, full=False, mask=False))
        conv = ConvEvaluator(e)
        t_conv = median_ms(lambda: conv(leaves))
        used = tree.used.double()
        say("%-12s %6d %10.3f %10.3f %10.3f %12.3g %11.3f %10.3f %7.0f/%d" % (
            w["label"], B, sel, back, sel + back + t_obs, B / ((sel + back) * 1e-3), t_obs, t_conv,
            float(used.mean()), int(used.max())))
        say("             passes ms per round: select %s | backup %s; engine = select + observe + backup" % (
            " ".join("%.3f" % x for x in w["sel"]), " ".join("%.3f" % x for x in w["back"])))
        del conv, out
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
