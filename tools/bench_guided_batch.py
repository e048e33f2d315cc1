"""Time guided tree search with several leaves per tree and round (StrategoEngine.guided_select(leaves_per_tree=L) /
guided_backup) on one GPU.

    python tools/bench_guided_batch.py [--passes 3] [--baseline DIR] [--out FILE]

1. One leaf per round against another build (--baseline DIR: a checkout of another commit with its library built):
   tools/bench_guided_search.py of DIR and of this tree, run alternately in their own processes, --passes times each;
   every pass's select and backup times per workload are printed.
2. The same simulations with more leaves per round: 128 simulations per tree on Barrage with 16, 256 and 4 096
   de-phased trees, L in {1, 4, 8, 16, 32}.  L = 1 is 128 rounds of one leaf; L > 1 is one round of one leaf (in an
   empty tree every leaf of the first round is the root) and then ceil(127 / L) rounds of L, 1 + L * ceil(127 / L)
   simulations.  Per search:
   - engine ms: guided_select, observe (partial observation, float32) and guided_backup of every round, with one fixed
     logits tensor (float32, random multiples of 1/8) and values tensor per L, so the tree grows as it would under a
     network without the network's cost;
   - end-to-end ms: the same rounds with the conv evaluator of examples/guided_mcts.py (observe inside) in place of
     the fixed tensors;
   - rounds, the simulations run, the duplicate-leaf fraction (leaves of a round that another leaf of the same tree
     and round already reached, over the end-to-end search) and used mean / max at the end.
   Each search is timed with one pair of CUDA events around it, on a fresh tree.  The (trees, L) cases alternate for
   --passes passes and the median pass is reported with every pass.
The card name and power limit are printed first."""
import argparse
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "examples"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_guided_search import card, dephased  # noqa: E402
from guided_mcts import ConvEvaluator, schedule  # noqa: E402
from stratego_env_b200.config import BARRAGE_STRATEGO_CONFIG  # noqa: E402
from stratego_env_b200.engine import StrategoEngine  # noqa: E402

SIMULATIONS = 128
TREES = (16, 256, 4096)
LEAVES = (1, 4, 8, 16, 32)


def against_baseline(baseline, passes, say):
    """part 1: bench_guided_search.py of the baseline checkout and of this tree, alternated"""
    runs = {"baseline": [], "this tree": []}
    for p in range(passes):
        for label, root in (("baseline", baseline), ("this tree", ROOT)):
            q = subprocess.run([sys.executable, os.path.join(root, "tools", "bench_guided_search.py"), "--rounds", "1"],
                               cwd=root, capture_output=True, text=True, check=True)
            rows = [ln for ln in q.stdout.splitlines() if ln.split()[:1] in (["barrage"], ["standard"])]
            runs[label].append(rows)
            for ln in rows:
                say("pass %d %-9s %s" % (p + 1, label, ln))
    return runs


def search(e, roots, L, nodes, evaluate):
    """one search of fresh trees: (ms, rounds, simulations, duplicate leaves, leaves, tree)"""
    B = roots.num_envs
    tree = e.guided_tree(roots, nodes)
    plan = schedule(SIMULATIONS, L)
    dup = torch.zeros((), dtype=torch.long, device=e.device)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for Lr in plan:
        leaves = e.guided_select(roots, tree, leaves_per_tree=Lr)
        logits, values = evaluate(leaves)
        e.guided_backup(tree, leaves, logits, values)
        if Lr > 1:
            s = leaves.node.view(B, Lr).sort(1).values
            dup += (s[:, 1:] == s[:, :-1]).sum()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), len(plan), sum(plan), int(dup), B * sum(plan), tree


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--passes", type=int, default=3)
    ap.add_argument("--baseline", default=None, help="checkout of another commit, its library built: part 1")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    say("card: %s" % card())
    if args.baseline:
        say("1. one leaf per round: tools/bench_guided_search.py --rounds 1 of the baseline (%s) and of this tree, "
            "alternated, %d passes" % (args.baseline, args.passes))
        against_baseline(os.path.abspath(args.baseline), args.passes, say)
    e = StrategoEngine(BARRAGE_STRATEGO_CONFIG, device="cuda:0")
    conv = ConvEvaluator(e)
    nodes = 1 + 48 * (1 + max(LEAVES) * -(-(SIMULATIONS - 1) // max(LEAVES)))
    say("2. %d simulations per tree on Barrage, pool %d nodes; engine = select + observe + backup with fixed logits; "
        "end-to-end = select + conv evaluator + backup; median of %d alternated passes" % (SIMULATIONS, nodes,
                                                                                           args.passes))
    cases = []
    for B in TREES:
        roots = dephased(e, B, 120)
        for L in LEAVES:
            g = torch.Generator(device="cuda").manual_seed(5)
            fixed = {}
            for Lr in set(schedule(SIMULATIONS, L)):
                fixed[Lr] = ((torch.randint(-4, 5, (B * Lr,) + tuple(e.spatial_action_size), generator=g,
                                            device="cuda") / 8).float(),
                             (torch.randint(-16, 17, (B * Lr,), generator=g, device="cuda") / 16).float(),
                             e.alloc_outputs(B * Lr, partial=True, full=False, mask=False))

            def engine_only(leaves, fixed=fixed):
                logits, values, out = fixed[leaves.per_tree]
                e.observe(leaves.states, out=out, partial=True, full=False, mask=False)
                return logits, values
            cases.append(dict(B=B, L=L, roots=roots, engine_only=engine_only, eng=[], e2e=[]))
    for c in cases:  # warm-up: every shape, the conv evaluator's algorithms
        search(e, c["roots"], c["L"], nodes, c["engine_only"])
        search(e, c["roots"], c["L"], nodes, conv)
    for _ in range(args.passes):
        for c in cases:
            c["eng"].append(search(e, c["roots"], c["L"], nodes, c["engine_only"])[0])
            ms, rounds, sims, dup, total, tree = search(e, c["roots"], c["L"], nodes, conv)
            c["e2e"].append(ms)
            used = tree.used.double()
            c.update(rounds=rounds, sims=sims, dup=dup / total, used=(float(used.mean()), int(used.max())))
    say("%6s %3s %7s %5s %11s %11s %9s %14s %10s %15s" % (
        "trees", "L", "rounds", "sims", "engine ms", "e2e ms", "e2e x L=1", "sims/s e2e", "dup leaves",
        "used mean/max"))
    base = {}
    for c in cases:
        eng, e2e = statistics.median(c["eng"]), statistics.median(c["e2e"])
        base.setdefault(c["B"], e2e)
        say("%6d %3d %7d %5d %11.2f %11.2f %9.2f %14.3g %10.3f %9.0f/%d" % (
            c["B"], c["L"], c["rounds"], c["sims"], eng, e2e, base[c["B"]] / e2e, c["B"] * c["sims"] / (e2e * 1e-3),
            c["dup"], c["used"][0], c["used"][1]))
        say("           passes ms: engine %s | end-to-end %s" % (" ".join("%.2f" % x for x in c["eng"]),
                                                                 " ".join("%.2f" % x for x in c["e2e"])))
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
