"""Time random playouts (StrategoEngine.playout, sx_playout) on one GPU against the leanest chain of fused steps that
computes the same games.

    python tools/bench_playout.py [--rounds 3] [--out FILE]

(profiles/r7c_playout.txt is this tool's output.)  Workloads:
- 262 144 Barrage games and 131 072 Standard games, de-phased (game b first plays its own number of random moves in
  [1, 120)), played to the end;
- the shape of examples/pimc_one_ply.py: the children of 256 de-phased Barrage games x 16 determinized worlds, played
  for at most 200 plies;
- 262 144 Micro games de-phased over [1, 12), played to the end (reported; a Micro warp works on a 12-cell board).

The chain is what a user writes without the new call, in its leanest form: step_all with sample_next and only
next_action and the six scalars as outputs (no mask, no observation), each step's next_action feeding the next step
(two action buffers, no copies), exactly as many launches as the longest game needs and no host synchronisation in
between: the most favourable case for the chain.  Both arms start from the same state (restored by a device copy
outside the timed window) and the same first action (the draw of a rejected step_all, which leaves the state as it
is).  Before timing, the outputs are checked identical: every game's rows, plies and scalars from the chain (kept from
the step that reported done) against the playout.  Then the arms alternate for `--rounds` rounds, each timed with CUDA
events around the whole call; the median is reported with every round, and plies per second = the plies of all games
over that time.  The card name and power limit are printed first, and the distribution of the game lengths per
workload."""
import argparse
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from stratego_env_b200.config import VERSION_CONFIGS, as_version  # noqa: E402
from stratego_env_b200.engine import StrategoEngine  # noqa: E402

SEED = 17
SCALARS = ("reward", "done", "winner", "ending_invalid", "illegal", "player")
STATE = ("board", "aux", "captured")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def dephased(e, B, steps, seed=1):
    """B games, game b played for its own number of random moves in [1, steps) (at least one, so that every game's
    state is one a step wrote)"""
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


def first_action(e, st):
    """the SX_SAMPLE_NEXT draw on each game's current state: a step_all of a rejected action (-1) does not change the
    game and draws from it"""
    B = st.num_envs
    out = e.alloc_outputs(B, partial=False, full=False, mask=False, sample=True)
    e.step_all(st.clone(), torch.full((B,), -1, dtype=torch.int32, device="cuda"), out, sample_next=True, seed=SEED)
    return out["next_action"].clone()


def chain(e, st, a, launches, outs):
    """the leanest chain: `launches` fused steps, each step's next_action the next step's action"""
    for i in range(launches):
        out = outs[i & 1]
        e.step_all(st, a, out, sample_next=True, seed=SEED)
        a = out["next_action"]


def check_identical(e, st0, a0, cap):
    """the chain with each game's rows kept from the step that reported done, against the playout; returns the plies"""
    B = st0.num_envs
    got = st0.clone()
    res = e.playout(got, max_plies=cap, seed=SEED)
    launches = int(res.plies.max().item())
    cur, final = st0.clone(), st0.clone()
    fin = (st0.aux[:, 2] & 1) == 1
    plies = torch.zeros(B, dtype=torch.int32, device="cuda")
    sc = e.alloc_outputs(B, partial=False, full=False, mask=False)
    out = e.alloc_outputs(B, partial=False, full=False, mask=False, sample=True)
    a = a0.clone()
    for _ in range(launches):
        e.step_all(cur, a, out, sample_next=True, seed=SEED)
        live = ~fin
        for name in STATE:
            setattr(final, name, torch.where(live[:, None], getattr(cur, name), getattr(final, name)))
        for name in SCALARS:
            sc[name] = torch.where(live, out[name], sc[name])
        plies += live.to(torch.int32)
        fin |= out["done"] == 1
        a = out["next_action"].clone()
    live = (st0.aux[:, 2] & 1) == 0
    same = all(torch.equal(getattr(got, n), getattr(final, n)) for n in STATE)
    same &= torch.equal(res.plies, plies)
    same &= all(torch.equal(getattr(res, n)[live], sc[n][live]) for n in SCALARS)
    if not same:
        raise SystemExit("playout and the chain differ")
    return res.plies, launches


def e2e(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e-3


def workloads():
    for name, B, steps in (("barrage", 262144, 120), ("standard", 131072, 120)):
        e = StrategoEngine(VERSION_CONFIGS[as_version(name)], device="cuda:0")
        yield "%s %d" % (name, B), e, dephased(e, B, steps), None
    e = StrategoEngine(VERSION_CONFIGS[as_version("barrage")], device="cuda:0")
    worlds = e.sample_hidden_states(dephased(e, 256, 60, seed=2), n_samples=16, seed=3)
    yield "pimc children", e, e.expand_moves(worlds).states, 200
    e = StrategoEngine(VERSION_CONFIGS[as_version("micro")], device="cuda:0")
    yield "micro 262144", e, dephased(e, 262144, 12), None


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
    say("%-14s %7s %6s %7s %9s %11s %11s %9s %9s %7s" % (
        "workload", "games", "cap", "steps", "plies", "playout ms", "chain ms", "Mply/s", "chain", "speedup"))
    for label, e, st0, cap in workloads():
        B = st0.num_envs
        a0 = first_action(e, st0)
        plies, launches = check_identical(e, st0, a0, cap)
        total = int(plies.sum().item())
        st = st0.clone()
        outs = [e.alloc_outputs(B, partial=False, full=False, mask=False, sample=True) for _ in range(2)]
        for name in STATE:  # warm-up of both arms
            getattr(st, name).copy_(getattr(st0, name))
        e.playout(st, max_plies=cap, seed=SEED)
        chain(e, st, a0, 2, outs)
        t_play, t_chain = [], []
        for _ in range(args.rounds):
            for name in STATE:
                getattr(st, name).copy_(getattr(st0, name))
            t_play.append(e2e(lambda: e.playout(st, max_plies=cap, seed=SEED)))
            for name in STATE:
                getattr(st, name).copy_(getattr(st0, name))
            t_chain.append(e2e(lambda: chain(e, st, a0, launches, outs)))
        tp, tc = statistics.median(t_play), statistics.median(t_chain)
        say("%-14s %7d %6s %7d %9d %11.2f %11.2f %9.1f %9.1f %6.2fx" % (
            label, B, "-" if cap is None else cap, launches, total, tp * 1e3, tc * 1e3, total / tp / 1e6,
            total / tc / 1e6, tc / tp))
        q = torch.quantile(plies.float(), torch.tensor([0.5, 0.9, 0.99, 1.0], device="cuda")).tolist()
        say("               plies per game: mean %.1f, median %.0f, p90 %.0f, p99 %.0f, max %.0f" % (
            total / B, *q))
        say("               rounds ms: playout %s | chain %s" % (
            " ".join("%.2f" % (x * 1e3) for x in t_play), " ".join("%.2f" % (x * 1e3) for x in t_chain)))
        del e, st0, st, outs
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
