"""Determinized guided search on Barrage: PUCT select and backup on the device, the leaves evaluated by the caller.

At each of its turns the searcher, for every game in the batch at once:
1. draws K complete worlds that agree with what it knows (sample_hidden_states, viewer = the player to move);
2. grows one guided tree per world for --simulations simulations, every tree of every game in each launch:
   guided_select (one leaf per tree) -> the evaluator on the leaves -> guided_backup (priors from the evaluator's
   logits, its value backed up).  With --leaves-per-tree L > 1 a round selects L leaves per tree under a virtual loss:
   one round of one leaf (in an empty tree every leaf would be the root), then ceil((simulations - 1) / L) rounds of
   L, so the evaluator sees L times the rows in far fewer rounds;
3. sums the root children's visit counts (root_stats) over the K worlds and plays the most visited move, ties to the
   lowest flat index.
No step of a round synchronises the host.  Evaluators:
- rollout: uniform logits and, as the value, one random playout (at most --rollout-plies plies) of a copy of the
  leaves.  It needs no trained network, so its results against the random player and against
  examples/determinized_mcts.py mean something;
- conv: the untrained conv trunk of examples/rollout_conv_policy.py with a policy head (logits [B, R, C, A]) and a
  value head (mean pool, linear, tanh) on observe(leaves).  Its play is that of an untrained network: it is here to
  time a network in the loop.
The searcher is player +1 and moves first; the setup is that of examples/determinized_mcts.py (same games, seed and
random opponent).  --opponent mcts plays player -1 with determinized_mcts's searcher (--mcts-iterations iterations,
the same worlds and playout cap).

    python examples/guided_mcts.py [--games 256] [--worlds 16] [--simulations 128] [--rollout-plies 100]
                                   [--evaluator rollout|conv] [--opponent random|mcts] [--leaves-per-tree 1]

With the defaults (rollout evaluator) the searcher won 250 and lost 6 of 256 games against the random player, in
7.7 s, and won 139 and lost 117 of 256 against determinized MCTS, in 8.9 s, on a B200 at 1 000 W
(profiles/r7f_examples.txt).  With --leaves-per-tree 8 (129 simulations in 17 rounds) it won 137 and lost 119 against
determinized MCTS with the search taking 2.2 s instead of 5.3 s, same card (profiles/r7h_examples.txt).
"""
import argparse
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from stratego_env_b200.config import BARRAGE_STRATEGO_CONFIG  # noqa: E402
from stratego_env_b200.engine import DeviceState, StrategoEngine  # noqa: E402


def to_move_sign(state):
    """+1 / -1 (float32): the player to move of every game (aux_pack: bit 4 of word 2)"""
    return torch.where(((state.aux[:, 2] >> 4) & 1) == 0, 1.0, -1.0)


class RolloutEvaluator:
    """uniform logits; the value of a leaf is one random playout of a copy of it, from its player to move's side"""

    def __init__(self, e, plies, seed):
        self.e, self.plies, self.seed, self.calls = e, plies, seed, 0
        self.logits = {}  # rows -> zeros

    def __call__(self, leaves):
        B = leaves.node.shape[0]
        if B not in self.logits:
            self.logits[B] = torch.zeros((B,) + tuple(self.e.spatial_action_size), dtype=torch.float32,
                                         device=self.e.device)
        copy = leaves.states.clone()
        self.calls += 1
        res = self.e.playout(copy, max_plies=self.plies, seed=self.seed, env_base=self.calls * B)
        return self.logits[B], res.reward * to_move_sign(leaves.states)


class ConvEvaluator:
    """the conv trunk of examples/rollout_conv_policy.py (untrained) with a policy and a value head"""

    def __init__(self, e, channels=64, dtype=torch.bfloat16):
        R, C, A = e.spatial_action_size
        torch.manual_seed(0)
        self.e, self.dtype = e, dtype
        self.trunk = torch.nn.Sequential(
            torch.nn.Conv2d(e.po_channels, channels, 3, padding=1), torch.nn.ReLU(),
            torch.nn.Conv2d(channels, channels, 3, padding=1), torch.nn.ReLU()).to(e.device, dtype)
        self.policy = torch.nn.Conv2d(channels, A, 3, padding=1).to(e.device, dtype)
        self.value = torch.nn.Linear(channels, 1).to(e.device, dtype)
        for m in (self.trunk, self.policy):
            m.to(memory_format=torch.channels_last)
        self.out = {}  # rows -> observation buffers

    @torch.no_grad()
    def __call__(self, leaves):
        B = leaves.node.shape[0]
        if B not in self.out:
            self.out[B] = self.e.alloc_outputs(B, partial=True, full=False, mask=False)
        obs = self.e.observe(leaves.states, out=self.out[B], partial=True, full=False, mask=False)["partial_obs"]
        h = self.trunk(obs.permute(0, 3, 1, 2).to(self.dtype))
        logits = self.policy(h).permute(0, 2, 3, 1).contiguous()
        values = torch.tanh(self.value(h.mean((2, 3)))).float().view(B)
        return logits, values


def schedule(simulations, leaves_per_tree):
    """leaves per tree of each round: `simulations` rounds of one leaf, or with L > 1 one round of one leaf and then
    ceil((simulations - 1) / L) rounds of L"""
    L = leaves_per_tree
    return [1] * simulations if L == 1 else [1] + [L] * -(-(simulations - 1) // L)


def search(e, st, games, K, simulations, evaluator, seed, draw, c_puct=1.25, leaves_per_tree=1):
    """the searcher's move (flat spatial index, its own frame) in each game of `games` (all with the searcher to move)"""
    n = games.numel()
    sub = DeviceState(st.board[games], st.aux[games], st.captured[games])
    worlds = e.sample_hidden_states(sub, n_samples=K, seed=seed, draw=draw)  # row g * K + k: world k of game g
    plan = schedule(simulations, leaves_per_tree)
    tree = e.guided_tree(worlds, 1 + 48 * sum(plan))
    for L in plan:
        leaves = e.guided_select(worlds, tree, c_puct=c_puct, leaves_per_tree=L)
        logits, values = evaluator(leaves)
        e.guided_backup(tree, leaves, logits, values)
    visits, _ = tree.root_stats()
    total = visits.view(n, K, -1).sum(1)
    return torch.argmax(total, dim=1).to(torch.int32)  # the first of equal maxima: the lowest index


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=256)
    ap.add_argument("--worlds", type=int, default=16)
    ap.add_argument("--simulations", type=int, default=128)
    ap.add_argument("--rollout-plies", type=int, default=100)
    ap.add_argument("--evaluator", choices=("rollout", "conv"), default="rollout")
    ap.add_argument("--opponent", choices=("random", "mcts"), default="random")
    ap.add_argument("--mcts-iterations", type=int, default=128)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--leaves-per-tree", type=int, default=1)
    args = ap.parse_args()
    G, K = args.games, args.worlds
    if args.opponent == "mcts":
        from determinized_mcts import search as mcts_search

    e = StrategoEngine(BARRAGE_STRATEGO_CONFIG, device="cuda:0")
    evaluator = (RolloutEvaluator(e, args.rollout_plies, args.seed) if args.evaluator == "rollout"
                 else ConvEvaluator(e))
    st = e.alloc_state(G)
    e.reset(st, seed=args.seed, shuffle=True)
    out = e.alloc_outputs(G, partial=False, full=False, mask=True, sample=True)
    e.observe(st, out=out, partial=False, full=False, mask=True)
    random_actions = e.sample_valid(out["valid_mask"], seed=args.seed)
    to_move = out["player"].clone()
    winner = torch.zeros(G, dtype=torch.int8, device=e.device)
    finished = torch.zeros(G, dtype=torch.bool, device=e.device)
    torch.cuda.synchronize()
    t0 = time.time()
    decisions, simulations, t_search = 0, 0, 0.0
    for ply in range(int(BARRAGE_STRATEGO_CONFIG["max_turns"]) + 1):
        games = torch.nonzero((to_move == 1) & ~finished).flatten()
        actions = random_actions.clone()
        if games.numel():
            torch.cuda.synchronize()
            ts = time.time()
            actions[games] = search(e, st, games, K, args.simulations, evaluator, args.seed, ply,
                                    leaves_per_tree=args.leaves_per_tree)
            torch.cuda.synchronize()
            t_search += time.time() - ts
            decisions += games.numel()
            simulations += games.numel() * K * sum(schedule(args.simulations, args.leaves_per_tree))
        if args.opponent == "mcts":
            other = torch.nonzero((to_move == -1) & ~finished).flatten()
            if other.numel():
                actions[other] = mcts_search(e, st, other, K, args.mcts_iterations, args.rollout_plies,
                                             args.seed + 1, ply)
        e.step_all(st, actions, out, auto_reset=False, sample_next=True, seed=args.seed)
        ended = (out["done"] == 1) & ~finished
        winner = torch.where(ended, out["winner"], winner)
        finished |= ended
        if bool(finished.all()):
            break
        random_actions = out["next_action"].clone()
        to_move = out["player"].clone()
    elapsed = time.time() - t0
    wins, losses = int((winner == 1).sum()), int((winner == -1).sum())
    opponent = ("uniform random" if args.opponent == "random" else
                "determinized MCTS (%d worlds, %d iterations, %d-ply playouts)" % (K, args.mcts_iterations,
                                                                                   args.rollout_plies))
    plan = schedule(args.simulations, args.leaves_per_tree)
    per_tree = ("%d simulations" % args.simulations if args.leaves_per_tree == 1 else
                "%d simulations in %d rounds of up to %d leaves per tree" % (sum(plan), len(plan), args.leaves_per_tree))
    print("guided search, %s evaluator (%d worlds, %s%s) vs %s, %d Barrage games, %d plies, %.1f s" % (
        args.evaluator, K, per_tree, ", %d-ply playouts" % args.rollout_plies if args.evaluator == "rollout"
        else "", opponent, G, ply + 1, elapsed))
    print("searcher wins %d, losses %d, unfinished or turn limit %d; %d searcher decisions" % (
        wins, losses, G - wins - losses, decisions))
    print("searcher: %d simulations in %.2f s, %.3g simulations/s (select + evaluator + backup, every tree of a "
          "decision in each launch)" % (simulations, t_search, simulations / t_search if t_search else 0.0))


if __name__ == "__main__":
    main()
