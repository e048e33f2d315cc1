"""Transpositions and information sets: what a table keyed by position saves a search.

1. Play a batch of Barrage games a few random moves in; the player to move in each game is the searcher.
2. Draw K complete game states per game that agree with what the searcher knows (sample_hidden_states).
3. Expand every world three plies deep with expand_moves, one batched call per ply.
4. At each depth, count the nodes, the distinct positions by state key (what a transposition table stores) and the
   distinct information sets the searcher sees by its information-set key (the nodes of an information-set tree: all
   K worlds of one game share them until a move reveals a difference).

    python examples/transpositions.py [--games 32] [--worlds 8] [--plies 3]
"""
import argparse
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from stratego_env_b200.batched_env import BatchedStrategoEnv  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=32)
    ap.add_argument("--worlds", type=int, default=8)
    ap.add_argument("--plies", type=int, default=3)
    args = ap.parse_args()
    B, K = args.games, args.worlds

    env = BatchedStrategoEnv({"version": "barrage"}, num_envs=B, seed=1, auto_reset=False, sample_actions=True)
    obs = env.reset()
    for _ in range(20):
        obs, _, _, _ = env.step(obs["sampled_action"])
    searcher = obs["player"].to(torch.int8)  # the player to move in each game, +1 / -1

    nodes = env.sample_hidden_states(n_samples=K)  # row b * K + k: world k of game b
    viewer = searcher.repeat_interleave(K)  # the searcher of each node's game
    e = env.engine
    print("%d Barrage games x %d worlds, expanded %d plies deep" % (B, K, args.plies))
    print("%5s %10s %16s %22s" % ("ply", "nodes", "distinct states", "searcher's info sets"))
    for ply in range(args.plies + 1):
        n = nodes.num_envs
        states = torch.unique(e.state_keys(nodes)).numel()
        infosets = torch.unique(e.state_keys(nodes, info_set=True, viewer=viewer)).numel()
        print("%5d %10d %16d %22d" % (ply, n, states, infosets))
        if ply < args.plies:
            ex = e.expand_moves(nodes)
            nodes, viewer = ex.states, viewer[ex.parent]
    print("a transposition table keyed by state key holds %.1f %% of the deepest nodes; an information-set tree, %.2f %%"
          % (100.0 * states / n, 100.0 * infosets / n))


if __name__ == "__main__":
    main()
