"""Determinized MCTS on Barrage: a searcher against the uniformly random player, or head to head against one-ply PIMC.

At each of its turns the searcher, for every game in the batch at once:
1. draws K complete worlds that agree with what it knows (sample_hidden_states, viewer = the player to move);
2. runs a Monte Carlo tree search in every world (search: --iterations iterations, PUCT with a uniform prior, leaves
   scored by random playouts of at most --rollout-plies plies), all K worlds of all games in one launch;
3. sums the root children's visit counts (root_stats) over the K worlds and plays the most visited move, ties to the
   lowest flat index.  Every world has the same legal moves for the searcher: its own pieces are known.
The searcher is player +1 and moves first.  Against the random player the setup is that of examples/pimc_one_ply.py
(same games, seed and opponent), so the two win counts compare directly.  --opponent pimc plays player -1 with the
one-ply PIMC searcher of examples/pimc_one_ply.py (its `search`: --pimc-worlds worlds, rollouts of at most
--pimc-plies plies).

    python examples/determinized_mcts.py [--games 256] [--worlds 16] [--iterations 128] [--rollout-plies 100]
                                         [--opponent random|pimc]

With the defaults the searcher won 249 and lost 7 of 256 games against the random player, in 5.5 s, and won 191 and
lost 65 of 256 against one-ply PIMC, in 5.4 s, on a B200 at 1 000 W (profiles/r7e_examples.txt).
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


def search(e, st, games, K, iterations, plies, seed, draw):
    """the searcher's move (flat spatial index, its own frame) in each game of `games` (all with the searcher to move)"""
    n = games.numel()
    sub = DeviceState(st.board[games], st.aux[games], st.captured[games])
    worlds = e.sample_hidden_states(sub, n_samples=K, seed=seed, draw=draw)  # row g * K + k: world k of game g
    tree = e.search(worlds, iterations, max_plies=plies, seed=seed ^ (draw << 20))
    visits, _ = tree.root_stats()
    total = visits.view(n, K, -1).sum(1)
    return torch.argmax(total, dim=1).to(torch.int32)  # the first of equal maxima: the lowest index


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=256)
    ap.add_argument("--worlds", type=int, default=16)
    ap.add_argument("--iterations", type=int, default=128)
    ap.add_argument("--rollout-plies", type=int, default=100)
    ap.add_argument("--opponent", choices=("random", "pimc"), default="random")
    ap.add_argument("--pimc-worlds", type=int, default=16)
    ap.add_argument("--pimc-plies", type=int, default=200)
    ap.add_argument("--seed", type=int, default=1)
    args = ap.parse_args()
    G, K = args.games, args.worlds
    if args.opponent == "pimc":
        from pimc_one_ply import search as pimc_search

    e = StrategoEngine(BARRAGE_STRATEGO_CONFIG, device="cuda:0")
    st = e.alloc_state(G)
    e.reset(st, seed=args.seed, shuffle=True)
    out = e.alloc_outputs(G, partial=False, full=False, mask=True, sample=True)
    e.observe(st, out=out, partial=False, full=False, mask=True)
    random_actions = e.sample_valid(out["valid_mask"], seed=args.seed)
    to_move = out["player"].clone()
    winner = torch.zeros(G, dtype=torch.int8, device=e.device)
    finished = torch.zeros(G, dtype=torch.bool, device=e.device)
    t0 = time.time()
    decisions = 0
    for ply in range(int(BARRAGE_STRATEGO_CONFIG["max_turns"]) + 1):
        games = torch.nonzero((to_move == 1) & ~finished).flatten()
        actions = random_actions.clone()
        if games.numel():
            actions[games] = search(e, st, games, K, args.iterations, args.rollout_plies, args.seed, ply)
            decisions += games.numel()
        if args.opponent == "pimc":
            other = torch.nonzero((to_move == -1) & ~finished).flatten()
            if other.numel():
                actions[other] = pimc_search(e, st, other, args.pimc_worlds, args.pimc_plies, args.seed + 1, ply)
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
                "one-ply PIMC (%d worlds, %d-ply rollouts)" % (args.pimc_worlds, args.pimc_plies))
    print("determinized MCTS (%d worlds, %d iterations, %d-ply random playouts) vs %s, %d Barrage games, %d plies, "
          "%.1f s" % (K, args.iterations, args.rollout_plies, opponent, G, ply + 1, elapsed))
    print("searcher wins %d, losses %d, unfinished or turn limit %d; %d searcher decisions" % (
        wins, losses, G - wins - losses, decisions))


if __name__ == "__main__":
    main()
