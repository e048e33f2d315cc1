"""One-ply PIMC (perfect-information Monte Carlo) on Barrage: a searcher against the uniformly random player.

At each of its turns the searcher, for every game in the batch at once:
1. draws K complete worlds that agree with what it knows (sample_hidden_states, viewer = the player to move);
2. expands every world (expand_moves): one child per legal move, the same action list in every world;
3. plays every child on with uniformly random moves (playout) for at most --rollout-plies plies, scoring a win +1, a
   loss -1 and an unfinished rollout or a turn-limit ending 0;
4. averages the score per (game, position in the action list) over the K worlds and plays the argmax.
The random player moves uniformly among its legal moves.  The searcher is player +1 and moves first.

    python examples/pimc_one_ply.py [--games 256] [--worlds 16] [--rollout-plies 200]

With the defaults the searcher won 228 and lost 28 of 256 games, in 1.4 s on a B200 at 1 000 W
(profiles/r7c_examples.txt).
"""
import argparse
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from stratego_env_b200.config import BARRAGE_STRATEGO_CONFIG  # noqa: E402
from stratego_env_b200.engine import DeviceState, StrategoEngine  # noqa: E402


def search(e, st, games, K, plies, seed, draw):
    """the searcher's move (flat spatial index, its own frame) in each game of `games` (all with the searcher to move)"""
    n = games.numel()
    sub = DeviceState(st.board[games], st.aux[games], st.captured[games])
    worlds = e.sample_hidden_states(sub, n_samples=K, seed=seed, draw=draw)  # row g * K + k: world k of game g
    ex = e.expand_moves(worlds)
    T = ex.states.num_envs
    mover = -ex.player.float()  # the player who made the move (the child's player to move is the other one)
    rollout = e.playout(ex.states, max_plies=plies, seed=seed ^ draw)  # a child that is already over plays nothing
    score = torch.where(rollout.done == 1, rollout.winner.float() * mover, torch.zeros_like(mover))
    # child row -> (game, position j in the action list); the K worlds of a game share one action list
    game = ex.parent // K
    j = torch.arange(T, device=e.device) - ex.offsets[ex.parent]
    n_act = (ex.offsets[1:] - ex.offsets[:-1]).view(n, K)[:, 0]
    base = torch.zeros(n + 1, dtype=torch.int64, device=e.device)
    base[1:] = torch.cumsum(n_act, 0)
    slots = int(base[-1].item())
    total = torch.zeros(slots, device=e.device).scatter_add_(0, base[game] + j, score)  # K x the mean
    slot_game = torch.repeat_interleave(torch.arange(n, device=e.device), n_act, output_size=slots)
    slot_j = torch.arange(slots, device=e.device) - base[slot_game]
    best = torch.full((n,), -float("inf"), device=e.device).scatter_reduce_(0, slot_game, total, "amax")
    cand = torch.where(total == best[slot_game], slot_j, torch.full_like(slot_j, 1 << 30))
    j_best = torch.full((n,), 1 << 30, dtype=torch.int64, device=e.device).scatter_reduce_(0, slot_game, cand, "amin")
    return ex.actions[ex.offsets[torch.arange(n, device=e.device) * K] + j_best]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=256)
    ap.add_argument("--worlds", type=int, default=16)
    ap.add_argument("--rollout-plies", type=int, default=200)
    ap.add_argument("--seed", type=int, default=1)
    args = ap.parse_args()
    G, K = args.games, args.worlds

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
    for ply in range(int(BARRAGE_STRATEGO_CONFIG["max_turns"]) + 1):
        games = torch.nonzero((to_move == 1) & ~finished).flatten()
        actions = random_actions.clone()
        if games.numel():
            actions[games] = search(e, st, games, K, args.rollout_plies, args.seed, ply)
        e.step_all(st, actions, out, auto_reset=False, sample_next=True, seed=args.seed)
        ended = (out["done"] == 1) & ~finished
        winner = torch.where(ended, out["winner"], winner)
        finished |= ended
        if bool(finished.all()):
            break
        random_actions = out["next_action"].clone()
        to_move = out["player"].clone()
    wins, losses = int((winner == 1).sum()), int((winner == -1).sum())
    print("one-ply PIMC (%d worlds, %d-ply random rollouts) vs uniform random, %d Barrage games, %d plies, %.1f s"
          % (K, args.rollout_plies, G, ply + 1, time.time() - t0))
    print("searcher wins %d, losses %d, unfinished or turn limit %d" % (wins, losses, G - wins - losses))


if __name__ == "__main__":
    main()
