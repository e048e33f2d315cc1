"""Determinized rollouts: estimate each game's value for the player to move without looking at the opponent's hidden
pieces.

1. Play a batch of Barrage games a few random moves in.
2. Draw K complete game states per game that agree with what the player to move knows (sample_hidden_states).
3. Play every sampled world to its end with uniformly random moves (playout: one launch, no host loop).
4. Average the outcome per original game, from the point of view of its player to move.

    python examples/determinized_rollouts.py [--games 1024] [--worlds 32] [--max-plies 3000]
"""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from stratego_env_b200.batched_env import BatchedStrategoEnv  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=1024)
    ap.add_argument("--worlds", type=int, default=32)
    ap.add_argument("--max-plies", type=int, default=3000)
    args = ap.parse_args()
    B, K = args.games, args.worlds

    env = BatchedStrategoEnv({"version": "barrage"}, num_envs=B, seed=1, auto_reset=False, sample_actions=True)
    obs = env.reset()
    for _ in range(20):
        obs, _, _, _ = env.step(obs["sampled_action"])
    me = obs["player"].clone()  # the player to move in each original game

    worlds = env.sample_hidden_states(n_samples=K)  # row b * K + k: world k of game b
    res = env.engine.playout(worlds, max_plies=args.max_plies, seed=2)
    winner, finished = res.winner, res.done == 1
    value = (winner.view(B, K).float() * me.view(B, 1).float()).mean(1)  # +1 win, -1 loss, 0 draw or unfinished
    print("%d games x %d worlds, longest playout %d plies, %.1f %% of the worlds finished" % (
        B, K, int(res.plies.max().item()), 100 * finished.float().mean().item()))
    print("value for the player to move: mean %+.3f, min %+.3f, max %+.3f" % (value.mean().item(), value.min().item(),
                                                                             value.max().item()))
    print("first games:", " ".join("%+.2f" % v for v in value[:8].tolist()))


if __name__ == "__main__":
    main()
