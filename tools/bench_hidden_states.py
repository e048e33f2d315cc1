"""Time sx_sample_hidden_states (determinization of the opponent's hidden pieces) on one GPU, next to one fused step
over the same games.

    python tools/bench_hidden_states.py [--launches 50] [--out FILE]

Cases: Barrage 262 144 games x K = 1 and 16, Standard 131 072 x K = 1 and 16, 64 Standard games x 4 096 samples.  The
states are de-phased first (game b plays its own number of random moves in [0, 120)), the viewer is the player to move.
Per case: 5 warm-up launches, then `--launches` launches between two CUDA events.  Reported: rows (samples) per second,
the bytes a launch writes (board + aux + capture list per row) and that write rate as a share of the device-to-device
copy rate measured in the same process (a 2 GiB torch copy: read + written bytes over time), and for the first four cases
one fused step (PO observation + mask + sampled next action, auto-reset) over the same games, for scale.  The card name
and power limit are printed first."""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from stratego_env_b200.config import BARRAGE_STRATEGO_CONFIG, STANDARD_STRATEGO_CONFIG  # noqa: E402
from stratego_env_b200.engine import StrategoEngine  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def timed(fn, launches, warmup=5):
    for _ in range(warmup):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(launches):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / launches * 1e-3  # seconds per launch


def copy_rate():
    n = 2 << 30
    src = torch.empty(n, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)
    src.fill_(1)
    t = timed(lambda: dst.copy_(src), 20)
    return 2 * n / t


def dephased(e, B, steps=120, seed=1):
    st = e.alloc_state(B)
    e.reset(st, seed=seed, shuffle=True)
    out = e.alloc_outputs(B, partial=False, full=False, mask=True, sample=True)
    e.observe(st, out=out, partial=False, full=False, mask=True)
    actions = e.sample_valid(out["valid_mask"], seed=seed)
    g = torch.Generator(device="cuda").manual_seed(seed)
    target = torch.randint(0, steps, (B,), generator=g, device="cuda")
    for s in range(steps):
        a = torch.where(target > s, actions, torch.full_like(actions, -1))
        e.step_all(st, a, out, auto_reset=False, sample_next=True, seed=seed, shuffle=True)
        actions = torch.where(target > s, out["next_action"], actions)
    return st


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    say("card: %s" % card())
    peak = copy_rate()
    say("device-to-device copy: %.2f TB/s (read + written bytes of a 2 GiB torch copy)" % (peak / 1e12))
    cases = [("barrage", BARRAGE_STRATEGO_CONFIG, 262144, 1), ("barrage", BARRAGE_STRATEGO_CONFIG, 262144, 16),
             ("standard", STANDARD_STRATEGO_CONFIG, 131072, 1), ("standard", STANDARD_STRATEGO_CONFIG, 131072, 16),
             ("standard", STANDARD_STRATEGO_CONFIG, 64, 4096)]
    say("%-9s %8s %6s %10s %12s %10s %9s %12s" % ("variant", "games", "K", "ms", "Mrows/s", "MB written", "of copy",
                                                  "fused step ms"))
    engines, states = {}, {}
    for name, cfg, B, K in cases:
        e = engines.setdefault(name, StrategoEngine(cfg, device="cuda:0"))
        st = states.get((name, B))
        if st is None:
            st = states[(name, B)] = dephased(e, B)
        out = e.alloc_state(B * K)
        lay = e.layout
        row_bytes = lay.board_stride + 2 * lay.aux_stride + 2 * lay.captured_stride
        t = timed(lambda: e.lib.sx_sample_hidden_states(e._cfg, st.as_struct(), B, 0, None, K, 5, 1, out.as_struct(),
                                                        None, torch.cuda.current_stream().cuda_stream), args.launches)
        written = B * K * row_bytes
        fused = "-"
        if B >= 4096:
            work = st.clone()
            o = e.alloc_outputs(B, partial=True, full=False, mask=True, sample=True)
            e.observe(work, out=o)
            bufs = [e.sample_valid(o["valid_mask"], seed=2), o["next_action"]]

            def step():  # plays the sampled actions; the two action buffers alternate as input and output
                o["next_action"] = bufs[1]
                e.step_all(work, bufs[0], o, auto_reset=True, sample_next=True, seed=2, shuffle=True)
                bufs.reverse()
            fused = "%.3f" % (timed(step, args.launches) * 1e3)
        say("%-9s %8d %6d %10.4f %12.1f %10.1f %8.1f%% %12s" % (name, B, K, t * 1e3, B * K / t / 1e6, written / 1e6,
                                                                100 * written / t / peak, fused))
        del out
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
