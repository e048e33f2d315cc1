"""Time move expansion (StrategoEngine.expand_moves: sx_count_moves + sx_expand_moves) on one GPU against the
composition it replaces, on the same games.

    python tools/bench_expand.py [--launches 20] [--rounds 5] [--out FILE]

(profiles/r7a_expand_moves.txt is this tool's output.)  Workloads: 262 144 Barrage games and 131 072 Standard games,
de-phased (game b plays its own number of random moves in [0, 120) first), and 262 144 Micro games (de-phased over
[0, 12): Micro games last 20 plies).  The composition is what a user writes without the new call: valid_mask, nonzero,
dropping the noop channel, index_select of the three state tensors, step on the gathered rows.

Before timing, both paths run once at full size and every output (children, actions, parents, offsets, the six
scalars) must be identical.  Per workload: children per game; the count pass and the expand pass alone (5 warm-up
launches, then `--launches` launches between two CUDA events); expand_moves end to end and the composition end to end
(CUDA events around the whole call, host synchronisation included), alternated in one process for `--rounds` rounds,
median reported; children per second; the bytes the expand pass writes as a share of the device-to-device copy rate
measured in the same process.  The card name and power limit are printed first."""
import argparse
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from stratego_env_b200 import _lib  # noqa: E402
from stratego_env_b200.config import VERSION_CONFIGS, as_version  # noqa: E402
from stratego_env_b200.engine import DeviceState, StrategoEngine  # noqa: E402


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


def dephased(e, B, steps, seed=1):
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


def composition(e, st):
    """the five separate passes: mask, nonzero (a host synchronisation), noop dropped, gather, step"""
    B, A = st.num_envs, e.spatial_channels
    mask = e.valid_mask(st)
    mask[..., A - 1] = 0
    parent, idx = torch.nonzero(mask.reshape(B, -1), as_tuple=True)
    kids = DeviceState(st.board.index_select(0, parent), st.aux.index_select(0, parent),
                       st.captured.index_select(0, parent))
    actions = idx.to(torch.int32)
    out = e.step(kids, actions)
    return kids, actions, parent, out


def check_identical(e, st):
    ex = e.expand_moves(st)
    kids, actions, parent, out = composition(e, st)
    same = torch.equal(ex.actions, actions) and torch.equal(ex.parent, parent)
    same &= torch.equal(ex.offsets[1:] - ex.offsets[:-1], torch.bincount(parent, minlength=st.num_envs))
    for name in ("board", "aux", "captured"):
        same &= torch.equal(getattr(ex.states, name), getattr(kids, name))
    for name in ("reward", "done", "winner", "ending_invalid", "illegal", "player"):
        same &= torch.equal(getattr(ex, name), out[name])
    if not same:
        raise SystemExit("expand_moves and the composition differ")
    return ex


def e2e(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e-3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    say("card: %s" % card())
    peak = copy_rate()
    say("device-to-device copy: %.2f TB/s (read + written bytes of a 2 GiB torch copy)" % (peak / 1e12))
    stream = lambda: torch.cuda.current_stream().cuda_stream  # noqa: E731
    say("%-9s %7s %8s %8s %8s %9s %9s %10s %9s %8s" % (
        "variant", "games", "kids", "kids/gm", "count ms", "expand ms", "e2e ms", "compose ms", "Gkids/s", "of copy"))
    for name, B, steps in (("barrage", 262144, 120), ("standard", 131072, 120), ("micro", 262144, 12)):
        e = StrategoEngine(VERSION_CONFIGS[as_version(name)], device="cuda:0")
        st = dephased(e, B, steps)
        ex = check_identical(e, st)
        T = ex.states.num_envs
        counts = torch.empty(B, dtype=torch.int32, device="cuda")
        t_count = timed(lambda: _lib.check(e.lib.sx_count_moves(e._cfg, st.as_struct(), B, counts.data_ptr(), stream())),
                        args.launches)
        out = e.alloc_state(T)
        scal = e.alloc_outputs(T, partial=False, full=False, mask=False)
        acts = torch.empty(T, dtype=torch.int32, device="cuda")
        sstruct = e._outputs_struct(scal)
        t_expand = timed(lambda: _lib.check(e.lib.sx_expand_moves(e._cfg, st.as_struct(), B, ex.offsets.data_ptr(), T,
                                                                  out.as_struct(), acts.data_ptr(), sstruct, stream())),
                         args.launches)
        del out, scal, acts
        e.expand_moves(st)  # warm-up of both paths' allocations and launches
        composition(e, st)
        fused, comp = [], []
        for _ in range(args.rounds):  # alternated in one process
            fused.append(e2e(lambda: e.expand_moves(st)))
            comp.append(e2e(lambda: composition(e, st)))
        t_fused, t_comp = statistics.median(fused), statistics.median(comp)
        lay = e.layout
        row_bytes = lay.board_stride + 2 * lay.aux_stride + 2 * lay.captured_stride + 4 + 4 + 5  # + action + 6 scalars
        written = T * row_bytes
        say("%-9s %7d %8d %8.2f %8.3f %9.3f %9.3f %10.3f %9.2f %7.1f%%" % (
            name, B, T, T / B, t_count * 1e3, t_expand * 1e3, t_fused * 1e3, t_comp * 1e3, T / t_fused / 1e9,
            100 * written / t_expand / peak))
        say("          e2e rounds ms: expand_moves %s | composition %s" % (
            " ".join("%.3f" % (x * 1e3) for x in fused), " ".join("%.3f" % (x * 1e3) for x in comp)))
        del e, st, ex
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
