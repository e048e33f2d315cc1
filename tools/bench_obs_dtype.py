"""float32 against bfloat16 observations, in one process on one GPU (obs_dtype of StrategoEngine).

    python tools/bench_obs_dtype.py [--out FILE] [--sweep] [--quick]

  * fused step: each workload of bench.py, de-phased as bench.py does it (render-free steps from a seeded reset), then
    the float32 and the bfloat16 engine step copies of the same state, alternating, CUDA events around the timed steps;
    the roofline fraction uses the algorithmic bytes of the element type (observations at 4 or 2 bytes per element)
  * --sweep: warps per SM x issue point of the 16-bit tiles (sx_config_set_tuning), the evidence behind the built-in
    shapes of sx_kernels.cu (shape16)
  * rollout: the Standard conv-policy rollout of bench.py (131 072 games), float32 observations + the .to(bf16) cast
    against bf16 observations fed to the policy directly
  * e2e: HostBufferEnv (host actions in, host outputs out) with float32 and bf16 observations
Prints the card name and power limit first."""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bench import WORKLOADS, measured_peak  # noqa: E402
from stratego_env_b200.config import VERSION_CONFIGS, as_version  # noqa: E402
from stratego_env_b200.engine import StrategoEngine, load_setup_table  # noqa: E402

STEP_WORKLOADS = ["barrage", "standard", "standard_both", "micro", "tiny", "octa", "medium", "fives", "standard2"]
SWEEP_WORKLOADS = ["barrage", "standard", "standard_both", "octa", "medium", "fives", "standard2", "micro"]
LOG = []


def say(line=""):
    print(line, flush=True)
    LOG.append(line)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def bytes_per_step(lay, full, eb):
    """bench.py's algorithmic bytes (SURVEY.md 8(d)) with `eb` bytes per observation element"""
    obs = lay.cells * 67 * eb + (lay.cells * 79 * eb if full else 0)
    state = lay.cells + 4 * lay.pieces_per_side + 16
    return obs + lay.cells * lay.spatial_channels + 2 * state + 13


class Workload:
    def __init__(self, name, envs=None):
        w = WORKLOADS[name]
        self.name, self.w, self.B, self.full = name, w, envs or w["envs"], w["full"]
        self.cfg = VERSION_CONFIGS[as_version(w["version"])]
        self.table = load_setup_table(w["table"]) if w["table"] else None
        eng = self.engine(torch.float32)
        self.setups = eng.upload_setups(self.table) if self.table is not None else None
        self.st0 = eng.alloc_state(self.B)
        eng.reset(self.st0, seed=1, setups=self.setups, shuffle=self.setups is None)
        lean = eng.alloc_outputs(self.B, partial=False, full=False, mask=False, sample=True)
        acts = eng.sample_valid(eng.valid_mask(self.st0), seed=1)
        for _ in range(w["dephase"]):
            eng.step_all(self.st0, acts, lean, auto_reset=True, sample_next=True, setups=self.setups,
                         shuffle=self.setups is None, seed=1)
            acts, lean["next_action"] = lean["next_action"], acts
        torch.cuda.synchronize()
        self.a0 = acts.clone()

    def engine(self, dtype):
        return StrategoEngine(self.cfg, device="cuda:0", p2_rot180=self.table is None, obs_dtype=dtype)

    def runner(self, eng):
        st, acts = self.st0.clone(), self.a0.clone()
        out = eng.alloc_outputs(self.B, partial=True, full=self.full, mask=True, sample=True)

        def run(n):
            nonlocal acts
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n):
                eng.step_all(st, acts, out, auto_reset=True, sample_next=True, setups=self.setups,
                             shuffle=self.setups is None, seed=1)
                acts, out["next_action"] = out["next_action"], acts
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / n
        return run


def step_table(names, steps, reps):
    peak, peak_src = measured_peak()
    say("== fused step, float32 vs bfloat16 observations (alternating, %d reps x %d steps, min ms per step; "
        "peak %.0f GB/s: %s)" % (reps, steps, peak, peak_src))
    for name in names:
        wl = Workload(name)
        engines = {"f32": wl.engine(torch.float32), "bf16": wl.engine(torch.bfloat16)}
        runs = {k: wl.runner(e) for k, e in engines.items()}
        times = {k: [] for k in runs}
        for k in runs:
            runs[k](4)
        for _ in range(reps):
            for k in runs:
                runs[k](2)
                times[k].append(runs[k](steps))
        res = {}
        for k, e in engines.items():
            ms = min(times[k])
            nb = bytes_per_step(e.layout, wl.full, 4 if k == "f32" else 2)
            info = e.launch_info(partial=True, full=wl.full, mask=True)
            res[k] = ms
            say("%-14s %-4s B=%-8d %7.3f ms  %8.1f M env-steps/s  %6d B/step  %6.0f GB/s  frac %.3f  warps %2d  %s  "
                "(reps %s)" % (name, k, wl.B, ms, wl.B / ms / 1e3, nb, wl.B * nb / ms / 1e6, wl.B * nb / ms / 1e6 / peak,
                               info["warps_per_block"], "toy" if info["thread_per_game"] else "warp",
                               " ".join("%.3f" % t for t in times[k])))
        say("%-14s bf16 / f32 throughput: %.3f" % (name, res["f32"] / res["bf16"]))
        del wl, engines, runs
        torch.cuda.empty_cache()


def sweep(names, steps, reps):
    say("== 16-bit launch-shape sweep (sx_config_set_tuning: warps per SM : issue point 0 late / 1 after outcome / 2 top)")
    for name in names:
        wl = Workload(name)
        warps = [4, 6, 8, 10, 12, 16, 20, 24, 32] if wl.B <= 524288 else [8, 12, 16, 24, 32]
        best = None
        for wp in warps:
            for issue in (0, 1, 2):
                e = wl.engine(torch.bfloat16)
                e.set_tuning(wp, issue)
                run = wl.runner(e)
                run(4)
                ms = min(run(steps) for _ in range(reps))
                info = e.launch_info(partial=True, full=wl.full, mask=True)
                say("%-14s bf16 warps:issue=%2d:%d (resident %2d, %s) %7.3f ms  %8.1f M env-steps/s" % (
                    name, wp, issue, info["warps_per_block"], "toy" if info["thread_per_game"] else "warp", ms,
                    wl.B / ms / 1e3))
                if best is None or ms < best[0]:
                    best = (ms, wp, issue)
                del e, run
        say("%-14s best bf16 shape: warps %d issue %d, %.3f ms" % (name, best[1], best[2], best[0]))
        del wl
        torch.cuda.empty_cache()


def rollout(envs, steps, reps):
    from stratego_env_b200 import BatchedStrategoEnv, GameVersions, ObservationModes
    say("== Standard conv-policy rollout, %d games (policy in bf16, as bench.py's rollout leg)" % envs)
    legs = {}
    for dtype, tag in ((torch.float32, "f32 obs + .to(bf16)"), (torch.bfloat16, "bf16 obs fed directly")):
        env = BatchedStrategoEnv({"version": GameVersions.STANDARD, "human_inits": True,
                                  "observation_mode": ObservationModes.PARTIALLY_OBSERVABLE},
                                 num_envs=envs, device="cuda:0", seed=3, obs_dtype=dtype)
        torch.manual_seed(0)
        A = env.spatial_action_size[2]
        policy = torch.nn.Sequential(
            torch.nn.Conv2d(67, 64, 3, padding=1), torch.nn.ReLU(), torch.nn.Conv2d(64, 64, 3, padding=1), torch.nn.ReLU(),
            torch.nn.Conv2d(64, A, 3, padding=1)).to("cuda:0", torch.bfloat16).to(memory_format=torch.channels_last)
        legs[tag] = [env, policy, env.reset()]

    def run(tag, n):
        env, policy, obs = legs[tag]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            x = obs["partial_observation"].permute(0, 3, 1, 2)
            if x.dtype != torch.bfloat16:
                x = x.to(torch.bfloat16)
            logits = policy(x).permute(0, 2, 3, 1).contiguous()
            obs, _, _, infos = env.step(env.sample_actions_from_logits(logits))
        e1.record()
        torch.cuda.synchronize()
        legs[tag][2] = obs
        assert not infos["illegal_action"].any().item()
        return e0.elapsed_time(e1) / n
    times = {t: [] for t in legs}
    with torch.no_grad():
        for t in legs:
            run(t, 3)
        for _ in range(reps):
            for t in legs:
                times[t].append(run(t, steps))
    for t, v in times.items():
        say("rollout %-24s %7.3f ms per step  %7.2f M env-steps/s  (reps %s)" % (
            t, min(v), envs / min(v) / 1e3, " ".join("%.3f" % x for x in v)))
    legs.clear()
    torch.cuda.empty_cache()


def e2e(envs, steps, reps):
    from stratego_env_b200.host_env import HostBufferEnv
    import time
    say("== e2e through host buffers (HostBufferEnv, Barrage, %d games, PO + mask, 16 chunks)" % envs)
    wl = WORKLOADS["barrage"]
    cfg = VERSION_CONFIGS[as_version(wl["version"])]
    table = load_setup_table(wl["table"])
    envs_by = {}
    for dtype, tag in ((torch.float32, "f32"), (torch.bfloat16, "bf16")):
        eng = StrategoEngine(cfg, device="cuda:0", p2_rot180=False, obs_dtype=dtype)
        h = HostBufferEnv(eng, envs, setups=table, seed=5, n_chunks=16)
        envs_by[tag] = [h, h.reset()]
    times = {t: [] for t in envs_by}

    def run(tag, n):
        h, host = envs_by[tag]
        t0 = time.perf_counter()
        for _ in range(n):
            h.actions.copy_(host["next_action"])
            host = h.step()
        t1 = time.perf_counter()
        envs_by[tag][1] = host
        return (t1 - t0) / n * 1e3
    for t in envs_by:
        run(t, 2)
    for _ in range(reps):
        for t in envs_by:
            times[t].append(run(t, steps))
    for t, v in times.items():
        h = envs_by[t][0]
        say("e2e %-5s %7.3f ms per step  %6.2f M env-steps/s  D2H %6.2f MB per step  %5.1f GB/s  (reps %s)" % (
            t, min(v), envs / min(v) / 1e3, h.d2h_bytes_per_step / 1e6, h.d2h_bytes_per_step / min(v) / 1e6,
            " ".join("%.2f" % x for x in v)))
    for h, _ in envs_by.values():
        h.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the report to this file")
    ap.add_argument("--sweep", action="store_true", help="run the 16-bit launch-shape sweep")
    ap.add_argument("--no-steps", action="store_true", help="skip the fused-step table")
    ap.add_argument("--quick", action="store_true", help="fewer steps (a smoke run, not a measurement)")
    ap.add_argument("--workloads", default=",".join(STEP_WORKLOADS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_obs_dtype.py measures on a GPU; none found")
    steps, reps = (3, 1) if args.quick else (20, 3)
    say("card: %s" % card())
    if not args.no_steps:
        step_table(args.workloads.split(","), steps, reps)
    if args.sweep:
        sweep(SWEEP_WORKLOADS, steps, reps)
    rollout(131072, 10 if not args.quick else 2, reps)
    e2e(131072, 5 if not args.quick else 1, reps)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(LOG) + "\n")


if __name__ == "__main__":
    main()
