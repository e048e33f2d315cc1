"""Launch-shape sweep of the SHIPPED library through sx_config_set_tuning (result-preserving knobs only): one process,
one de-phased state, many (warps per SM, issue point, compact movers) settings; `-` keeps the built-in choice.
    python tools/sweep_tuning.py <workload> "<warps>:<issue 0|1|2>:<compact 0|1>,..." [envs]"""
import sys

import torch

sys.path.insert(0, ".")
from bench import WORKLOADS, algorithmic_bytes_per_step  # noqa: E402
from stratego_env_b200.config import VERSION_CONFIGS, as_version  # noqa: E402
from stratego_env_b200.engine import StrategoEngine, load_setup_table  # noqa: E402


def main():
    wl = sys.argv[1] if len(sys.argv) > 1 else "barrage"
    combos = [tuple(c.split(":")) for c in (sys.argv[2] if len(sys.argv) > 2 else "-:-:-").split(",")]
    w = WORKLOADS[wl]
    B = int(sys.argv[3]) if len(sys.argv) > 3 else w["envs"]
    cfg = VERSION_CONFIGS[as_version(w["version"])]
    table = load_setup_table(w["table"]) if w["table"] else None
    shuffle = table is None
    eng = StrategoEngine(cfg, device="cuda:0", p2_rot180=table is None)
    setups = eng.upload_setups(table) if table is not None else None
    st0 = eng.alloc_state(B)
    eng.reset(st0, seed=1, setups=setups, shuffle=shuffle)
    lean = eng.alloc_outputs(B, partial=False, full=False, mask=False, sample=True)
    first = eng.alloc_outputs(B, partial=False, full=False, mask=True, sample=False)
    eng.observe(st0, out=first, partial=False, full=False, mask=True)
    actions = eng.sample_valid(first["valid_mask"], seed=1)
    del first
    for _ in range(w["dephase"]):
        eng.step_all(st0, actions, lean, auto_reset=True, sample_next=True, setups=setups, shuffle=shuffle, seed=1)
        actions, lean["next_action"] = lean["next_action"], actions
    torch.cuda.synchronize()
    a0 = actions.clone()
    lay = eng.layout
    nbytes = algorithmic_bytes_per_step(lay.cells, lay.spatial_channels, lay.pieces_per_side, w["full"])
    out = eng.alloc_outputs(B, partial=True, full=w["full"], mask=True, sample=True)
    for combo in combos:
        e = StrategoEngine(cfg, device="cuda:0", p2_rot180=table is None)
        e.set_tuning(*[-1 if v in ("", "-") else int(v) for v in combo])
        st, acts = st0.clone(), a0.clone()
        times = []
        for rep in range(3):
            for phase, n in (("warm", 4), ("timed", 20)):
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(n):
                    e.step_all(st, acts, out, auto_reset=True, sample_next=True, setups=setups, shuffle=shuffle, seed=1)
                    acts, out["next_action"] = out["next_action"], acts
                e1.record()
                torch.cuda.synchronize()
                if phase == "timed":
                    times.append(e0.elapsed_time(e1) / n)
        ms = min(times)
        info = e.launch_info(partial=True, full=w["full"], mask=True)
        print("%-14s warps:issue:compact=%-8s warps %2d regs %3d : %7.3f ms  %6.1f M env-steps/s  %5.0f GB/s  frac %.3f  (reps %s)" % (
            wl, ":".join(combo), info["warps_per_block"], info["regs_per_thread"], ms, B / ms / 1e3, B * nbytes / ms / 1e6,
            B * nbytes / ms / 1e6 / 6546.6, " ".join("%.3f" % t for t in times)), flush=True)


if __name__ == "__main__":
    main()
