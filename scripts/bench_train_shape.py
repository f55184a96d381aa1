"""Training step at the reference's own training shape: `lq_size: 60`, `batch_size_per_gpu: 16` of train_SAVSR_Vimeo90K_asBI.yml
(16 x 7 x 3 x 60 x 60 per GPU), one scale per step from a fixed rotation.  Three arms in one process, timed alternately:

  native_trainer  trainplan.NativeTrainer, one CUDA graph per scale (forward + loss + backward) plus one for Adam + EMA
  native_trainer_cosine  the same with a cosine schedule stepped after every step (torch.optim.lr_scheduler.CosineAnnealingLR on
                  tr.optimizer): the lr changes every step, so each step adds one one-float fill of the device lr before the optimizer graph
  module_native   the module as the reference's optimize_parameters drives it: SAVSR.train(), net(lq), the caller's Charbonnier,
                  backward(), torch.optim.Adam -- the native launch list behind one autograd node (trainplan.ModuleTraining)
  module_stage_a  the same loop with native_training = False: the ATen tape of savsr_b200/train.py (what this shape ran before
                  the native attention kernels took more than 8 samples)

Every scale of the rotation is warmed up first (graphs captured).  Each timed window is a host clock around --steps steps that ends in a
device synchronise.  Prints one JSON line.  Usage: python scripts/bench_train_shape.py --batch 16 --lq 60 --steps 16 [--rounds 3]
(the cost of a schedule: --batch 4 --lq 64 --arms native_trainer,native_trainer_cosine)
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import flops_per_frame, hw_out  # noqa: E402

# eight scales of the 60-entry list of vimeo90k_dataset.py:178-202, symmetric and asymmetric (the rotation of bench.py's train_cfg5)
SCALES = [(2, 2), (3, 3), (4, 4), (1.5, 4), (2.7, 2.7), (1.1, 1.1), (3.5, 2), (4, 1.5)]


def gpu_identity(index: int) -> dict:
    """Card name and power limit, read in the same run as the timings (a read-only nvidia-smi query)."""
    out = dict(name=torch.cuda.get_device_name(index))
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30)
        pl, mx = (v.strip() for v in r.stdout.strip().split(","))
        out.update(power_limit_w=float(pl), max_sm_clock_mhz=int(mx))
    except (OSError, ValueError, subprocess.SubprocessError) as e:
        out.update(power_limit_w=None, query_error=str(e))
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--batch", type=int, default=16, help="LR crops per GPU (the YAML's batch_size_per_gpu)")
    ap.add_argument("--lq", type=int, default=60, help="LR crop side (the YAML's lq_size)")
    ap.add_argument("--steps", type=int, default=16, help="steps per timed window and arm (a multiple of the 8-scale rotation is fairest)")
    ap.add_argument("--rounds", type=int, default=3, help="timed windows per arm, the arms alternating")
    ap.add_argument("--arms", default="native_trainer,module_native,module_stage_a")
    args = ap.parse_args()
    if args.steps < 1 or args.rounds < 1:
        ap.error("--steps and --rounds must be >= 1")
    if not torch.cuda.is_available():
        sys.exit("bench_train_shape.py measures on a CUDA device; none is visible")
    import savsr_b200
    from savsr_b200 import train as T
    from savsr_b200 import trainplan as TP

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    torch.backends.cudnn.benchmark = True                     # lbasicsr/train.py sets it (stage A's ATen ops use cuDNN)
    b, h = args.batch, args.lq
    torch.manual_seed(0)
    sd = savsr_b200.SAVSR().state_dict()
    gen = torch.Generator().manual_seed(100)
    lq = torch.rand(b, 7, 3, h, h, generator=gen).to(dev)
    gts = {s: torch.rand(b, 3, *hw_out(h, h, s), generator=gen).to(dev) for s in SCALES}

    def new_net():
        net = savsr_b200.SAVSR().to(dev)
        net.load_state_dict(sd, strict=True)
        net.train()
        return net

    arms = {}
    for name in args.arms.split(","):
        mem0 = torch.cuda.memory_allocated(dev)
        torch.cuda.reset_peak_memory_stats(dev)
        net = new_net()
        if name in ("native_trainer", "native_trainer_cosine"):
            tr = TP.NativeTrainer(net, use_graph=True)
            sched = torch.optim.lr_scheduler.CosineAnnealingLR(tr.optimizer, T_max=1_000_000, eta_min=1e-7) if name.endswith("cosine") else None

            def step(i, tr=tr, sched=sched):
                s = SCALES[i % len(SCALES)]
                loss = tr.step(lq, gts[s], s)
                if sched is not None:
                    sched.step()
                return loss
            warm = len(SCALES)                                 # the first step of each scale captures its graph
        elif name in ("module_native", "module_stage_a"):
            net.native_training = name == "module_native"
            opt = torch.optim.Adam(net.parameters(), lr=2e-4, betas=(0.9, 0.99))

            def step(i, net=net, opt=opt):
                s = SCALES[i % len(SCALES)]
                net.set_scale(s)
                opt.zero_grad(set_to_none=True)
                loss = T.charbonnier(net(lq), gts[s])
                loss.backward()
                opt.step()
                return loss.detach()
            warm = 2 * len(SCALES) if name == "module_native" else len(SCALES)   # the module captures a scale's graphs at its second use
        else:
            ap.error(f"unknown arm {name}")
        for i in range(warm):
            step(i)
        torch.cuda.synchronize(dev)
        ent = dict(step=step, ms=[], loss=None, net=net,
                   max_memory_allocated_gib=round(torch.cuda.max_memory_allocated(dev) / 2 ** 30, 2),
                   arm_memory_gib=round((torch.cuda.max_memory_allocated(dev) - mem0) / 2 ** 30, 2))
        if name.startswith("native_trainer"):
            plan = next(iter(tr.plans.values()))
            ent["arena_gib"] = round(plan.arena_t.numel() * 2 / 2 ** 30, 2)
            ent["t_arena_gib"] = round(plan.tarena.numel() * 2 / 2 ** 30, 2)
            ent["slots"], ent["t_slots"] = plan.n_slots, plan.n_tslots
        state = net.__dict__.get("_train_state")
        if name == "module_native":
            assert state is not None and all(p.g_fwd is not None for p in state.plans.values()), "module arm is not on the native graphs"
        if name == "module_stage_a":
            assert state is None, "stage-A arm took the native path"
        arms[name] = ent

    def timed(ent):
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        last = None
        for i in range(args.steps):
            last = ent["step"](i)
        torch.cuda.synchronize(dev)
        ent["ms"].append((time.perf_counter() - t0) * 1e3 / args.steps)
        ent["loss"] = float(last)

    for _ in range(args.rounds):
        for ent in arms.values():
            timed(ent)

    step_flops = statistics.fmean(3.0 * flops_per_frame(h, h, *hw_out(h, h, s)) * b for s in SCALES)
    out = {"metric": "train_step_ms_at_yaml_shape", "gpu": gpu_identity(0), "batch": b, "lq": [h, h], "frames": 7,
           "scales": [list(s) for s in SCALES], "steps_per_window": args.steps, "rounds": args.rounds,
           "timing": "host perf_counter around --steps steps ending in torch.cuda.synchronize; arms alternate per round; inputs device-resident",
           "flops": "algorithmic: 3 x the forward FLOPs of DESIGN section 4 per sample, mean over the rotation",
           "algorithmic_tflop_per_step": round(step_flops / 1e12, 3), "arms": {}}
    for name, ent in arms.items():
        ms = statistics.median(ent["ms"])
        row = {"ms_per_step": round(ms, 2), "ms_per_step_rounds": [round(v, 2) for v in ent["ms"]],
               "samples_per_s": round(b / (ms / 1e3), 1), "algorithmic_tflops": round(step_flops / (ms / 1e3) / 1e12, 1),
               "last_loss": round(ent["loss"], 5), "max_memory_allocated_gib": ent["max_memory_allocated_gib"], "arm_memory_gib": ent["arm_memory_gib"]}
        for k in ("arena_gib", "t_arena_gib", "slots", "t_slots"):
            if k in ent:
                row[k] = ent[k]
        out["arms"][name] = row
    if "native_trainer" in arms and "native_trainer_cosine" in arms:
        out["cosine_schedule_cost_ms"] = round(statistics.median(arms["native_trainer_cosine"]["ms"]) - statistics.median(arms["native_trainer"]["ms"]), 3)
    if "module_native" in arms and "module_stage_a" in arms:
        out["module_native_speedup_vs_stage_a"] = round(statistics.median(arms["module_stage_a"]["ms"]) / statistics.median(arms["module_native"]["ms"]), 2)
    out["memory_note"] = ("max_memory_allocated_gib: the process peak after the arm's warm-up over the whole rotation (arms are built in the order "
                          "listed, so it includes the arms before it); arm_memory_gib: that peak minus what was allocated before the arm was built")
    print(json.dumps(out))


if __name__ == "__main__":
    main()
