#!/usr/bin/env python
"""bench.py — self-play throughput of the B200 engine on BASELINE.json's headline config.

    python bench.py --gpus N --steps K --warmup W          (N>1: launched by torch.distributed.run)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   (also writes the search state, see dump_outputs)

Workload (config.workload = "C3"): 19x19 Go (wq), 1024 concurrent games per GPU, 800 sims/move,
20-block x 256 dual net (F=18, FC=512, A'=362, DefaultConf batch 256), two random-init nets (agents A
and B, agogo.go:50-58), synthetic data = the self-play positions themselves.
  step   = one MCTS wave over all resident games: PUCT select/expand-prep for every game ->
           batched dual-net evaluation of both agents' leaves -> expand + backup
           (i.e. n_games simulations; every 801st wave is a move's root evaluation).
  value  = simulations/s over all GPUs, device-timed (CUDA events inside the engine are used for
           the kernel roofline; the step loop itself is bracketed by barrier + synchronize).
  e2e    = the same metric through the reference-facing call az_arena_step (one full Arena.Play
           ply: Search + Apply + Example read-back into host buffers), wall clock, host<->device
           copies inside the timed region.
The reference arm times the CPU oracle (restatement of the reference algorithm; no Go toolchain in
this image, see DESIGN.md) on the host cores: one step = one simulation of one game.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from agogo_b200 import _capi as K  # noqa: E402

WORKLOADS = {
    # name: (size, n_games, sims, k, blocks, fc, batch)
    "C3": dict(size=19, n_games=1024, sims=800, k=256, blocks=20, fc=512, batch=256),
    "C2": dict(size=9, n_games=256, sims=400, k=64, blocks=6, fc=128, batch=256),
}


def flops_per_eval(w):
    hw = w["size"] ** 2
    k, b, fc, a1 = w["k"], w["blocks"], w["fc"], hw + 1
    tower = 2 * b * (2 * 9 * k * k * hw) + 2 * 9 * 18 * k * hw
    heads = 2 * k * 2 * hw + 2 * 2 * hw * a1 + 2 * k * hw + 2 * hw * fc + 2 * fc
    return tower + heads


KERNELS = {
    # az_profile kernel_kind -> (label, tensor passes per algorithmic MAC, precision line)
    0: ("k_conv3x3_tc<BN,true,64> (fused residual-block conv, one CTA per 128 x BN tile, fp16 hi/lo 3-pass tcgen05)", 3.0,
        "fp32 semantics on fp16 tensor cores: hi/lo operand split, 3 tcgen05 passes, fp32 TMEM accumulate"),
    1: ("k_conv3x3_tc2 (fused residual-block conv, CTA pair / cta_group::2, per-tap tiles, fp16 hi/lo 3-pass tcgen05)", 3.0,
        "fp32 semantics on fp16 tensor cores: hi/lo operand split, 3 tcgen05 passes, fp32 TMEM accumulate"),
    2: ("k_conv3x3_tc2_f8 (CTA pair, per-tap tiles, hi*hi kind::f16 + E5M2 x E4M3 correction passes kind::f8f6f4)", 2.0,
        "AZ_FLAG_FAST_TOWER: fp16 main pass + two FP8 correction passes (~14.5-bit operands), fp32 TMEM accumulate"),
    3: ("k_conv3x3_tc2_halo<true> (CTA pair, activation halo tile + 9 row-shifted descriptor views, hi*hi kind::f16 + "
        "E5M2 x E4M3 correction passes kind::f8f6f4)", 2.0,
        "AZ_FLAG_FAST_TOWER: fp16 main pass + two FP8 correction passes (~14.5-bit operands), fp32 TMEM accumulate"),
    4: ("k_conv3x3_tc2_halo<false> (CTA pair, activation halo tile + 9 row-shifted descriptor views, fp16 hi/lo 3-pass "
        "tcgen05)", 3.0,
        "fp32 semantics on fp16 tensor cores: hi/lo operand split, 3 tcgen05 passes, fp32 TMEM accumulate"),
    5: ("k_net_small (whole 6 x 64 network of a leaf in one CTA: activations resident in shared memory, nine row-shifted "
        "descriptor views per layer, filters streamed by TMA, fp16 hi/lo 3-pass tcgen05, heads fused)", 3.0,
        "fp32 semantics on fp16 tensor cores: hi/lo operand split, 3 tcgen05 passes, fp32 TMEM accumulate"),
}


def make_desc(w, n_games, device, seed, sims=None, batch=None, flags=0):
    s = w["size"]
    return K.make_desc(K.GAME_WQ, s, s, 0, komi=7.5, sims=sims if sims is not None else w["sims"], n_games=n_games,
                       seed=seed, device=device, max_moves=2 * s * s, flags=flags,
                       nn=dict(k=w["k"], shared_layers=w["blocks"], fc=w["fc"], batch_size=batch or w["batch"],
                               features=18, action_space=s * s + 1))


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                if len(parts) >= 7:
                    self.rows.append(parts)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        reasons = []
        for name, col in (("hw_slowdown", 3), ("hw_thermal_slowdown", 4), ("sw_thermal_slowdown", 5), ("sw_power_cap", 6)):
            if any(r[col].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][1]),
                "power_w_max": max(float(r[2]) for r in self.rows), "samples": len(self.rows), "reasons": reasons}


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return p, "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def oracle_lib():
    so = os.path.join(ROOT, "oracle", "libazoracle.so")
    if not os.path.exists(so):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle")], stdout=subprocess.DEVNULL)
    return K.load(so)


DUMP_GAMES = 64  # games in the --dump-outputs sample


def dump_outputs(e, n_games, out_dir):
    """What a caller reads back after the last timed wave (az_tree_dump, az_game_state), for a fixed, seeded sample of
    games: visit count N, value sum W and prior P of every root child by move (pass last) in both agents' trees (zeros
    where a tree has no such child or no root yet), and the board.  Written as DIR/<name>.npy, float32 / float64."""
    games = np.sort(np.random.default_rng(0).choice(n_games, min(n_games, DUMP_GAMES), replace=False))
    A1 = e.action_space + 1
    visits = np.zeros((len(games), 2, A1), np.float64)
    wsum = np.zeros((len(games), 2, A1), np.float32)
    prior = np.zeros((len(games), 2, A1), np.float32)
    board = np.zeros((len(games), e.cells), np.float32)
    for i, g in enumerate(games.tolist()):
        for t in (0, 1):
            ch = e.tree_dump(g, t)
            ch = ch[ch[:, 0] == 1]  # rows: depth, move, N, W bits, P bits, expanded, n_children
            mv = np.where(ch[:, 1] == K.PASS, A1 - 1, ch[:, 1])
            visits[i, t, mv] = ch[:, 2]
            wsum[i, t, mv] = ch[:, 3].copy().view(np.float32)
            prior[i, t, mv] = ch[:, 4].copy().view(np.float32)
        board[i] = e.game_state(g)["board"]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("games", games.astype(np.float64)), ("root_visits", visits), ("root_value_sum", wsum),
                    ("root_prior", prior), ("board", board)):
        np.save(os.path.join(out_dir, name + ".npy"), a)


def setup_nets(e, seed):
    e.net_init(0, seed + 100)
    e.net_init(1, seed + 101)
    e.set_inferer(0, K.INF_DUAL)
    e.set_inferer(1, K.INF_DUAL)


def cpu_reference_run(w, steps, warmup, threads=None, faithful=False):
    """One step = one pipeline() iteration (1 leaf evaluation at useful-work batch 1) of ONE game on the
    oracle, OpenMP over the host cores inside the conv loops."""
    lib = oracle_lib()
    ncores = len(os.sched_getaffinity(0))
    # small train batch: the oracle only reads batch row 0 at inference; keeps its memory modest
    e = lib.create(make_desc(w, 1, 0, 1234, batch=2))
    setup_nets(e, 1234)
    e.arena_begin(1, False)
    e.search_begin()  # root evaluation
    # "all the host threads it can use": try the full set and a few smaller teams (shared hosts / cgroup quotas
    # make the largest team the slowest one surprisingly often) and keep the fastest
    set_threads = lib.dll.azo_set_threads
    best_t, best_dt = None, None
    for t in sorted({ncores, max(1, ncores // 2), max(1, ncores // 4), max(1, ncores // 8)}, reverse=True):
        set_threads(t)
        e.search_run(1)
        t0 = time.perf_counter()
        e.search_run(1)
        d = time.perf_counter() - t0
        if best_dt is None or d < best_dt:
            best_t, best_dt = t, d
    set_threads(best_t)
    for _ in range(warmup):
        e.search_run(1)
    t0 = time.perf_counter()
    e.search_run(steps)
    dt = time.perf_counter() - t0
    c = e.counters()
    e.arena_finish()
    out = dict(value=steps / dt, seconds=dt, cores=best_t, nproc=ncores, evals=c["evals"])
    if faithful:
        # the reference's own cost per simulation: Inferencer.Infer pads every evaluation to ActionSpace samples (1 real
        # board + A-1 zero boards, meta.go:125-135,174-177) and runs the whole batch; timed here as ONE such evaluation
        A = w["size"] ** 2
        planes = np.zeros((A, 18 * A), np.float32)
        planes[0] = probe_planes(w, 1)[0]
        t0 = time.perf_counter()
        e.infer(0, planes)
        dtf = time.perf_counter() - t0
        out["faithful_value"] = 1.0 / dtf
        out["faithful_sample"] = "1 leaf evaluation padded to ActionSpace = %d samples as the reference does, %.1f s" % (A, dtf)
    e.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C3", choices=list(WORKLOADS))
    ap.add_argument("--games", type=int, default=0, help="override games per GPU (debug)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the dual.Train / gradient all-reduce block")
    ap.add_argument("--no-fast", action="store_true", help="skip the AZ_FLAG_FAST_TOWER arm")
    ap.add_argument("--fast-tower", action="store_true", help="run the main arm with AZ_FLAG_FAST_TOWER (experiments)")
    ap.add_argument("--cpu-steps", type=int, default=24)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the main arm's timed steps, write rank 0's search state for a fixed sample of games to "
                         "DIR/<name>.npy (identical inputs from run to run: compare two builds output for output)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    w = dict(WORKLOADS[args.workload])
    if args.games:
        w["n_games"] = args.games
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    warmup = max(args.warmup, 3)
    fpe = flops_per_eval(w)
    config = {"workload": "%s: %dx%d Go (wq) self-play, %d games/GPU, %d sims/move, %d-block x %d dual net, two random-init "
                          "nets" % (args.workload, w["size"], w["size"], w["n_games"], w["sims"], w["blocks"], w["k"]),
              "games_per_gpu": w["n_games"], "sims_per_move": w["sims"],
              "parallelism": "games sharded across %d GPU(s), no collective on the self-play path" % world,
              "step": "one MCTS wave = n_games simulations (select -> batched dual-net eval -> expand/backup)",
              "l2": "inputs larger than L2: activations ~%d MB per conv layer per agent vs 126 MB L2" %
                    (w["n_games"] // 2 * (w["size"] + 1) ** 2 * w["k"] * 4 * 2 // 2 ** 20),
              "flops_per_eval": fpe}

    if args.impl == "reference":
        if rank != 0:
            return 0
        # torchrun pins OMP_NUM_THREADS=1; the reference arm gets every host thread this process may run on
        # (set before libgomp loads); passive waiting keeps it sane on shared hosts
        if os.environ.get("OMP_NUM_THREADS", "1") == "1":
            os.environ["OMP_NUM_THREADS"] = str(len(os.sched_getaffinity(0)))
        os.environ.setdefault("OMP_WAIT_POLICY", "passive")
        r = cpu_reference_run(w, args.steps, warmup, faithful=True)
        line = {"impl": "reference", "metric": "mcts_sims_per_sec", "value": r["value"], "unit": "sims/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": warmup, "ms_per_step": 1e3 * r["seconds"] / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": dict(config, step="one simulation of one game (bounded sample of the GPU arm's wave)"),
                "faithful_sims_per_sec": r.get("faithful_value"), "faithful_sample": r.get("faithful_sample"),
                "cpu_baseline": {"value": r["value"], "unit": "sims/s", "cores": r["cores"], "nproc": r["nproc"], "threads": r["cores"],
                                 "kind": "port", "useful_work_sims_per_sec": r["value"], "faithful_sims_per_sec": r.get("faithful_value"),
                                 "sample": "oracle (C++ restatement of mcts+dualnet), 1 game, %d pipeline iterations, "
                                           "1 leaf eval each at useful-work batch 1 (the reference pads every eval to "
                                           "ActionSpace=%d samples, meta.go:125-135: divide by that for its faithful rate)"
                                           % (args.steps, w["size"] ** 2)},
                "e2e": {"value": r["value"], "unit": "sims/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "moves_per_sec": r["value"] / (w["sims"] + 1)}
        print(json.dumps(line))
        return 0

    dist = torch = None
    if world > 1:  # plumbing only: process group for barrier / max-over-ranks
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"  # the VERSION banner goes to stdout; stdout carries exactly one JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # stdout carries exactly one JSON line
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lib = K.load()
    ctx = dict(lib=lib, w=w, args=args, rank=rank, world=world, local_rank=local_rank, dist=dist, torch=torch, warmup=warmup)
    probe = probe_planes(w, 32)
    main_arm = selfplay_arm(ctx, flags=K.FLAG_FAST_TOWER if args.fast_tower else 0, do_e2e=not args.no_e2e, probe=probe,
                            do_train=not args.no_train, dump_dir=args.dump_outputs if rank == 0 else None)
    fast_arm = None
    if not args.no_fast and not args.fast_tower and world == 1:
        fast_arm = selfplay_arm(ctx, flags=K.FLAG_FAST_TOWER, do_e2e=False, probe=probe, do_train=False, steps=min(args.steps, 60))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return 0

    peaks, peak_src = load_peaks()
    roofline = roofline_of(main_arm.get("roof_arm") or main_arm, w, peaks, peak_src)
    if main_arm.get("roof_arm"):
        roofline["region"] = ("separate region of %d steps with CUDA events around every launch (plain launches); `value` is timed "
                              "over the captured wave graph without them" % main_arm["roof_arm"]["steps"])
    cpu_baseline = None
    if not args.no_cpu_baseline and world == 1:
        os.environ.setdefault("OMP_WAIT_POLICY", "passive")
        r = cpu_reference_run(w, args.cpu_steps, 1, faithful=True)
        cpu_baseline = {"value": r["value"], "unit": "sims/s", "cores": r["cores"], "nproc": r["nproc"], "threads": r["cores"],
                        "kind": "port",
                        "sample": "oracle, 1 game x %d pipeline iterations (1 leaf eval each, useful-work batch 1), %.1f s"
                                  % (args.cpu_steps, r["seconds"]),
                        "useful_work_sims_per_sec": r["value"],
                        "faithful_sims_per_sec": r.get("faithful_value"),
                        "faithful_sample": r.get("faithful_sample")}
    cnt, sims, evals = main_arm["cnt"], main_arm["cnt"]["sims"], main_arm["cnt"]["evals"]
    # tree-kernel traffic from COUNTED events (SURVEY §8d): 12 B per child scanned by Select (N, W, P), 8 B per level
    # (meta, first), 20 B per node created, 8 B read-modify-write per node backed up
    tree_bytes = 12 * cnt["select_children"] + 8 * cnt["select_levels"] + 20 * cnt["created"] + 8 * cnt["backup_nodes"]
    tree = {"counted_bytes_per_sim": tree_bytes / max(sims, 1), "select_children_per_sim": cnt["select_children"] / max(sims, 1),
            "levels_per_sim": cnt["select_levels"] / max(sims, 1), "nodes_created_per_eval": cnt["created"] / max(evals, 1),
            "null_results": cnt["null_results"],
            "note": "k_select + k_expand_backup take ~0.14 ms of a wave (profiles/r01_summary.md): latency-bound pointer chase, "
                    "not bandwidth-bound"}
    value = main_arm["value"]
    kind = main_arm["prof"].get("kernel_kind", -1)
    line = {"metric": "mcts_sims_per_sec", "value": value, "unit": "sims/s", "n_gpus": world, "steps": args.steps,
            "warmup": warmup, "ms_per_step": 1e3 * main_arm["dt_max"] / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32",
            "precision": KERNELS.get(kind, KERNELS[1])[2] + "; parity vs the fp32 oracle: tests/test_gpu_engine.py::"
                         "test_tc_tower_full_depth_c3 (1e-4 on policy and value)",
            "data": "synthetic", "config": config, "moves_per_sec": value / (w["sims"] + 1),
            "evals_per_sec": main_arm["tot_evals"] / main_arm["dt_max"],
            "tflops_algorithmic": main_arm["tot_evals"] / main_arm["dt_max"] * fpe / 1e12,
            "e2e": main_arm["e2e"], "gpu_launches": int(main_arm["tot_launch"]), "roofline": roofline, "tree": tree,
            "cpu_baseline": cpu_baseline, "clocks": main_arm["clocks"],
            "timing": "CUDA events on the engine's stream around exactly `steps` steps, barrier+synchronize both sides, max over ranks"
                      + (" (wave graph replayed; per-launch events in a second region, see roofline.region)" if main_arm.get("roof_arm") else "")}
    if main_arm.get("train") is not None:
        line["train"] = main_arm["train"]
    if fast_arm is not None:
        rf = roofline_of(fast_arm, w, peaks, peak_src)
        dp = float(np.abs(fast_arm["probe_out"][0] - main_arm["probe_out"][0]).max())
        dv = float(np.abs(fast_arm["probe_out"][1] - main_arm["probe_out"][1]).max())
        line["fast_tower"] = {"flag": "AZ_FLAG_FAST_TOWER (opt-in)", "value": fast_arm["value"], "unit": "sims/s",
                              "steps": fast_arm["steps"], "ms_per_step": 1e3 * fast_arm["dt_max"] / fast_arm["steps"],
                              "roofline": rf, "clocks": fast_arm["clocks"],
                              "max_abs_dpolicy_vs_default": dp, "max_abs_dvalue_vs_default": dv,
                              "probe": "%d synthetic 19x19 positions through both precision modes of THIS run's nets" % len(probe),
                              "note": "FP8 correction passes (E5M2 x E4M3): ~14.5-bit operands; within 1.3e-5 of the fp32 oracle "
                                      "on well-conditioned nets, up to 1.4e-4 on the reference's random init (gain > 1 per "
                                      "layer) — outside the 1e-4 bar, hence not the default"}
    print(json.dumps(line))
    return 0


def probe_planes(w, n):
    """Plausible WQEncoder planes for the precision probe (stones +-1 in the history planes, one to-move plane)."""
    rng = np.random.default_rng(77)
    hw = w["size"] ** 2
    x = np.zeros((n, 18, hw), np.float32)
    for b in range(n):
        for q in range(7):
            board = rng.choice([0.0, 1.0, -1.0], size=hw, p=[0.6, 0.2, 0.2]).astype(np.float32)
            x[b, q] = board
            x[b, 8 + q] = -board
        x[b, 16 if b % 2 == 0 else 17] = 1.0 if b % 2 == 0 else -1.0
    return x.reshape(n, -1)


def roofline_of(arm, w, peaks, peak_src):
    prof, evals = arm["prof"], arm["cnt"]["evals"]
    hw = w["size"] ** 2
    kind = prof.get("kernel_kind", -1)
    label, passes, _ = KERNELS.get(kind, KERNELS[1])
    if w["k"] < 128 and kind in (0, 1):
        label = "k_conv3x3_tc<%d,true,64> (fused residual-block conv, one CTA per 128 x %d tile, fp16 hi/lo 3-pass tcgen05)" % (2 * w["k"], 2 * w["k"])
    # dominant kernel: the fused 3x3 conv of one residual block (both branches, C -> 2C), one launch per block per agent.
    # Algorithmic FLOPs of all its launches in the timed region: every evaluated leaf passes through `blocks` of them
    conv_flops = 2 * 9 * w["k"] * (2 * w["k"]) * hw * evals * w["blocks"]
    conv_s = prof["conv_ms"] / 1e3
    achieved = conv_flops / conv_s / 1e12 if conv_s > 0 else None
    peak = peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops"))
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "conv_traffic.json")  # per-kernel dram bytes per launch from committed ncu --set full captures
    if os.path.exists(tp):
        try:
            ent = json.load(open(tp)).get("%s/%d" % (arm["workload"], kind))
            if ent:
                traffic, traffic_src = ent["dram_bytes_per_launch"], ent["source"]
        except Exception:
            pass
    pad = {19: 384.0 / 361.0, 9: 100.0 / 81.0}.get(w["size"], 1.0)
    return {"bound": "tensor", "kernel": label, "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
            "frac": (achieved / peak) if achieved else None,
            "peak_source": "%s bf16 dense, sustained (kernel timed inside a long step)" % peak_src,
            "traffic": traffic, "traffic_source": traffic_src, "launches_timed": prof["conv_launches"],
            "avg_launch_ms": prof["conv_ms"] / max(prof["conv_launches"], 1),
            "algorithmic_flops_per_launch": conv_flops / max(prof["conv_launches"], 1),
            "share_of_step": conv_s / arm["dt"],
            "tensor_passes_per_mac": passes,
            "executed_tflops_f16_equivalent": (achieved * passes * pad) if achieved else None,
            "note": "%g tensor-core passes (fp16-rate equivalents) per algorithmic MAC over %.3fx padded rows: the algorithmic "
                    "fraction of the bf16 peak tops out at %.3f" % (passes, pad, 1.0 / (passes * pad))}


def selfplay_arm(ctx, flags, do_e2e, probe, do_train, steps=None, dump_dir=None):
    """One engine, one precision mode: warm-up, the timed region of `steps` MCTS waves, optionally the end-to-end ply and
    the training / collective block, then the precision probe; the engine is closed before returning.  With `dump_dir`
    the search state after the first timed region is written there (dump_outputs)."""
    lib, w, args, rank, world, local_rank = ctx["lib"], ctx["w"], ctx["args"], ctx["rank"], ctx["world"], ctx["local_rank"]
    dist, torch, warmup = ctx["dist"], ctx["torch"], ctx["warmup"]
    steps = steps or args.steps
    e = lib.create(make_desc(w, w["n_games"], local_rank, 1000 + rank, flags=flags))
    setup_nets(e, 1000 + 10 * rank)
    n_games = w["n_games"]

    def barrier():
        e.counters()  # synchronises the engine's stream (all of this process's GPU work)
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize(local_rank)

    # step generator: waves continue across move boundaries
    state = {"in_search": False, "left": 0}
    e.arena_begin(n_games, False)

    def one_step():
        if not state["in_search"]:
            e.search_begin()          # root evaluation wave (1 eval per game)
            state["in_search"], state["left"] = True, w["sims"]
            return 0
        e.search_run(1)
        state["left"] -= 1
        if state["left"] == 0:
            e.search_end()
            state["in_search"] = False
        return 1

    for _ in range(warmup):
        one_step()

    def timed_region(mode=1, n=None):
        e.counters_reset()
        barrier()
        sampler = ClockSampler(local_rank)
        sampler.start()
        e.profile(mode)                      # records the start event on the engine's stream
        for _ in range(n or steps):
            one_step()
        prof = e.profile(False)              # stop event + synchronise: device time of exactly `steps` steps
        barrier()
        sampler.stop_flag = True
        return prof, sampler.summary(), e.counters()

    # A launch-bound small net (k_net_small, kernel_kind 5) is timed the way it runs in production — the captured wave
    # graph replayed, no events inside the wave (az_profile mode 2) — and the per-launch kernel times behind the roofline
    # come from a second, shorter region with the events on (plain launches).  Everywhere else the events cost nothing
    # measurable against millisecond kernels and one region serves both.
    e.profile(True)
    two_regions = e.profile(False)["kernel_kind"] == 5
    prof, clocks, cnt = timed_region(2 if two_regions else 1)
    if dump_dir:  # here, not after a re-measure: the dumped state is always warm-up + `steps` waves from the opening
        dump_outputs(e, n_games, dump_dir)
    bad = {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    if bad & set(clocks.get("reasons", [])) and world == 1:  # rejected: re-measure once (timing rules)
        prof, clocks2, cnt = timed_region(2 if two_regions else 1)
        clocks2["rejected_first_run"] = True
        clocks = clocks2
    roof_arm = None
    if two_regions:
        p2, _, c2 = timed_region(1, min(steps, 100))
        roof_arm = dict(prof=p2, cnt=c2, dt=p2["region_ms"] / 1e3, workload=args.workload, steps=min(steps, 100))
        prof = dict(prof, kernel_kind=p2["kernel_kind"])
    dt = prof["region_ms"] / 1e3
    tot = [dt, float(cnt["sims"]), float(cnt["evals"]), float(cnt["kernel_launches"])]
    dt_max = dt
    if dist is not None:
        tt = torch.tensor(tot, dtype=torch.float64, device="cuda:%d" % local_rank)
        mx = tt.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(tt, op=dist.ReduceOp.SUM)
        dt_max, tot = mx[0].item(), tt.tolist()
    out = dict(value=tot[1] / dt_max, dt=dt, dt_max=dt_max, tot_evals=tot[2], tot_launch=tot[3], prof=prof, clocks=clocks,
               cnt=cnt, steps=steps, e2e=None, train=None, workload=args.workload, roof_arm=roof_arm)

    # finish the ply in flight (untimed) and leave the arena
    if state["in_search"]:
        e.search_run(state["left"])
        e.search_end()
        state["in_search"] = False
    e.arena_finish()
    e.examples(clear=True)

    # ---- e2e: one full Arena.Play ply through az_arena_step, examples read back to host
    if do_e2e:
        e.arena_begin(n_games, True)
        barrier()
        t1 = time.perf_counter()
        e.arena_step()
        barrier()
        dt_e = time.perf_counter() - t1
        if dist is not None:
            te = torch.tensor([dt_e], dtype=torch.float64, device="cuda:%d" % local_rank)
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
            dt_e = te[0].item()
        e.arena_finish()
        e.examples(clear=True)
        d2h = n_games * (18 * w["size"] ** 2 + w["size"] ** 2 + 1 + 2) * 4 + 8
        out["e2e"] = {"value": world * n_games * w["sims"] / dt_e, "unit": "sims/s", "h2d_bytes_per_step": n_games * 4,
                      "d2h_bytes_per_step": d2h,
                      "step": "az_arena_step: one full ply (1 root eval + %d sims per game) + example read-back" % w["sims"],
                      "seconds": dt_e, "moves_per_sec": world * n_games / dt_e,
                      "note": "the path's inputs are the two nets' weights, uploaded once per epoch by az_net_set_params / "
                              "az_agent_set_inferer, not per ply; per ply the host sends the coin flips and receives the examples"}

    # ---- dual.Train at this workload's net and DefaultConf batch: one step (forward + backward + SGD), and at N > 1 the
    # fused gradient all-reduce + SGD kernel over NVLink peer memory (K8), the path's only exchange step
    if do_train:
        out["train"] = train_block(ctx, e, w)

    out["probe_out"] = e.infer(0, probe)
    e.close()
    return out


def train_block(ctx, e, w):
    rank, world, local_rank, dist, torch = ctx["rank"], ctx["world"], ctx["local_rank"], ctx["dist"], ctx["torch"]
    B, hw = w["batch"], w["size"] ** 2
    res = {"batch": B, "net": "%d-block x %d, %dx%d" % (w["blocks"], w["k"], w["size"], w["size"]),
           "params": int(e.param_count()[1])}
    try:
        if world > 1:
            uid = K.comm_unique_id(ctx["lib"])
            t = torch.tensor(list(uid), dtype=torch.uint8, device="cuda:%d" % local_rank)
            dist.broadcast(t, 0)
            e.comm_init(rank, world, bytes(t.cpu().tolist()))
            dist.barrier()
            ms, nbytes = e.comm_bench(1, 5)
            mt = torch.tensor([ms], dtype=torch.float64, device="cuda:%d" % local_rank)
            dist.all_reduce(mt, op=dist.ReduceOp.MAX)
            ms = mt.item()
            gbs = nbytes / (ms / 1e3) / 1e9
            res.update({"k8_kernel": "k_allreduce_sgd_p2p (reduce-scatter + SGD + all-gather over NVLink peer memory, one kernel)",
                        "k8_ms": ms, "nvlink_bytes_per_rank_per_direction": nbytes, "gbs_per_direction": gbs,
                        "peak_gbs_per_direction": 770.0, "frac": gbs / 770.0,
                        "peak_source": "measured peer copy, /opt/skills/guides/B200_PROFILING.md"})
        rng = np.random.default_rng(5 + rank)
        X = rng.choice([0.0, 1.0, -1.0], size=(B, 18 * hw)).astype(np.float32)
        Pi = np.zeros((B, hw + 1), np.float32)
        Pi[np.arange(B), rng.integers(0, hw + 1, B)] = 1
        V = rng.choice([-1.0, 1.0], B).astype(np.float32)
        e.train(1, X.copy(), Pi.copy(), V.copy(), 1, 1)  # warm-up: workspace allocation
        if dist is not None:
            dist.barrier()
        iters = 2
        t0 = time.perf_counter()
        costs = e.train(1, X.copy(), Pi.copy(), V.copy(), 1, iters)
        dt = (time.perf_counter() - t0) / iters
        if dist is not None:
            mt = torch.tensor([dt], dtype=torch.float64, device="cuda:%d" % local_rank)
            dist.all_reduce(mt, op=dist.ReduceOp.MAX)
            dt = mt.item()
        fwd = B * flops_per_eval(w)
        res.update({"step_ms": dt * 1e3, "step": "az_train, one batch of %d per rank: H2D batch copy + forward (BN train mode) + "
                    "backward + %s, host-synchronised" % (B, "fused all-reduce/SGD" if world > 1 else "SGD"),
                    "algorithmic_tflops": world * 3 * fwd / dt / 1e12, "cost": float(costs[-1])})
    except Exception as ex:  # the self-play line must survive a failure of the training block
        res["error"] = str(ex)[:300]
    return res


if __name__ == "__main__":
    sys.exit(main())
