#!/usr/bin/env python
"""Headline benchmark: Leduc transitions/sec of the fused NFSP rollout (env step + NFSP act + memories).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --steps K --warmup W --dump-outputs DIR  # the same, and what its last timed step computed -> DIR/*.npy
    python bench.py --impl reference --steps K --warmup W    # CPU arm: the REFERENCE's own Python (leduc.newenv +
                                                             # main.train + Agent.play + both memories) on all host cores

One "step" = one pass of the hot path over one batch: `rollout(T)` (T decisions for every game: observe,
remember, act with the eta-mixed nets, env.step, terminal observations, auto re-deal) followed by the
move of the staged records into both players' ring (M_RL) and reservoir (M_SL) memories.
Workload (BASELINE.json configs[4] per GPU == configs[2] scaled to 1M games): 2^20 games per GPU,
eta 0.1, epsilon 0.06, Glorot-initialised 30-64-3 nets, synthetic Philox deals.  Weak scaling: games
shard by global id with no data-path collective (SURVEY.md 8e).

Prints ONE JSON line (contract in the task statement).  `value` is device-timed with inputs resident in
HBM; `e2e` adds, per step, the pinned-host -> device copy of the four nets' weights, the sampling of a
256-row minibatch from all four memories and the device -> host read of those batches and the counters.
Outside the timed region one shard of the workload (65 536 games x 8 decisions, same seed / eta / epsilon /
nets) is replayed against the CPU oracle: `parity_checked`.
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GAMES_PER_GPU = 1 << 20
T_PER_CALL = 8
ENV_T_PER_CALL = 32  # env-only K1 beside the headline: transitions per game and launch (trace planes: 402 MB)
ETA, EPS, SEED = 0.1, 0.06, 1234
RL_CAP, SL_CAP = 1 << 25, 1 << 23  # records per player (16 B each): one step's records never wrap the ring
BATCH = 256
BYTES_PER_TRANSITION = 33.6  # SURVEY 8d cfg 3: state 16 + RL record 16 + eta * SL record 16
ENV_BYTES_PER_TRANSITION = 28.0  # SURVEY 8d cfg 2: state 16 + 12-byte trace record


KERNEL_OF_VARIANT = {"default": "rollout_states_kernel", "states": "rollout_states_kernel", "cuda": "rollout_kernel",
                     "tcgen05": "rollout_tc_kernel", "tcgen05_ws": "rollout_tq_kernel", "sorted": "rollout_sorted_kernel",
                     "pairs": "rollout_pairs_kernel"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md): NVML every 2 ms, nvidia-smi
    (one query per ~0.1 s) if NVML cannot be loaded."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag, self.source = index, [], False, "nvidia-smi"
        self.nvml = None
        try:
            import pynvml

            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(visible.split(",")[index]) if visible and visible.split(",")[index].isdigit() else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml, self.source = pynvml, "nvml"
        except Exception:
            self.nvml = None

    def _nvml_row(self):
        n = self.nvml
        mhz = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
        r = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle) if hasattr(n, "nvmlDeviceGetCurrentClocksEventReasons")
                else n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
        bits = (0x8, 0x40, 0x20, 0x4)  # HwSlowdown, HwThermalSlowdown, SwThermalSlowdown, SwPowerCap
        return [mhz, self.max_mhz] + ["Active" if r & b else "Not Active" for b in bits]

    def run(self):
        while not self.stop_flag:
            try:
                if self.nvml is not None:
                    self.rows.append(self._nvml_row())
                    time.sleep(0.002)
                    continue
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 6:
                    self.rows.append(f)
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.rows:
            return None
        sm = sorted(float(r[0]) for r in self.rows)
        reasons = [n for i, n in enumerate(self.NAMES) if any(str(r[2 + i]).lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "samples": len(self.rows), "source": self.source}


def cpu_rollout_rate(threads, games_per_thread, t_steps, reps):
    """Oracle port of the same workload on `threads` host threads (independent game shards)."""
    import torch

    from oracle import orc

    # Keras-default Glorot nets, same formula as the GPU arm's (agent.py:101-103,110-112); the product
    # package is deliberately not imported on this arm
    g = torch.Generator().manual_seed(SEED)
    wt = torch.zeros((4, 2179), dtype=torch.float32)
    l1, l2 = (6.0 / 94) ** 0.5, (6.0 / 67) ** 0.5
    for k in range(4):
        wt[k, :1920] = (torch.rand(1920, generator=g) * 2 - 1) * l1
        wt[k, 1984:2176] = (torch.rand(192, generator=g) * 2 - 1) * l2
    w = wt.numpy()
    nets = orc.Nets([dict(W1=w[k, :1920].reshape(30, 64), b1=w[k, 1920:1984], W2=w[k, 1984:2176].reshape(64, 3),
                          b2=w[k, 2176:]) for k in range(4)])
    eta_u, eps_u = orc.u32_frac(ETA), orc.u32_frac(EPS)
    batches = []
    for t in range(threads):
        b = orc.NfspBatch(games_per_thread, SEED, game0=t * games_per_thread)
        b.reset(0, eta_u)
        batches.append(b)
    cap = 3 * games_per_thread * t_steps + 8

    def work(b, step0):
        b.rollout_act(step0, t_steps, nets, eta_u, eps_u, rec_cap=cap)

    def one(step0):
        ths = [threading.Thread(target=work, args=(b, step0)) for b in batches]
        t0 = time.perf_counter()
        for th in ths:
            th.start()
        for th in ths:
            th.join()
        return time.perf_counter() - t0

    one(1)  # warm-up
    times = [one(1 + (i + 1) * t_steps) for i in range(reps)]
    trans = threads * games_per_thread * t_steps
    return trans, times


REF_HANDS_PER_STEP = 1500  # hands per process and step of the reference arm (about 0.3 s of its Python per step)


def reference_rates(procs, hands, kind="nfsp", reps=1):
    """The reference's own code (oracle/ref_timing.py: /root/reference, or the verbatim copy under baseline/_ref that
    travels to the GPU box) on `procs` processes; returns the list of per-repetition results."""
    from oracle import ref_timing

    return [ref_timing.run(kind, hands, procs) for _ in range(reps)]


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import ref_timing

    cores = max(1, os.cpu_count() or 1)
    if ref_timing.reference_root() is None:
        print(json.dumps({"impl": "reference", "unavailable": "no reference tree (neither /root/reference nor baseline/_ref)"}))
        return
    runs = reference_rates(cores, REF_HANDS_PER_STEP, "nfsp", args.warmup + args.steps)[args.warmup:]
    trans = sum(r["transitions"] for r in runs)
    secs = sum(r["seconds"] for r in runs)
    value = trans / secs
    sample = ("%d processes x %d hands per step of the reference's own leduc.newenv.Env + main.train + Agent.play + "
              "ReplayBuffer / ReservoirBuffer (Keras nets replaced by np.random.rand(1,1,3): an upper bound of its rate)"
              % (cores, REF_HANDS_PER_STEP))
    line = {"impl": "reference", "metric": "leduc_transitions_per_sec", "value": value, "unit": "transitions/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / len(runs),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "nfsp_rollout on the CPU: " + sample, "hands_per_step": cores * REF_HANDS_PER_STEP,
                       "transitions_per_step": trans / len(runs), "cpu": runs[0]["cpu"],
                       "baseline_config": "BASELINE.json configs[0] driver (reference path), NFSP loop of configs[2]"},
            "cpu_baseline": {"value": value, "unit": "transitions/s", "cores": cores, "kind": "reference", "sample": sample,
                             "cpu": runs[0]["cpu"]},
            "e2e": {"value": value, "unit": "transitions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def parity_check(nfsp_b200, dev, game0):
    """One shard of the benchmarked workload against the CPU oracle, outside every timed region: 65 536 games x 8
    decisions with the bench's seed, eta, epsilon and nets (debug launch, teacher-forced on the kernel's own score
    vectors) -- trace planes and record multisets bit for bit, score vectors within 1e-5 -- and the production launch
    from the same start must leave the same game words, counters and records."""
    import numpy as np
    import torch

    from oracle import orc

    n, steps = 1 << 16, T_PER_CALL
    mk = lambda: nfsp_b200.SelfPlay(n, seed=SEED, game0=game0, device=dev, eta=ETA, epsilon=EPS, rl_capacity=1 << 21,  # noqa: E731
                                    sl_capacity=1 << 18, max_steps_per_call=steps)
    sp = mk()
    out = sp.rollout(steps, insert=False, debug=True)
    rl, sl = sp.staged()
    vec = out["vec"].cpu().numpy()
    tr = out["raw"].cpu().numpy().view(np.uint32)
    w = sp.weights.cpu().numpy()
    b = orc.NfspBatch(n, SEED, game0=game0)
    b.reset(0, orc.u32_frac(ETA))
    ref = b.rollout_act(1, steps, orc.Nets([nfsp_b200.split_net(w[k]) for k in range(4)]), orc.u32_frac(ETA),
                        orc.u32_frac(EPS), forced_vec=vec)
    canon = lambda a: (lambda v: v[np.lexsort(v.T[::-1])])(np.ascontiguousarray(a).view(np.uint32).reshape(-1, 4))  # noqa: E731
    ok = (np.array_equal(tr[0], ref["trace"]["obs"]) and np.array_equal(tr[1].view(np.float32), ref["trace"]["reward"])
          and np.array_equal(tr[2], ref["trace"]["misc"]))
    err = float(np.abs(vec - ref["vec"]).max())
    ok = ok and err <= 1e-5
    for p in range(2):
        ok = ok and np.array_equal(canon(rl[p]), canon(ref["rl"][p])) and np.array_equal(canon(sl[p]), canon(ref["sl"][p]))
    prod = mk()
    prod.rollout(steps, insert=False)
    prl, psl = prod.staged()
    ok = ok and np.array_equal(prod.env.state_words().cpu().numpy(), sp.env.state_words().cpu().numpy())
    ok = ok and prod.read_stats() == sp.read_stats()
    for p in range(2):
        ok = ok and np.array_equal(canon(prl[p]), canon(rl[p])) and np.array_equal(canon(psl[p]), canon(sl[p]))
    return bool(ok), {"games": n, "decisions": steps, "game0": int(game0), "max_abs_score_error": err,
                      "what": "trace planes, RL/SL record multisets, counters and game words vs oracle/leduc_oracle.c; "
                              "debug and production launch"}


DUMP_RL_ROWS, DUMP_SL_ROWS, DUMP_GAMES, DUMP_SEED = 1 << 18, 1 << 17, 1 << 18, 7  # 42 MB of float64 in all
DUMP_MAX_BYTES = 64 << 20


def mark_last_step(sp):
    """Called before the last timed step, outside its timer.  Notes where the step's tickets start in every memory, and
    fills the SL staging areas with -1 (no record has that first word: an observation is a 30-bit mask), because the
    step's insert launch clears the per-segment counts that would otherwise tell its staged records from older ones."""
    for st in sp.stage_sl:
        st.fill_(-1)
    return {"rl": [int(m.total.item()) for m in sp.rl], "sl": [int(m.total.item()) for m in sp.sl]}


def canonical_sample(recs, rows, seed):
    """int32 [m, 4] records -> a host array of at most `rows` of them, independent of the order the kernels appended them
    in: sorted by their four words, then a fixed, seeded choice of positions."""
    import torch

    order = torch.arange(recs.shape[0], device=recs.device)
    for k in (3, 2, 1, 0):  # least significant word first: stable passes give the lexicographic order
        key = recs[order, k].to(torch.int64) & 0xFFFFFFFF
        order = order[torch.sort(key, stable=True).indices]
    if order.numel() > rows:
        pick = torch.randperm(order.numel(), generator=torch.Generator().manual_seed(seed))[:rows].sort().values
        order = order[pick.to(order.device)]
    return recs[order].cpu().numpy()


def dump_outputs(sp, mark, out_dir):
    """What the last timed step handed its caller, as float64 .npy files (every field is exact in float64):
      rl_records_p{0,1}  [rows, 7] s, s2, r, a, t, player, flags of the RL records the step wrote into player p's ring
      sl_records_p{0,1}  [rows, 4] s, a[0..2] of the SL records the step moved into player p's reservoir
      game_words         [DUMP_GAMES, 3] game id, low and high 32 bits of its packed state after the step
      stats              [16] the rollout counters (cumulative since the SelfPlay was built)
    Records are sorted and sampled by canonical_sample: the order in which warps append them changes from run to run,
    the set does not.  Which of the SL records a reservoir keeps depends on that order, so the reservoirs' slots are not
    dumped."""
    import numpy as np
    import torch

    from nfsp_b200.batched import RL_DT, SL_DT

    os.makedirs(out_dir, exist_ok=True)
    out = {}
    for p in range(2):
        ring = sp.rl[p]
        slots = torch.arange(mark["rl"][p], int(ring.total.item()), device=ring.store.device) % ring.capacity
        r = canonical_sample(ring.data[slots], DUMP_RL_ROWS, DUMP_SEED + p).view(RL_DT).reshape(-1)
        out["rl_records_p%d" % p] = np.stack([r[f].astype(np.float64) for f in RL_DT.names], axis=1)
        st = sp.stage_sl[p]
        staged = st[st[:, 0] != -1]
        if staged.shape[0] != int(sp.sl[p].total.item()) - mark["sl"][p]:
            raise RuntimeError("staged SL records of the last step do not match the reservoir's ticket count")
        s = canonical_sample(staged, DUMP_SL_ROWS, DUMP_SEED + 2 + p).view(SL_DT).reshape(-1)
        out["sl_records_p%d" % p] = np.concatenate([s["s"].astype(np.float64)[:, None], s["a"].astype(np.float64)], axis=1)
    words = sp.env.state_words().cpu().numpy().view(np.uint32).reshape(-1, 2)
    games = np.sort(np.random.default_rng(DUMP_SEED).choice(len(words), min(DUMP_GAMES, len(words)), replace=False))
    out["game_words"] = np.concatenate([games[:, None], words[games]], axis=1).astype(np.float64)
    out["stats"] = sp.stats.cpu().numpy().astype(np.float64)
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError("dump of %d bytes exceeds %d" % (total, DUMP_MAX_BYTES))
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def workload_config():
    return {"workload": "nfsp_rollout: %d games/GPU x %d decisions per step, eta=%.2f eps=%.2f, 4 acting nets 30-64-3, "
                        "ring %d + reservoir %d records per player, sample %d" %
                        (GAMES_PER_GPU, T_PER_CALL, ETA, EPS, RL_CAP, SL_CAP, BATCH),
            "games_per_gpu": GAMES_PER_GPU, "decisions_per_step": T_PER_CALL, "l2": "flushed between timed steps",
            "memories": "both reservoirs are filled by untimed steps first: every timed insert is Algorithm R's random replacement",
            "records": "RL records written straight into the rings by the rollout kernel (direct_rings), SL records "
                       "staged and moved into the reservoirs by one insert launch",
            "nets": "default variant: the four nets are evaluated on the 702 decision states of the game (same operations as the "
                    "per-decision kernel) and the decisions read that table; the table is rebuilt from the "
                    "weights inside every timed step.  extra.other_variants.cuda is the per-decision evaluation",
            "baseline_config": "BASELINE.json configs[4] per GPU (configs[2] at 1M games)"}


def buffer_kernels(nfsp_b200, dev, ev, n_rec=1 << 23):
    """K3/K4/K5 beside the headline (SURVEY 8d cfg 4): insert batches of 2^23 staged records into a 2^24-slot
    ring / reservoir (HBM streaming / scatter), and the 256-row sample+gather (latency)."""
    import torch

    hbm, _ = peaks()
    recs = torch.randint(0, 1 << 30, (n_rec, 4), dtype=torch.int32, device=dev)
    out = {}
    ring = nfsp_b200.DeviceRing(1 << 24, 1, dev)
    res = nfsp_b200.DeviceReservoir(1 << 24, 2, dev)
    for name, mem, bytes_per in (("ring_insert", ring, 32.0), ("reservoir_insert", res, 40.0)):
        ms = []
        for k in range(8):
            cnt = torch.tensor([n_rec], dtype=torch.int32, device=dev)
            a, b = ev(), ev()
            a.record()
            mem.insert(recs, cnt)
            b.record()
            b.synchronize()
            if k >= 3:
                ms.append(a.elapsed_time(b))
        t = sum(ms) / len(ms)
        gbs = n_rec * bytes_per / (t * 1e-3) / 1e9
        out[name] = {"records": n_rec, "ms": t, "records_per_sec": n_rec / (t * 1e-3), "achieved_gbs": gbs,
                     "algorithmic_bytes_per_record": bytes_per, "frac_of_hbm_peak": gbs / hbm}
    # SURVEY 8d cfg 4 as stated: the 2 000 000-slot reservoir (stamps + payload stay in the 126 MB L2), batches of 2^20
    res2m = nfsp_b200.DeviceReservoir(2_000_000, 3, dev)
    n_small = 1 << 20
    ms = []
    for k in range(11):
        cnt = torch.tensor([n_small], dtype=torch.int32, device=dev)
        a, b = ev(), ev()
        a.record()
        res2m.insert(recs[:n_small], cnt)
        b.record()
        b.synchronize()
        if k >= 3:
            ms.append(a.elapsed_time(b))
    t = sum(ms) / len(ms)
    out["reservoir_insert_2M_slots"] = {"records": n_small, "ms": t, "records_per_sec": n_small / (t * 1e-3),
                                        "achieved_gbs": n_small * 40.0 / (t * 1e-3) / 1e9,
                                        "frac_of_hbm_peak": n_small * 40.0 / (t * 1e-3) / 1e9 / hbm,
                                        "note": "tickets 3M..11M into 2M slots: 18-66% of the records are accepted"}
    ms = []
    for k in range(13):
        a, b = ev(), ev()
        a.record()
        ring.sample(BATCH)
        res.sample(BATCH)
        b.record()
        b.synchronize()
        if k >= 3:
            ms.append(a.elapsed_time(b))
    out["sample_256_rl_plus_sl_us"] = 1e3 * sum(ms) / len(ms)
    return out


def run_gpu(args):
    import torch
    import torch.distributed as dist

    import nfsp_b200
    from nfsp_b200 import sharding

    rank, world, local = sharding.env_rank_world()
    if args.gpus > 1 and world == 1:
        raise SystemExit("launch with torch.distributed.run for --gpus > 1")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    game0, n = sharding.shard_games(GAMES_PER_GPU * world, rank, world)
    sp = nfsp_b200.SelfPlay(n, seed=SEED, game0=game0, device=dev, eta=ETA, epsilon=EPS, rl_capacity=RL_CAP,
                            sl_capacity=SL_CAP, max_steps_per_call=T_PER_CALL, variant=args.variant,
                            direct_rings=args.variant in ("default", "states", "cuda", "pairs"))
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    w_host = sp.weights.cpu().pin_memory()
    stats_host = torch.empty(sp.stats.shape, dtype=sp.stats.dtype).pin_memory()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731

    def timed_steps(k, e2e):
        gc.collect()
        gc.disable()  # a collector pause inside a host-driven step shows up as a straggler rank (max over ranks)
        try:
            return _timed_steps(k, e2e)
        finally:
            gc.enable()

    def _timed_steps(k, e2e):
        tot_ms, ker_ms = 0.0, 0.0
        for _ in range(k):
            flush_buf.zero_()  # L2 flush, outside the timed events
            a, b, c = ev(), ev(), ev()
            a.record()
            # e2e: pinned host -> device copy of the four nets and the rebuild of the kernels' weight image, in the same
            # library call that launches the rollout
            # value: the nets are resident in HBM; everything the kernels derive from them -- the weight images and, for the
            # default variant, the table of the nets' outputs on the 702 decision states -- is rebuilt from them inside the
            # timed region of EVERY step (as after a learner update): no step runs on outputs computed before its timer
            sp.rollout(T_PER_CALL, insert=False, weights_host=w_host if e2e else None, refresh_weights=not e2e)
            b.record()
            sp.flush()
            if e2e:  # the learner's four minibatches and the counters come back to the host in ONE slab, one copy
                sp.sample_minibatches(BATCH, to_host=True, with_stats=True)
            c.record()
            c.synchronize()
            tot_ms += a.elapsed_time(c)
            ker_ms += a.elapsed_time(b)
        return tot_ms, ker_ms

    # steady state of the memories before anything is timed: both reservoirs full, so that every timed insert is
    # Algorithm R's random replacement (the expensive regime: ~26 us per step while a reservoir still fills by appending,
    # ~45 us once it replaces, profiles/time_flush.py); value and e2e are then measured in the same regime
    prefill = 0
    while min(int(m.total.item()) for m in sp.sl) < SL_CAP and prefill < 200:
        sp.rollout(T_PER_CALL)
        prefill += 1
    timed_steps(args.warmup, False)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    if args.dump_outputs and rank == 0:  # every step ends in a synchronise: timing the last one on its own changes nothing
        tot_ms, ker_ms = timed_steps(args.steps - 1, False)
        mark = mark_last_step(sp)
        last_tot, last_ker = timed_steps(1, False)
        tot_ms, ker_ms = tot_ms + last_tot, ker_ms + last_ker
        dump_outputs(sp, mark, args.dump_outputs)  # before the e2e steps write into the same memories
    else:
        tot_ms, ker_ms = timed_steps(args.steps, False)
    barrier()
    t_e2e, _ = timed_steps(max(1, min(args.warmup, 2)), True)  # e2e warm-up (pinned buffers, sample kernels)
    barrier()
    e2e_ms, _ = timed_steps(args.steps, True)
    barrier()
    sampler.stop_flag = True
    tot_ms = sharding.max_over_ranks(tot_ms, dev)
    e2e_ms = sharding.max_over_ranks(e2e_ms, dev)
    trans_all = GAMES_PER_GPU * world * T_PER_CALL * args.steps
    value = trans_all / (tot_ms * 1e-3)
    e2e_value = trans_all / (e2e_ms * 1e-3)
    st = sharding.allreduce_stats(sp.stats)

    # learner beside it (SURVEY 8 f-1; BASELINE configs[4]): update_strategy() of both agents = 8 SGD steps of the
    # four nets, each with ONE all-reduce of the flat gradient+stats buffer (NCCL when world > 1)
    from nfsp_b200.learner import Learner

    learner = Learner(sp, cfg=nfsp_b200.load_config(None))
    for _ in range(2):
        learner.update()
    barrier()
    a, b = ev(), ev()
    a.record()
    for _ in range(10):  # device time of an update: nothing read back in between (as in the training loop)
        learner.update(sync=False)
    b.record()
    b.synchronize()
    learner_ms = sharding.max_over_ranks(a.elapsed_time(b) / 10, dev)
    lstats = learner.update()  # one synchronised update for the statistics
    # the full self-play iteration of BASELINE configs[4]: rollout(8) + memory inserts + update_strategy() of both agents
    # (with its all-reduces when world > 1), nothing read back between iterations
    barrier()
    a, b = ev(), ev()
    a.record()
    for _ in range(5):
        sp.rollout(T_PER_CALL)
        learner.update(sync=False)
    b.record()
    b.synchronize()
    train_ms = sharding.max_over_ranks(a.elapsed_time(b) / 5, dev)
    # the same iteration with the update beside the next rollout (learner.PipelinedTrainer: acting nets one update behind)
    from nfsp_b200.learner import PipelinedTrainer

    pipe_ms = None
    if learner.one_launch:  # needs the one-launch fit (with several GPUs: peer memory); every rank takes the same branch
        trainer = PipelinedTrainer(sp, learner)
        for _ in range(3):
            trainer.step(T_PER_CALL)
        barrier()
        a, b = ev(), ev()
        a.record()
        for _ in range(10):
            trainer.step(T_PER_CALL)
        b.record()
        b.synchronize()
        pipe_ms = sharding.max_over_ranks(a.elapsed_time(b) / 10, dev)
        trainer.finish()
        torch.cuda.synchronize()

    # after all those updates every rank must hold bit-identical nets (the gradient sum is taken in rank order everywhere)
    chk = sp.weights.view(torch.int32).to(torch.int64).sum().reshape(1)
    if world > 1:
        lo, hi = chk.clone(), chk.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        weights_same = bool(int(lo.item()) == int(hi.item()))
    else:
        weights_same = True
    weights_same = weights_same and bool(torch.isfinite(sp.weights).all().item())

    # env-only K1 (BASELINE configs[1]) beside it, same games count, trace planes written
    env = nfsp_b200.BatchedNfspEnv(n, seed=SEED, game0=game0, device=dev)
    env.reset()
    tr = torch.empty((3, ENV_T_PER_CALL, n), dtype=torch.int32, device=dev)
    from nfsp_b200.batched import _ptr, _stream, check, lib

    def env_step():
        check(lib().nfsp_env_step(env._h, None, None, ENV_T_PER_CALL, 1, ETA, _ptr(tr), _stream(dev)))

    for _ in range(3):
        env_step()
    env_ms = 0.0
    for _ in range(args.steps):
        flush_buf.zero_()
        a, b = ev(), ev()
        a.record()
        env_step()
        b.record()
        b.synchronize()
        env_ms += a.elapsed_time(b)
    env_rate = n * ENV_T_PER_CALL * args.steps / (env_ms * 1e-3)

    # the README's env (leduc/env.py, ENV_LEGACY) beside it: README iterations of 2 transitions, records written
    leg = nfsp_b200.BatchedLegacyEnv(n, seed=SEED, game0=game0, device=dev)
    leg.reset()
    leg_iters = ENV_T_PER_CALL // 2  # as many transitions per game and launch as the NFSP env kernel above
    rec = torch.empty((3, leg_iters, n, 2), dtype=torch.int32, device=dev)

    def legacy_step():
        check(lib().nfsp_legacy_rollout(leg._h, None, leg_iters, _ptr(rec), _stream(dev)))

    for _ in range(3):
        legacy_step()
    leg_ms = 0.0
    for _ in range(args.steps):
        flush_buf.zero_()
        a, b = ev(), ev()
        a.record()
        legacy_step()
        b.record()
        b.synchronize()
        leg_ms += a.elapsed_time(b)
    legacy_rate = 2 * n * leg_iters * args.steps / (leg_ms * 1e-3)
    del rec, leg

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    buffers = buffer_kernels(nfsp_b200, dev, ev) if world == 1 else None
    # the other variants of the rollout kernel, kernel only, for the record
    others = {}
    for other in ("states", "cuda", "pairs", "sorted", "tcgen05", "tcgen05_ws"):
        spo = nfsp_b200.SelfPlay(n, seed=SEED, game0=game0, device=dev, eta=ETA, epsilon=EPS, rl_capacity=1 << 16,
                                 sl_capacity=1 << 16, max_steps_per_call=T_PER_CALL, variant=other)
        other_ms = 0.0
        for k in range(3 + args.steps):
            flush_buf.zero_()
            a, b = ev(), ev()
            a.record()
            spo.rollout(T_PER_CALL, insert=False)
            b.record()
            b.synchronize()
            spo.counts.zero_()
            if k >= 3:
                other_ms += a.elapsed_time(b)
        others[other] = {"kernel_transitions_per_sec": n * T_PER_CALL * args.steps / (other_ms * 1e-3),
                         "kernel_ms_per_launch": other_ms / args.steps}
        del spo
    # BASELINE configs[2] + configs[3] as stated: 65 536 parallel games, ring of 200 000 + reservoir of 2 000 000 records per
    # player, rollout(8) + the move of the records into the memories (a launch laps the ring: staged path) + 256-row sample
    def time_64k(rl_cap, direct):
        s64 = nfsp_b200.SelfPlay(1 << 16, seed=SEED, device=dev, eta=ETA, epsilon=EPS, rl_capacity=rl_cap,
                                 sl_capacity=2000000, max_steps_per_call=T_PER_CALL, direct_rings=direct)
        ms, ms_s = 0.0, 0.0
        for k in range(3 + args.steps):
            a, b, c = ev(), ev(), ev()
            a.record()
            s64.rollout(T_PER_CALL)
            b.record()
            s64.sample_minibatches(BATCH)
            c.record()
            c.synchronize()
            if k >= 3:
                ms += a.elapsed_time(b)
                ms_s += b.elapsed_time(c)
        return ms, ms_s

    ms64, ms64s = time_64k(200000, False)
    rate64 = (1 << 16) * T_PER_CALL * args.steps / (ms64 * 1e-3)
    # the same with rings one launch cannot lap (2 * 65536 * 8 <= 2^21): the rollout kernel writes them in place
    ms64d, _ = time_64k(1 << 21, True)
    rate64d = (1 << 16) * T_PER_CALL * args.steps / (ms64d * 1e-3)
    hbm, which = peaks()
    # the rollout kernel alone: CUDA events around its launch (for the default variant the timed steps' events also cover the
    # two small launches that rebuild the images, so its kernel-only figure comes from the per-variant loop above)
    if args.variant in ("default", "states"):
        ker_ms = others["states"]["kernel_ms_per_launch"] * args.steps
    kernel_rate = n * T_PER_CALL * args.steps / (ker_ms * 1e-3)
    achieved = kernel_rate * BYTES_PER_TRANSITION / 1e9
    roofline = {"bound": "hbm", "kernel": KERNEL_OF_VARIANT[args.variant], "achieved": achieved, "peak": hbm, "unit": "GB/s",
                "frac": achieved / hbm, "traffic": None, "peak_source": which,
                "algorithmic_bytes_per_transition": BYTES_PER_TRANSITION,
                "kernel_ms_per_launch": ker_ms / args.steps,
                "kernel_ms_note": "CUDA events around the rollout kernel's launch alone, L2 flushed before each launch"}
    if args.variant not in ("default", "states"):
        # what a dense 30x64 + 64x3 evaluation per decision would cost; the kernel's first layer is two row adds, not 1 920 MACs
        roofline["dense_equivalent_tflops"] = kernel_rate * 4224 / 1e12
    traffic_file = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(traffic_file):
        tf = json.load(open(traffic_file))
        if args.variant in ("default", "states"):
            roofline["traffic"] = tf.get("rollout_states_kernel_bytes_per_launch")
            if "rollout_states_kernel_ncu" in tf:
                # what bounds the kernel (ncu, not measured in this run): the game logic, Philox and the record append are
                # integer instructions on the ALU pipe; DRAM carries the records and the game words only
                roofline["limiter"] = "instruction issue on the integer ALU pipe, not HBM"
                roofline["ncu"] = tf["rollout_states_kernel_ncu"]
        elif args.variant == "cuda":
            roofline["traffic"] = tf.get("rollout_kernel_bytes_per_launch")
            if "rollout_kernel_ncu" in tf:
                # each decision has to bring 2 x 256 B of first-layer rows and 768 B of second-layer weights from shared
                # memory into registers
                roofline["limiter"] = "shared memory -> register bandwidth (LDS.128 instructions), not HBM"
                roofline["ncu"] = tf["rollout_kernel_ncu"]
    cpu, cpu_extra = None, {}
    if world == 1:
        cores = max(1, os.cpu_count() or 1)
        try:  # the reference's own Python (a reported baseline, never the product): NFSP loop on all cores and on one core,
            # and BASELINE configs[0] -- leduc.env.Env under the README driver, 100 000 hands -- on one core and on all cores
            r_all = reference_rates(cores, 3000, "nfsp")[0]
            cpu = {"value": r_all["transitions_per_sec"], "unit": "transitions/s", "cores": cores, "kind": "reference",
                   "cpu": r_all["cpu"],
                   "sample": "%d processes x 3000 hands: the reference's leduc.newenv.Env + main.train + Agent.play + both memories, "
                             "Keras predict replaced by np.random.rand(1,1,3) (upper bound of its rate)" % cores}
            r_one = reference_rates(1, 12000, "nfsp")[0]
            l_one = reference_rates(1, 100000, "legacy")[0]
            l_all = reference_rates(cores, max(1, 100000 // cores), "legacy")[0]
            cpu_extra["reference_nfsp_1core"] = {"transitions_per_sec": r_one["transitions_per_sec"], "hands": 12000}
            cpu_extra["reference_config1_env_100k_hands"] = {
                "what": "BASELINE configs[0]: leduc.env.Env, README driver (reset; step(a0,0); step(a1,1); get_new_state x2), uniform-random actions",
                "one_core": {"transitions_per_sec": l_one["transitions_per_sec"], "hands_per_sec": l_one["hands_per_sec"],
                             "seconds": l_one["seconds"], "hands": 100000},
                "all_cores": {"transitions_per_sec": l_all["transitions_per_sec"], "hands_per_sec": l_all["hands_per_sec"],
                              "seconds": l_all["seconds"], "processes": cores, "hands_per_process": l_all["hands_per_proc"]},
                "cpu": l_one["cpu"]}
        except Exception as e:
            cpu = {"value": None, "unit": "transitions/s", "cores": cores, "kind": "reference", "sample": "failed: %r" % (e,)}
        try:
            trans, times = cpu_rollout_rate(1, 65536, T_PER_CALL, 3)
            cpu_extra["port_1thread"] = {"transitions_per_sec": trans * len(times) / sum(times), "kind": "port",
                                         "sample": "65536 games x %d decisions x %d passes, oracle/leduc_oracle.c, 1 thread" % (T_PER_CALL, len(times))}
        except Exception as e:
            cpu_extra["port_1thread"] = {"transitions_per_sec": None, "sample": "failed: %r" % (e,)}
    parity_ok, parity_info = parity_check(nfsp_b200, dev, game0)
    gpu_trans = GAMES_PER_GPU * world * T_PER_CALL
    training = {"what": "rollout(8) + memory inserts + Learner.update(sync=False) per iteration; gradients of the 8 SGD steps "
                        "exchanged inside the fit kernel over peer memory when n_gpus > 1",
                "sequential_ms": train_ms, "sequential_transitions_per_sec": gpu_trans / (train_ms * 1e-3),
                "pipelined_ms": pipe_ms, "pipelined_transitions_per_sec": (gpu_trans / (pipe_ms * 1e-3)) if pipe_ms else None,
                "learner_update_ms": learner_ms, "gradient_exchange": "peer memory" if getattr(learner, "_peers", None) is not None else ("nccl" if world > 1 else "none")}
    configs = [
        {"config": "BASELINE configs[1]: batched Leduc env, %d games, uniform-random actions, env kernel only" % n,
         "kernel": "nfsp_step_fsm_kernel", "transitions_per_sec": env_rate,
         "frac_of_hbm_peak": env_rate * ENV_BYTES_PER_TRANSITION / 1e9 / hbm,
         "moved_frac_of_hbm_peak": env_rate * (12.0 + 16.0 / ENV_T_PER_CALL) / 1e9 / hbm},
        {"config": "BASELINE configs[2]+[3]: NFSP rollout, 65536 games, eta 0.1, ring 200000 + reservoir 2000000 per player, insert + 256-batch sample per step",
         "transitions_per_sec": rate64, "ms_per_step": ms64 / args.steps, "sample_us": 1e3 * ms64s / args.steps,
         "note": "one launch of 8 decisions laps a 200000-record ring: staged records + insert launch"},
        {"config": "the same 65536 games with rings of 2^21 records (a launch cannot lap them: RL records written in place)",
         "transitions_per_sec": rate64d, "ms_per_step": ms64d / args.steps},
        {"config": "BASELINE configs[4] per GPU: the headline line", "transitions_per_sec": value / world},
    ]
    h2d = int(w_host.numel() * 4)
    d2h = int(2 * BATCH * (30 + 3 + 1 + 30 + 1) * 4 + 2 * BATCH * 33 * 4 + sp.stats.numel() * 8)
    line = {"metric": "leduc_transitions_per_sec", "value": value, "unit": "transitions/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": tot_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(),
            "clocks": sampler.summary(),
            "e2e": {"value": e2e_value, "unit": "transitions/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms / args.steps},
            # per step: pack_images_kernel + states_pack_kernel (the nets' images and state table, rebuilt every step),
            # rollout_states_kernel (records into the rings in place), insert_kernel (both reservoirs)
            "gpu_launches": (4 if args.variant in ("default", "states") else 3) * args.steps,
            "roofline": roofline, "cpu_baseline": cpu,
            # the same workload with the nets evaluated at every decision (variant "cuda", the default until the state table):
            # the rollout kernel alone, same launch shape -- for readers who want the figure without the table
            "per_decision_forward": dict(others.get("cuda", {}), kernel="rollout_kernel",
                                         note="python bench.py --variant cuda runs the whole line on it"),
            "parity_checked": parity_ok, "parity": parity_info,
            # the iteration that communicates (BASELINE configs[4]): rollout + memories + update_strategy() of both agents
            "training_step": training, "weights_identical_on_all_ranks": weights_same,
            "configs": configs,
            "extra": {"cpu": cpu_extra, "env_only": {"kernel": "nfsp_step_fsm_kernel", "transitions_per_sec": env_rate,
                                   "achieved_gbs": env_rate * ENV_BYTES_PER_TRANSITION / 1e9,
                                   "frac_of_hbm_peak": env_rate * ENV_BYTES_PER_TRANSITION / 1e9 / hbm,
                                   "algorithmic_bytes_per_transition": ENV_BYTES_PER_TRANSITION,
                                   "transitions_per_launch": n * ENV_T_PER_CALL,
                                   # what the kernel really moves: the 16-byte state word once per launch, 12 bytes of trace per transition
                                   "moved_bytes_per_transition": 12.0 + 16.0 / ENV_T_PER_CALL,
                                   "moved_gbs": env_rate * (12.0 + 16.0 / ENV_T_PER_CALL) / 1e9,
                                   "moved_frac_of_hbm_peak": env_rate * (12.0 + 16.0 / ENV_T_PER_CALL) / 1e9 / hbm},
                      "env_only_legacy": {"kernel": "legacy_rollout_kernel", "transitions_per_sec": legacy_rate,
                                          "achieved_gbs": legacy_rate * 20.0 / 1e9, "frac_of_hbm_peak": legacy_rate * 20.0 / 1e9 / hbm,
                                          "algorithmic_bytes_per_transition": 20.0,
                                          "transitions_per_launch": 2 * n * leg_iters,
                                          "moved_bytes_per_transition": 12.0 + 8.0 / leg_iters,
                                          "moved_gbs": legacy_rate * (12.0 + 8.0 / leg_iters) / 1e9,
                                          "moved_frac_of_hbm_peak": legacy_rate * (12.0 + 8.0 / leg_iters) / 1e9 / hbm},
                      "variant": args.variant, "other_variants": others,
                      "rollout_64k_games": {"config": "BASELINE configs[2]+[3]: 65536 games, ring 200000 + reservoir 2000000, rollout(8) + memory inserts; then the 256-row sample of all four memories",
                                            "transitions_per_sec": rate64, "ms_per_step": ms64 / args.steps,
                                            "sample_256_all_memories_us": 1e3 * ms64s / args.steps},
                      "buffers": buffers,
                      "learner": {"update_ms": learner_ms, "sgd_steps_per_update": 8, "allreduce_floats": 4 * 2179 + 8,
                                  "exploitability_proxy": lstats.get("exploitability"), "trained_mask": lstats.get("trained")},
                      "hands": int(st[10]), "transitions_counted": int(st[11]), "records_dropped": int(st[12])}}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--variant", default="default", choices=["default", "states", "cuda", "pairs", "sorted", "tcgen05", "tcgen05_ws"],
                    help="rollout kernel: table of the nets' outputs per decision state (default), per-decision CUDA-core row sums, "
                         "net-sorted warp groups, tcgen05 tensor-core tiles")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (float64; rank 0's games)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
