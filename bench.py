#!/usr/bin/env python
"""bench.py — DQN training steps/sec (batch 32, 84x84x4 uint8 states) on N B200s, beside the CPU
restatement of the reference path (BASELINE.json metric).

One "step" = one ReplayMemory.getMinibatch() + one DeepQNetwork.train()
(/root/reference/src/agent.py:112-114) on synthetic frames of SURVEY §8(d):
replay 1M x 84x84 u8 (7.06 GB ring in HBM, a 10k-frame random block tiled), batch 32 per GPU,
A = 4, terminals ~ Bernoulli(0.005), random.seed(1), Xavier weights (RandomState(1)).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--math fp32|tcgen05]
                  [--dump-outputs DIR]

N > 1 is launched by the driver through torch.distributed.run (one rank per GPU, NCCL).  Rank 0
prints ONE JSON line.  `value` times the fused device path with inputs resident in HBM; `e2e`
times the public drop-in classes from HOST buffers (frames appended with mem.add, the host `random`
kept in lock-step, cost delivered to the callback inside train()); `roofline` comes from the in-graph
%globaltimer timeline of the production graph (208 profiled steps regardless of --steps) with the
replay-gather HBM fraction and the conv-stack tensor fraction as first-class fields;
`predict_latency` times the agent's action selection — see DESIGN.md §6.

--dump-outputs DIR writes, right after the timed steps and before anything else runs, what a caller of the fused
path holds after its last step: the weights and RMSProp state of every layer (<layer>_W.npy, <layer>_S.npy), the
step's cost (cost.npy) and its online / target Q-values (q_online.npy, q_target.npy), all float32 (13.5 MB at A = 4).
The inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import random
import subprocess
import sys
import threading
import time
import types

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "DQN training steps/sec (batch 32, 84x84x4)"
UNIT = "steps/s"
BLOCK = 10_000
NUM_ACTIONS = 4
LAYERS = ("conv1", "conv2", "conv3", "fc1", "fc2")

# algorithmic MACs per sample of each GEMM-shaped kernel (SURVEY §8d), nets = 2 for forward kernels
MAC = {"conv1": 20 * 20 * 32 * 256, "conv2": 9 * 9 * 64 * 512, "conv3": 7 * 7 * 64 * 576, "fc1": 3136 * 512}
N_PARAMS = 256 * 32 + 512 * 64 + 576 * 64 + 3136 * 512 + 512 * NUM_ACTIONS


def make_args(batch):
    return types.SimpleNamespace(screen_height=84, screen_width=84, history_length=4, batch_size=batch,
                                 discount_rate=0.99, learning_rate=0.00025, decay_rate=0.95, clip_error=1,
                                 min_reward=-1, max_reward=1, batch_norm=False, random_seed=1, device_id=0,
                                 datatype="float32", stochastic_round=False, optimizer="rmsprop",
                                 target_steps=10000, save_weights_prefix=None)


def synthetic_meta(size):
    g = np.random.default_rng(0)
    base = g.integers(0, 256, (BLOCK, 84, 84), dtype=np.uint8)
    actions = g.integers(0, NUM_ACTIONS, size, dtype=np.uint8)
    rewards = g.integers(-1, 2, size, dtype=np.int64)
    terminals = g.random(size) < 0.005
    return base, actions, rewards, terminals


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d.get("bf16_tflops_sustained"),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled every 100 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.t = [], []
        self.gpu = gpu_index
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
        except OSError:
            return
        th = threading.Thread(target=self._read, daemon=True)
        th.start()

    def _read(self):
        for line in self.p.stdout:
            self.rows.append(line.strip().split(", "))
            self.t.append(time.time())

    def stop(self, t0, t1):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        rows = [r for r, t in zip(self.rows, self.t) if t0 - 0.05 <= t <= t1 + 0.15] or self.rows[-3:]
        sm = [float(r[1]) for r in rows if len(r) >= 9]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in rows if len(r) >= 9 for n, v in zip(names, r[5:9]) if v.strip() == "Active"})
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(rows[0][2]) if rows and len(rows[0]) >= 3 else None,
                "power_w_max": max((float(r[3]) for r in rows if len(r) >= 9), default=None),
                "samples": len(sm), "reasons": reasons}


# ------------------------------------------------------------------------------------------ CPU arm
def cpu_arm(steps, warmup, replay, batch, max_seconds=None):
    """The reference's hot path restated on the host cores: getMinibatch (numpy ring, CPython
    `random`, oracle/replay_oracle.py) + train (torch-CPU fp32, oracle/dqn_torch.py)."""
    import torch
    from oracle import dqn_oracle as O
    from oracle.dqn_torch import TorchDQN
    from oracle.replay_oracle import ReplayOracle
    base, actions, rewards, terminals = synthetic_meta(replay)
    ring = ReplayOracle(replay, batch_size=batch)
    for s in range(0, replay, BLOCK):
        e = min(replay, s + BLOCK)
        ring.screens[s:e] = base[:e - s]
    ring.actions[:], ring.rewards[:], ring.terminals[:] = actions, rewards, terminals
    ring.count, ring.current = replay, 123456 % replay
    net = TorchDQN(O.xavier_init(NUM_ACTIONS, 1))
    rnd = random.Random(1)
    # "all the host threads it can use": oneDNN at batch 32 does not scale to 100+ cores, so pick the
    # thread count that is actually fastest on this box (2 probe steps each) and report it.
    best = (None, 1e9)
    for _ in range(5):                       # first touches of the 7 GB ring, oneDNN primitive creation
        net.train(ring.getMinibatch(rnd))
    for nt in sorted({8, 16, 32, 64, torch.get_num_threads()}):
        if nt > (os.cpu_count() or 8):
            continue
        torch.set_num_threads(nt)
        for _ in range(3):
            net.train(ring.getMinibatch(rnd))
        t0 = time.perf_counter()
        for _ in range(8):
            net.train(ring.getMinibatch(rnd))
        dt = (time.perf_counter() - t0) / 8
        if dt < best[1]:
            best = (nt, dt)
    torch.set_num_threads(best[0])
    for _ in range(max(warmup, 10)):         # a baseline measured cold would flatter the GPU arm
        net.train(ring.getMinibatch(rnd))
    t0 = time.perf_counter()
    done = 0
    for _ in range(steps):
        net.train(ring.getMinibatch(rnd))
        done += 1
        if max_seconds and time.perf_counter() - t0 > max_seconds:
            break
    dt = time.perf_counter() - t0
    return dict(value=done / dt, unit=UNIT, cores=torch.get_num_threads(), kind="port",
                sample="%d steps of (numpy-ring getMinibatch + torch-CPU fp32 train), replay %d, batch %d, "
                       "%d torch threads of %d host cpus" % (done, replay, batch, torch.get_num_threads(),
                                                             os.cpu_count())), dt, done


def run_reference(a, rank, world):
    if rank != 0:
        return
    cb, dt, done = cpu_arm(a.steps, a.warmup, a.replay, a.batch)     # exactly --steps timed steps, after a thorough warm-up
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": a.gpus,
            "steps": done, "warmup": a.warmup, "ms_per_step": 1e3 * dt / done, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(a, world),
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "Neon --backend cpu cannot run (Neon absent, no network) and /root/reference does not exist on "
                    "the GPU box, so neither the reference's deepqnetwork.py nor its replay_memory.py can be timed here: "
                    "this is the CPU restatement (oracle port: numpy ring + CPython random + torch-CPU fp32 train) of "
                    "getMinibatch+train on the box's host cores at its fastest thread count"}
    print(json.dumps(line), flush=True)


def workload_config(a, world, comm="NCCL grad all-reduce"):
    return {"workload": "configs[1]: synthetic 84x84 uint8 frames, replay %d, batch %d per GPU, history 4, A=%d "
                        "(fused getMinibatch+train, no env)" % (a.replay, a.batch, NUM_ACTIONS),
            "replay": a.replay, "batch_per_gpu": a.batch, "global_batch": a.batch * world, "num_actions": NUM_ACTIONS,
            "math_mode": a.math, "parallelism": "dp%d replicated-replay learners, %s" % (world, comm)
            if world > 1 else "single GPU",
            "l2_policy": "inputs larger than L2: random 35 KB windows of a 7.06 GB ring; weights/activations are the "
                         "step's own working set"}


# ------------------------------------------------------------------------------------------ GPU arm
def kernel_model(label, nb, world=1):
    """(bound, algorithmic bytes, algorithmic flops) of one launch of kernel `label` (DESIGN.md §4 kernel table).
    bound: "tensor" (GEMM-shaped, tcgen05), "hbm" (bytes that must move; L2-resident ones are marked in DESIGN),
    "nvlink" (peer stores), "latency" (a few hundred bytes of work: the launch itself is the cost)."""
    f = lambda macs, nets=1: 2.0 * macs * nb * nets
    n_fc1, A = 3136 * 512, NUM_ACTIONS
    small = {"conv1": 256 * 32, "conv2": 512 * 64, "conv3": 576 * 64, "fc2": 512 * A}
    table = {
        "sample": ("latency", 625 * 4 * 2 + 40 * 4, 0.0),
        "conv1_fwd": ("tensor", nb * 35280 + 2 * 4 * 256 * 32, f(MAC["conv1"], 2)),
        "conv2_fwd": ("tensor", 0, f(MAC["conv2"], 2)), "conv3_fwd": ("tensor", 0, f(MAC["conv3"], 2)),
        "fc1_fwd": ("tensor", 2 * 4 * n_fc1, f(MAC["fc1"], 2)),
        "head": ("latency", nb * (2 * 7 * 512 * 4 + 512 * 4 * (3 + A)), 2.0 * 2 * nb * 512 * A),
        "cost": ("latency", nb * 4, 0.0),
        "fc1_wgrad": ("tensor", 4 * n_fc1, f(MAC["fc1"]) * world), "fc1_wgrad+opt": ("tensor", 24 * n_fc1, f(MAC["fc1"])),
        "fc1_dgrad": ("tensor", 4 * n_fc1, f(MAC["fc1"])), "conv3_wgrad": ("tensor", 0, f(MAC["conv3"])),
        "conv3_dgrad": ("tensor", 0, f(MAC["conv3"])), "conv2_wgrad": ("tensor", 0, f(MAC["conv2"])),
        "conv2_dgrad": ("tensor", 0, f(MAC["conv2"])), "conv1_wgrad": ("tensor", nb * 35280, f(MAC["conv1"])),
        # elementwise kernels: bytes they must move (fp32 dW, W, S in; W, S out; fp16 hi/lo image out)
        "optimizer": ("hbm", 5 * 4 * N_PARAMS, 0.0),
        "opt_fc1": ("hbm", (5 * 4 + 4) * n_fc1, 0.0),   # the one fc1 tile image (hi + lo fp16) is refreshed in the same pass
        "opt_fc2": ("latency", (nb + 4) * 4 * small["fc2"], 0.0),
        "opt_conv1": ("latency", (5 * 4 + 4) * small["conv1"], 0.0),
        "opt_conv2": ("latency", (5 * 4 + 8) * small["conv2"], 0.0),
        "opt_conv3": ("latency", (5 * 4 + 8) * small["conv3"], 0.0),
        "gather": ("hbm", nb * (35280 + 2 * 28224), 0.0),
        # data-parallel schedule (comm_p2p.cuh)
        "push_h3": ("nvlink", world * nb * 3136 * 2 * 2, 0.0), "push_dz4": ("nvlink", world * nb * 512 * 2 * 2, 0.0),
        "wait_push": ("latency", 2 * world * 4, 0.0),
        "grad_reduce": ("hbm", 2 * 4 * N_PARAMS, 0.0), "xchg_all": ("nvlink", 2 * 4 * N_PARAMS, 0.0),
        "xchg_fc": ("nvlink", 2 * 4 * (n_fc1 + small["fc2"]), 0.0), "reduce_fc": ("hbm", 2 * 4 * n_fc1, 0.0),
    }
    for k, v in small.items():
        table["reduce_" + k] = ("latency", 2 * 4 * v, 0.0)
        table["xll_" + k] = ("nvlink", (world - 1) * 16 * (v // 2), 0.0)
        table["optx_" + k] = ("nvlink", (world - 1) * 16 * (v // 2), 0.0)
        table["xchg_" + k] = ("nvlink", 2 * 4 * v, 0.0)
    return table.get(label, ("latency", 0, 0.0))


def graph_timeline(net, mem, L, dev, stream, reps=13, batch=16, at=12):
    """In-graph timeline (GPU %globaltimer per launch, csrc/common.cuh::KTrace) of the PRODUCTION step — replayed CUDA
    graph, PDL chain and side branches live — averaged over `reps` recordings of the `at`-th step of a
    `batch`-step burst (reps * batch = 208 profiled steps, independent of --steps).  Returns
    ({label: (mean start us, mean end us, mean duration us)}, mean step span us)."""
    import torch
    acc, spans = {}, []
    for _ in range(reps):
        L.ktrace_begin(dev, step=at)
        net.train_fused(mem, batch)
        torch.cuda.synchronize()
        rows = [r for r in L.ktrace_end() if r[1] < 2 ** 63 and r[2] > 0]
        if not rows:
            continue
        t0 = min(r[1] for r in rows)
        spans.append((max(r[2] for r in rows) - t0) / 1e3)
        for name, a, b in rows:
            acc.setdefault(name, []).append(((a - t0) / 1e3, (b - t0) / 1e3))
    out = {k: (float(np.mean([x[0] for x in v])), float(np.mean([x[1] for x in v])),
               float(np.mean([x[1] - x[0] for x in v]))) for k, v in acc.items()}
    return out, float(np.mean(spans)) if spans else 0.0


def dump_outputs(out_dir, net):
    """What the last timed step left for its caller, as float32 .npy files (see the module docstring)."""
    os.makedirs(out_dir, exist_ok=True)
    ws, ss = net.get_weights()
    q_online, q_target = net.last_q()
    arrays = {"cost": net.last_costs(1), "q_online": q_online, "q_target": q_target}
    for name, w, st in zip(LAYERS, ws, ss):
        arrays[name + "_W"], arrays[name + "_S"] = w, st
    for name, arr in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(arr, dtype=np.float32))


def run_b200(a, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from simple_dqn_b200 import DeepQNetwork, ReplayMemory, _lib as L

    torch.cuda.set_device(local_rank)
    dev = local_rank
    t_start = time.time()

    def note(msg):      # progress on stderr (B200DQN_BENCH_VERBOSE=1): locating a stall on a multi-rank box
        if os.environ.get("B200DQN_BENCH_VERBOSE"):
            sys.stderr.write("[bench rank %d %.1fs] %s\n" % (rank, time.time() - t_start, msg))
            sys.stderr.flush()
    if world > 1:
        dist.init_process_group("cpu:gloo,cuda:nccl", rank=rank, world_size=world)
    stream = torch.cuda.Stream()          # non-default: enables CUDA-graph replay + side-stream branches
    torch.cuda.set_stream(stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    args = make_args(a.batch)
    args.device_id = dev
    base, actions, rewards, terminals = synthetic_meta(a.replay)
    gbatch = a.batch * world

    def new_mem(**kw):
        margs = make_args(gbatch)
        m = ReplayMemory(a.replay, margs, device=dev, stream=stream, **kw)
        for s in range(0, a.replay, BLOCK):
            e = min(a.replay, s + BLOCK)
            m.add_batch(actions[s:e], rewards[s:e], base[:e - s], terminals[s:e])
        m.set_cursor(a.replay, 123456 % a.replay)
        return m

    mem = new_mem(rng="device")
    net = DeepQNetwork(NUM_ACTIONS, args, device=dev, math_mode=a.math, stream=stream)
    net.update_target_network()
    if world > 1:
        from simple_dqn_b200.parallel import broadcast_unique_id
        net.comm_init(broadcast_unique_id(dist, DeepQNetwork.comm_unique_id, rank), rank, world)
    random.seed(1)
    mem.seed_device_rng(random)
    note("objects + communicator up")

    # ---- value: fused device path, inputs resident in HBM
    net.train_fused(mem, a.warmup)
    barrier()
    note("warm-up done")
    sampler = ClockSampler(dev)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_wall0 = time.time()
    ev0.record(stream)
    net.train_fused(mem, a.steps)
    ev1.record(stream)
    barrier()
    t_wall1 = time.time()
    ms = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64)
    if world > 1:
        msd = ms.cuda()
        dist.all_reduce(msd, op=dist.ReduceOp.MAX)
        ms = msd.cpu()
    ms_total = float(ms[0])
    note("timed region done: %.1f us/step" % (1e3 * ms_total / a.steps))
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    cost_tail = net.last_costs(min(a.steps, 8))
    assert np.isfinite(cost_tail).all(), cost_tail
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, net)
    launches = net.launches_per_step() * a.steps

    # ---- roofline: the in-graph timeline of the production step (same graph, PDL and branches as `value`)
    barrier()
    tl, span_us = graph_timeline(net, mem, L, dev, stream)
    note("in-graph timeline done: span %.1f us" % span_us)
    pk = peaks()
    tf_peak = pk["tf_sustained"] or pk["tf_burst"]
    dur = {k: v[2] for k, v in tl.items()}
    # the dominant kernel is chosen by algorithmic work, not by a noisy duration ranking: conv1_fwd carries the
    # largest FLOP count of the step AND every mandatory HBM byte (the replay gather)
    top = "conv1_fwd"
    bound, abytes, aflops = kernel_model(top, a.batch, world)
    roof = {"kernel": top, "bound": "tensor", "achieved": aflops / (dur[top] * 1e-6) / 1e12, "peak": tf_peak,
            "unit": "TFLOP/s"}
    roof["frac"] = roof["achieved"] / roof["peak"]
    roof["traffic"] = None
    tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")     # dram bytes per launch from the committed ncu capture
    if os.path.exists(tp):
        roof["traffic"] = json.load(open(tp)).get(a.math, {}).get(top)
    roof["peak_source"] = pk["source"] + ", sustained bf16 figure (kernel timed inside a long step)"
    roof["us_per_launch"] = dur[top]
    roof["share_of_step"] = dur[top] / span_us if span_us else None
    roof["how"] = ("in-graph %globaltimer timeline of the replayed production graph (first CTA start .. last CTA end, "
                   "so a PDL-parked prologue counts), mean of 13 recordings; kernel chosen by algorithmic work")
    roof["gather"] = {"kernel": "conv1_fwd (frames read in place from the ring, fused into the first conv layer)",
                      "algorithmic_bytes": a.batch * 35280, "achieved_gbs": a.batch * 35280 / (dur[top] * 1e-6) / 1e9,
                      "peak_gbs": pk["hbm_gbs"],
                      "frac_of_hbm_peak": a.batch * 35280 / (dur[top] * 1e-6) / 1e9 / pk["hbm_gbs"]}
    conv_flops = 2.0 * a.batch * (4 * (MAC["conv1"] + MAC["conv2"] + MAC["conv3"]) - MAC["conv1"])
    conv_us = sum(v for k, v in dur.items() if k.startswith("conv"))
    roof["conv_stack"] = {"gflop": conv_flops / 1e9, "kernel_time_us": conv_us,
                          "achieved_tflops": conv_flops / (conv_us * 1e-6) / 1e12 if conv_us else None,
                          "frac_of_peak": conv_flops / (conv_us * 1e-6) / 1e12 / tf_peak if conv_us else None,
                          "frac_of_peak_over_step": conv_flops / (ms_total / a.steps * 1e-3) / 1e12 / tf_peak}
    whole_step_flops = 2.0 * a.batch * (4 * sum(MAC.values()) - MAC["conv1"])
    roof["whole_step"] = {"gflop": whole_step_flops / 1e9, "span_us": span_us,
                          "achieved_tflops": whole_step_flops / (ms_total / a.steps * 1e-3) / 1e12,
                          "frac_of_peak": whole_step_flops / (ms_total / a.steps * 1e-3) / 1e12 / tf_peak,
                          "gather_gbs": a.batch * 35280 / (ms_total / a.steps * 1e-3) / 1e9}
    per_kernel = {}
    for k, (t_a, t_b, d) in sorted(tl.items(), key=lambda kv: kv[1][0]):
        kb, by, fl = kernel_model(k, a.batch, world)
        e = {"start_us": round(t_a, 2), "end_us": round(t_b, 2), "us": round(d, 2), "bound": kb}
        if fl:
            e["tflops"] = round(fl / (d * 1e-6) / 1e12, 2)
        if by:
            e["gbs"] = round(by / (d * 1e-6) / 1e9, 1)
        per_kernel[k] = e
    roof["per_kernel"] = per_kernel

    # ---- predict latency (agent.py:55-61 runs it on 90-95 % of env steps)
    from simple_dqn_b200 import StateBuffer
    pred = {}
    st_host = np.ascontiguousarray(np.broadcast_to(base[:4], (a.batch, 4, 84, 84)))
    sbuf = StateBuffer(make_args(a.batch), device=dev, stream=stream)
    for i in range(6):
        sbuf.add(base[i])
    for name, arg in (("host_states_full_batch", st_host), ("state_buffer_live_row", sbuf.getStateMinibatch())):
        for _ in range(20):
            net.predict(arg)
        t0 = time.perf_counter()
        for _ in range(200):
            net.predict(arg)
        pred[name + "_us"] = (time.perf_counter() - t0) / 200 * 1e6
    t0 = time.perf_counter()
    for i in range(200):
        sbuf.add(base[i % 64])
        net.predict(sbuf.getStateMinibatch())
    pred["state_buffer_add_plus_predict_us"] = (time.perf_counter() - t0) / 200 * 1e6
    note("predict latency done")

    # ---- e2e: the drop-in public API from HOST buffers (agent.py:100-114 without env / predict):
    # 4 x mem.add(host frame) [train_frequency 4], getMinibatch() with the HOST random stream
    # (MT state up + down), train(), cost read back for the stats callback.
    del mem
    mem2 = new_mem(rng="python", device_minibatch=True)
    random.seed(1)
    costs = []
    net.callback = types.SimpleNamespace(on_train=lambda c: costs.append(c))
    frames = [np.ascontiguousarray(base[i]) for i in range(64)]
    e2e_steps = max(300, min(a.steps, 1000))          # a fixed floor: the driver runs --steps 20

    def e2e_loop(n):
        for i in range(n):
            for j in range(4):
                mem2.add(int(actions[j]), int(rewards[j]), frames[(4 * i + j) % 64], bool(terminals[j]))
            net.train(mem2.getMinibatch(), 0)

    barrier()            # ring refill time differs per rank; peers wait inside exchange kernels only for bounded time
    e2e_loop(10)
    note("e2e warm-up done")
    barrier()
    t0 = time.perf_counter()
    e2e_loop(e2e_steps)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    note("e2e done")
    dts = torch.tensor([dt], dtype=torch.float64)
    if world > 1:
        d = dts.cuda()
        dist.all_reduce(d, op=dist.ReduceOp.MAX)
        dts = d.cpu()
    e2e = {"value": world * e2e_steps / float(dts[0]), "unit": UNIT,
           "h2d_bytes_per_step": 4 * 7056, "d2h_bytes_per_step": 4 + 4,
           "steps": e2e_steps,
           "what": "per step, through the drop-in classes: 4x ReplayMemory.add(host frame -> pinned bank -> HBM) + "
                   "getMinibatch() [device handle; the index draw rides in train()'s graph] + DeepQNetwork.train() in "
                   "lock-step with the host `random` stream (state up when it moved, words consumed back) + cost "
                   "delivered to the stats callback inside train() (host-mapped result words, one wait per step)"}
    assert len(costs) == e2e_steps + 10 and np.isfinite(costs).all()
    net.callback = None

    comm_mode, comm_ok = net.comm_status()
    if world > 1:          # orderly teardown on EVERY rank before rank 0 goes on to print
        torch.cuda.synchronize()
        dist.barrier()
        net.comm_destroy()
        dist.destroy_process_group()
    if rank != 0:
        return
    line = {"metric": METRIC, "value": world * a.steps / (ms_total * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms_total / a.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if a.math == "fp32" else "f16x3-split (fp32 accumulate)", "data": "synthetic",
            "config": workload_config(a, world, {"p2p": "NVLink peer memory, schedule '%s' (gather: fc1's operand rows "
                                                        "pushed to every rank, fc1_wgrad over the global batch, LL "
                                                        "one-shot all-reduce for conv1-3/fc2; comm_p2p.cuh)"
                                                        % os.environ.get("B200DQN_P2P_SCHED", "gather"),
                                                 "nccl": "NCCL grad all-reduce"}.get(comm_mode, comm_mode)),
            "comm_healthy": bool(comm_ok), "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
            "roofline": roof, "predict_latency": pred, "last_costs": [float(c) for c in cost_tail]}
    if world > 1:
        line["config"]["global_updates_per_s"] = a.steps / (ms_total * 1e-3)
        # NVLink bytes each rank SENDS per step (SURVEY §8e asks for the fraction of 770 GB/s per direction)
        n_params = 1683456 + 512 * NUM_ACTIONS
        small = n_params - 3136 * 512                           # conv1..3 + fc2, floats
        if comm_mode == "p2p" and os.environ.get("B200DQN_P2P_SCHED", "gather") == "gather":
            sent = (world - 1) * (a.batch * (3136 + 512) * 2 * 2    # H3 + dZ4 rows, fp16 hi + lo planes
                                  + small * 4 * 2)                  # LL lines: 8 B data + 8 B flags
            how = "(W-1) x (H3/dZ4 hi+lo rows + LL lines of conv1-3, fc2)"
        else:
            sent = 2 * (world - 1) * n_params * 4 // world
            how = "reduce-scatter + all-gather of the 6.74 MB gradient"
        gbs = sent / (ms_total / a.steps * 1e-3) / 1e9
        line["nvlink"] = {"sent_bytes_per_step_per_rank": int(sent), "what": how, "GBps_per_rank": gbs,
                          "frac_of_770GBps_per_dir": gbs / 770.0}
    if world == 1 and not a.no_cpu:
        cb, _, _ = cpu_arm(10 ** 9, 3, a.replay, a.batch, max_seconds=a.cpu_seconds)
        line["cpu_baseline"] = cb
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3000)
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--math", default=os.environ.get("B200DQN_MATH", "tcgen05"), choices=["fp32", "tcgen05"])
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--replay", type=int, default=1_000_000)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (b200 only)")
    a = ap.parse_args()
    assert a.warmup >= 3, "timing rules: at least 3 warm-up steps"
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if a.impl == "reference":
        if a.dump_outputs:
            ap.error("--dump-outputs writes the outputs of the b200 path; --impl reference has none to write")
        return run_reference(a, rank, world)
    run_b200(a, rank, world, local_rank)


if __name__ == "__main__":
    main()
