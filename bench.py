#!/usr/bin/env python
"""Benchmark of the AlphaQuoridorGNN hot path on B200 (contract: see the task statement / DESIGN.md section 7).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one batched leaf evaluation (BaseNetwork.predict semantics for B states: legal-move mask + graph build +
GNN forward + restriction to legal actions) over one batch of B = 16,384 synthetic legal positions per GPU --
BASELINE.json configs[2].  Headline metric: GNN board-evals/s.  The other BASELINE metrics are measured after the
headline and reported under "extra", each with its own roofline block and the CPU port of the same work timed in the
same run (rank 0, N = 1 only):
    extra.legal_mask     configs[1]: legal-move + wall-legality masks of 1,000,000 positions
    extra.train          configs[0]: forward + loss + backward + (all-reduce) + Adam at B = 256, and at B = 4096
    extra.mcts           configs[3]: 4,096 lock-step self-play games x 200 simulations per move, WHOLE games
    extra.train_cycle    configs[4]: the self-play record of extra.mcts -> data-parallel training (one epoch)

`--impl reference` times the CPU port of the reference path (oracle/: C restatement of game_logic + torch restatement of
pv_network_gnn) on the host cores; the reference itself is pure Python with un-vendored dependencies and cannot travel to
the GPU box.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_PER_BOARD_FWD = 5.79e6      # SURVEY.md section 8d
FLOP_PER_BOARD_FWDBWD = 16.9e6
BYTES_PER_POSITION_LEGAL = 72    # 32 B packed state in + 32 B mask + 8 B ordered pawn list out (DESIGN.md section 4)
BYTES_PER_BOARD_HEADS = 128 * 4 + 209 * 4 + 4 + 32
# dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed `ncu --set full` capture
# named here (a profiler cannot run inside the timed bench; the capture is of the same command line)
NCU_TRAFFIC = {("gcn_forward_kernel", 1, 16384): (632064, "profiles/r1_v3_kernels_ncu.csv: gcn_forward_tc2_kernel, dram read 0.632 MB + write 0 "
                                                  "(the 8 MB of pooled output is still in L2 when the kernel ends)")}
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, outputs):
    """Writes the result arrays of one leaf-evaluation step as <out_dir>/<name>.npy: float32, and float64 for the 32-bit legal-mask
    words, so every value is stored exactly.  When the boards do not fit in DUMP_MAX_BYTES, a fixed seeded sample of them is written;
    board_index.npy names the boards written, so two builds run with the same arguments compare output for output."""
    host = {k: v.cpu().numpy() for k, v in outputs.items()}
    host["mask"] = host["mask"].view(np.uint32).astype(np.float64)
    host = {k: v if v.dtype == np.float64 else v.astype(np.float32) for k, v in host.items()}
    B = len(host["priors"])
    per_board = sum(v[:1].nbytes for v in host.values()) + 8                  # + the board's index
    n = min(B, (DUMP_MAX_BYTES - 4096) // per_board)                          # 4 KB for the .npy headers
    idx = np.arange(B) if n == B else np.sort(np.random.default_rng(0).choice(B, n, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "board_index.npy"), idx.astype(np.float64))
    for k, v in host.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), v[idx])


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm": d["hbm_gbs"], "tensor_burst": d["bf16_tflops"], "tensor": d["bf16_tflops_sustained"],
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm": 6650.0, "tensor_burst": 1590.0, "tensor": 1400.0, "source": "fallback (B200_PROFILING.md)"}


def bind_to_gpu_numa(index):
    """Pin this process to the CPUs next to its GPU (sysfs local_cpulist of the GPU's PCI device) BEFORE any pinned host buffer is
    allocated, so that the buffers of the host-buffer path live on the GPU's NUMA node.  Best effort: returns a description."""
    if os.environ.get("AQ_BENCH_NUMA", "1") == "0":
        return "off"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(index)],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        bdf = out[-12:] if len(out) >= 12 else out  # nvidia-smi prints an 8-digit domain; sysfs uses 4
        with open(f"/sys/bus/pci/devices/{bdf}/local_cpulist") as f:
            cpulist = f.read().strip()
        cpus = set()
        for part in cpulist.split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return f"gpu {index} at {bdf}: no usable local cpus ({cpulist})"
        os.sched_setaffinity(0, cpus)
        return f"gpu {index} at {bdf}: bound to {len(cpus)} local cpus ({cpulist})"
    except Exception as e:  # sysfs not visible in this container, single-socket host, ...
        return f"unavailable ({type(e).__name__}: {e})"


class ClockSampler:
    """SM clocks and throttle reasons sampled DURING the timed regions, through NVML in this process (what nvidia-smi itself reads;
    a process per sample -- round 1 -- costs seconds on a fresh box and takes driver locks that the host path's CUDA calls contend
    for at N = 8).  Falls back to one long-running `nvidia-smi -lms` child if the NVML bindings are unavailable."""

    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index, period=0.1):
        self.index, self.period, self.rows, self.stop_flag, self.t, self.child, self.source = index, period, [], False, None, None, None

    def _run_nvml(self):
        import pynvml
        h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
        mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
        while not self.stop_flag:
            try:
                sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                rs = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h) if hasattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.rows.append((float(sm), float(mx), int(rs)))
            except Exception:
                pass
            time.sleep(self.period)

    def _run_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        self.child = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index), "-lms",
                                       str(int(self.period * 1000))], stdout=subprocess.PIPE, text=True)
        for line in self.child.stdout:
            c = [x.strip() for x in line.split(",")]
            if len(c) >= 6 and c[0].replace(".", "").isdigit():
                bits = sum(bit for (_, bit), v in zip(self.REASONS, c[2:6]) if v.lower().startswith("active"))
                self.rows.append((float(c[0]), float(c[1]), bits))
            if self.stop_flag:
                break

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.source, target = "nvml", self._run_nvml
        except Exception:
            self.source, target = "nvidia-smi -lms", self._run_smi
        self.t = threading.Thread(target=target, daemon=True)
        self.t.start()

    def stop(self):
        self.stop_flag = True
        if self.child is not None:
            self.child.terminate()
        if self.t:
            self.t.join(timeout=10)
        sm = [r[0] for r in self.rows]
        mx = [r[1] for r in self.rows]
        bits = 0
        for r in self.rows:
            bits |= r[2]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(n for n, b in self.REASONS if bits & b), "samples": len(self.rows), "source": self.source}


# ------------------------------------------------------------------------------------------------
# CPU ports (oracle/) of the same work: the reference arm and every cpu_baseline block
# ------------------------------------------------------------------------------------------------
def oracle_random_positions(n, seed):
    """Lock-step random games on the CPU with the C oracle (same move mix as positions.py)."""
    from oracle import quoridor_oracle as qo
    rng = np.random.default_rng(seed)
    out_rows, out_plies, total = [], [], 0
    while total < n:
        G = max(64, n // 32)  # ~32 plies deep, the same mix of game phases as positions.mixed_batches in run_ours
        rows = np.zeros((G, 68), np.uint8)
        rows[:, [0, 2]] = 76
        rows[:, [1, 3]] = 10
        plies = np.zeros(G, np.int16)
        for _ in range(116):
            if len(rows) == 0 or total >= n:
                break
            la = qo.legal_actions_batch(rows, plies)
            ok = la["n"] > 0
            rows, plies = rows[ok], plies[ok]
            acts, cnt = la["actions"][ok], la["n"][ok]
            out_rows.append(rows)
            out_plies.append(plies)
            total += len(rows)
            is_wall = (acts >= 81)
            valid = acts >= 0
            nw, npn = (is_wall & valid).sum(1), (~is_wall & valid).sum(1)
            use_wall = (nw > 0) & ((rng.random(len(rows)) < 0.5) | (npn == 0))
            pick = np.where(use_wall, npn + (rng.random(len(rows)) * nw).astype(np.int64),
                            (rng.random(len(rows)) * np.maximum(npn, 1)).astype(np.int64))
            pick = np.minimum(pick, cnt - 1)
            a = acts[np.arange(len(rows)), pick]
            rows, plies, flags = qo.next_batch(rows, plies, a)
            rows, plies = rows[flags == 0], plies[flags == 0]
    return np.concatenate(out_rows)[:n], np.concatenate(out_plies)[:n]


def oracle_leaf_eval(model, rows, plies, threads):
    """CPU port of one step: predict() semantics for a batch (pv_network_cnn.py:117-137 behaviour)."""
    from oracle import gnn_oracle, quoridor_oracle as qo
    la = qo.legal_actions_batch(rows, plies, nthreads=threads)
    x, ei, batch = gnn_oracle.graph_inputs_from_rows(rows)
    with torch.inference_mode():
        p, v = model(x, ei, batch)
    dense = torch.from_numpy(np.unpackbits(la["mask"].view(np.uint8), axis=1, bitorder="little")[:, :209].astype(bool))
    p = torch.where(dense, p, torch.zeros_like(p))
    s = p.sum(1, keepdim=True)
    p = p / torch.where(s == 0, torch.ones_like(s), s)
    return p, v


def time_cpu_leaf_eval(sample, steps, warmup, seed=1):
    from oracle import gnn_oracle, quoridor_oracle as qo
    qo.build()
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    model = gnn_oracle.GraphPolicyValueNetworkOracle().eval()
    rows, plies = oracle_random_positions(sample, seed)
    for _ in range(warmup):
        oracle_leaf_eval(model, rows, plies, threads)
    t0 = time.perf_counter()
    for _ in range(steps):
        oracle_leaf_eval(model, rows, plies, threads)
    dt = time.perf_counter() - t0
    return sample * steps / dt, dt / steps, threads


def time_cpu_legal_mask(sample=200_000, seed=3):
    """BASELINE configs[1] on the host: the C oracle's State.legal_actions() port over `sample` positions, all threads (OpenMP)."""
    from oracle import quoridor_oracle as qo
    threads = os.cpu_count() or 1
    rows, _ = oracle_random_positions(sample, seed)
    rows = rows[np.random.default_rng(seed).permutation(len(rows))]  # the generator emits plies in order: mix the game phases
    qo.legal_mask_only(rows[:2000], nthreads=threads)
    t0 = time.perf_counter()
    qo.legal_mask_only(rows, nthreads=threads)
    dt = time.perf_counter() - t0
    t1 = time.perf_counter()
    qo.legal_mask_only(rows[:sample // 8], nthreads=1)
    dt1 = time.perf_counter() - t1
    return {"value": sample / dt, "unit": "positions/s", "cores": threads, "kind": "port",
            "one_thread_positions_per_sec": (sample // 8) / dt1,
            "sample": f"{sample} synthetic positions (same move mix), C restatement of game_logic.legal_actions (oracle/quoridor_oracle.c, "
                      f"OpenMP, {threads} threads): {dt:.2f} s; one thread on {sample // 8}: {dt1:.2f} s"}


def time_cpu_train(B=256, steps=10, warmup=2, seed=5):
    """BASELINE configs[0] -- IS the CPU reference path: forward + loss + backward of the oracle network at B = 256 (plus Adam),
    all host threads and one thread."""
    from oracle import gnn_oracle
    rows, _ = oracle_random_positions(B, seed)
    x, ei, batch = gnn_oracle.graph_inputs_from_rows(rows)
    torch.manual_seed(1)
    pt = torch.softmax(torch.randn(B, 209), 1)
    vt = torch.randint(-1, 2, (B,)).float()
    out = {}
    for label, threads, n in (("all", os.cpu_count() or 1, steps), ("one", 1, max(2, steps // 3))):
        torch.set_num_threads(threads)
        torch.manual_seed(0)
        model = gnn_oracle.GraphPolicyValueNetworkOracle().train()
        opt = torch.optim.Adam(model.parameters(), lr=1e-3)

        def one_step():
            p, v = model(x, ei, batch)
            loss, _, _ = gnn_oracle.training_loss(p, v, pt, vt)
            opt.zero_grad()
            loss.backward()
            opt.step()

        for _ in range(warmup):
            one_step()
        t0 = time.perf_counter()
        for _ in range(n):
            one_step()
        out[label] = (B * n / (time.perf_counter() - t0), threads, n)
    torch.set_num_threads(os.cpu_count() or 1)
    v, threads, n = out["all"]
    return {"value": v, "unit": "samples/s", "cores": threads, "kind": "port", "one_thread_samples_per_sec": out["one"][0],
            "sample": f"{n} steps (after {warmup} warm-up) of B = {B}: torch-CPU restatement of pv_network_gnn forward + the reference loss + "
                      f"autograd backward + torch.optim.Adam, {threads} threads; one thread: {out['one'][2]} steps"}


def time_cpu_mcts(sims=200, roots=4, seed=7):
    """BASELINE configs[3] on the host: the port of pv_mcts_policy (oracle/mcts_oracle.py) at `sims` simulations with the torch-CPU
    GNN oracle as model.predict (batch of one per leaf, as the reference does), on a few mid-game roots, one process."""
    from oracle import gnn_oracle, mcts_oracle
    torch.set_num_threads(os.cpu_count() or 1)
    torch.manual_seed(0)
    model = gnn_oracle.GraphPolicyValueNetworkOracle().eval()
    rows, plies = oracle_random_positions(2048, seed)

    def predict(state):  # BaseNetwork.predict semantics (pv_network_cnn.py:117-137) for one state
        x, ei, batch = gnn_oracle.graph_inputs_from_rows(state.row[None, :])
        with torch.inference_mode():
            p, v = model(x, ei, batch)
        pol = p[0][state.legal_actions()]
        s = pol.sum()
        return (pol / (s if s else 1)).numpy(), float(v.item())

    pick = np.linspace(0, len(rows) - 1, roots).astype(int)
    mcts_oracle.pv_mcts_scores(predict, mcts_oracle.COracleState(rows[pick[0]], plies[pick[0]]), 8)  # warm-up
    t0 = time.perf_counter()
    for i in pick:
        mcts_oracle.pv_mcts_scores(predict, mcts_oracle.COracleState(rows[i], plies[i]), sims)
    dt = time.perf_counter() - t0
    return {"value": roots * sims / dt, "unit": "simulations/s", "cores": 1, "kind": "port",
            "sample": f"{roots} roots x {sims} simulations: port of pv_mcts_policy (pv_mcts.py:20-95) over the C game-logic oracle with the "
                      f"torch-CPU GNN oracle as model.predict (one leaf per call, torch using {os.cpu_count()} threads): {dt:.1f} s"}


def run_reference(args, rank, world):
    if rank != 0:
        return
    sample = 2048
    value, sec_per_step, threads = time_cpu_leaf_eval(sample, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": "gnn_board_evals_per_sec", "value": value, "unit": "board-evals/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec_per_step * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "leaf_eval (BASELINE configs[2]: batched predict = legal mask + GNN forward + legal renorm)",
                   "batch_per_step": sample, "note": "CPU port of the reference path (oracle/); the reference is pure "
                   "Python with un-vendored torch_geometric and cannot run on the GPU box"},
        "cpu_baseline": {"value": value, "unit": "board-evals/s", "cores": threads, "kind": "port",
                         "sample": f"{sample} synthetic positions per step, C oracle legal_actions (OpenMP) + torch CPU GNN forward"},
        "e2e": {"value": value, "unit": "board-evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def dp_check(dev, rank, world):
    """NCCL data-parallel PARITY inside the multi-GPU bench run (scripts/dp_check.py's assertions): three FlatTrainer steps with the
    batch sharded over the ranks and one all-reduce of the flat gradient per step give the gradients and losses of the
    single-GPU step on the whole batch, and every rank ends with bit-identical parameters."""
    import torch.distributed as dist
    from alphaquoridorgnn_b200 import positions, train_network
    from alphaquoridorgnn_b200.pv_network_gnn import GNNNetwork
    B = 250  # not divisible by 4 or 8: the shards differ in size
    packed = positions.random_positions(B, seed=7, games=64, device=dev)
    torch.manual_seed(1)
    pt = torch.softmax(torch.randn(B, 209), 1).to(dev)
    vt = torch.randint(-1, 2, (B,)).float().to(dev)
    report = {}
    for prec in ("fp32", "bf16"):
        torch.manual_seed(2)
        dp_net = GNNNetwork().to(dev).train()
        ref_net = GNNNetwork().to(dev).train()
        ref_net.load_state_dict(dp_net.state_dict())
        dp = train_network.FlatTrainer(dp_net, rank=rank, world_size=world, precision=prec)
        one = train_network.FlatTrainer(ref_net, precision=prec)
        lo, hi = train_network.shard_bounds(B, rank, world)
        worst = 0.0
        for _ in range(4):   # the first step of a shape runs eagerly, the second captures the CUDA graph, the others replay it
            l_dp = dp.step(packed[lo:hi].contiguous(), pt[lo:hi].contiguous(), vt[lo:hi].contiguous(), B).clone()
            dist.all_reduce(l_dp)
            l_one = one.step(packed, pt, vt, B)
            gerr = ((dp.grads - one.grads).norm() / one.grads.norm()).item()
            worst = max(worst, gerr)
            # fp32: summation order only.  bf16: the shard boundaries change which boards share a CTA, not the arithmetic per board, so
            # the sharded gradient differs from the single-GPU one by the fp32 summation order of the accumulators as well
            assert abs(l_dp.sum().item() - l_one.sum().item()) < 1e-5 and gerr < (1e-5 if prec == "fp32" else 1e-4), (prec, gerr)
        mine = dp.flat.clone()
        ref0 = mine.clone()
        dist.broadcast(ref0, 0)
        same = torch.tensor([1 if torch.equal(mine, ref0) else 0], device=dev)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        assert int(same.item()) == 1, "ranks diverged"
        dp.check()
        # the NCCL alternative gives the same gradient sum up to fp32 summation order
        torch.manual_seed(2)
        nc_net = GNNNetwork().to(dev).train()
        nc = train_network.FlatTrainer(nc_net, rank=rank, world_size=world, precision=prec, collective="nccl")
        torch.manual_seed(2)
        p2_net = GNNNetwork().to(dev).train()
        p2 = train_network.FlatTrainer(p2_net, rank=rank, world_size=world, precision=prec, use_graph=False)
        nc.step(packed[lo:hi].contiguous(), pt[lo:hi].contiguous(), vt[lo:hi].contiguous(), B)
        p2.step(packed[lo:hi].contiguous(), pt[lo:hi].contiguous(), vt[lo:hi].contiguous(), B)
        nerr = ((nc.grads - p2.grads).norm() / p2.grads.norm()).item()
        assert nerr < 1e-6, (prec, nerr)
        report[prec] = {"grad_rel_l2_vs_single_gpu": worst, "ranks_bit_identical": True, "collective": dp.collective,
                        "grad_rel_l2_peer_memory_vs_nccl": nerr}
    if rank == 0:
        print(f"dp_check ok (world {world}): {json.dumps(report)}", file=sys.stderr, flush=True)
    return report


def run_ours(args, rank, world, local_rank):
    import torch.distributed as dist
    from alphaquoridorgnn_b200 import _lib, positions, self_play, train_network
    from alphaquoridorgnn_b200 import game_logic as gl
    from alphaquoridorgnn_b200.pv_network_gnn import GNNNetwork, HostLeafEvaluator, PRECISIONS

    numa = bind_to_gpu_numa(local_rank)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    L = _lib.load()
    pk = peaks()
    B, K, Wm = args.batch, args.steps, args.warmup
    prec = PRECISIONS[args.precision]

    torch.manual_seed(0)
    net = GNNNetwork().to(dev).eval()
    net.precision = args.precision
    flat = net.flat_parameters()
    # inference weights prepared once, as prep_for_inference does (the weights do not change between evaluations)
    prep = net.prepared_weights() if prec == 1 else None
    nb = 4
    allpos, batches = positions.mixed_batches(nb, B, seed=1 + rank, device=dev)
    priors = torch.empty((B, 209), dtype=torch.float32, device=dev)
    value = torch.empty((B,), dtype=torch.float32, device=dev)
    mask = torch.empty((B, 8), dtype=torch.int32, device=dev)
    pawn = torch.empty((B, 8), dtype=torch.uint8, device=dev)
    pooled = torch.empty((L.aq_leaf_eval_ws_floats(B),), dtype=torch.float32, device=dev)  # leaf-eval workspace: pooled [B,128] | legal-mask task list
    lws = torch.empty((L.aq_legal_mask_ws_bytes(B),), dtype=torch.uint8, device=dev)
    flush = torch.empty((256 << 20,), dtype=torch.uint8, device=dev)
    st = _lib.stream_ptr(dev)
    P = _lib.ptr

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def reduce_max(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(fn, n, warm):
        """n launches of fn(i), L2 flushed before each, per-launch CUDA events on the launch stream -> (max over ranks of the
        mean ms per launch, this library's kernel launches per call, counted)."""
        for i in range(warm):
            fn(i)
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
        barrier()
        c0 = L.aq_launch_count()
        for i in range(n):
            flush.fill_(i & 0xFF)
            evs[i][0].record()
            fn(i)
            evs[i][1].record()
        launches = L.aq_launch_count() - c0
        barrier()
        return reduce_max(sum(a.elapsed_time(b) for a, b in evs) / n), launches

    def step(i, precision=prec, prepared=prep):
        _lib.check(L.aq_leaf_eval(P(flat), P(prepared), P(batches[i % nb]), B, P(priors), P(value), P(mask), P(pawn), P(pooled), precision, st),
                   "aq_leaf_eval")

    sampler = ClockSampler(local_rank)  # samples clocks / throttle reasons during ALL timed regions below
    sampler.start()
    ms_step, gpu_launches = timed(step, K, Wm)
    value_main = world * B / (ms_step * 1e-3)
    if args.dump_outputs and rank == 0:   # the buffers still hold the last timed step; the kernel timings below overwrite them
        dump_outputs(args.dump_outputs, {"priors": priors, "value": value, "mask": mask, "pawn": pawn})

    # ---- per-kernel durations (same inputs, same stream) for the roofline ------------------------
    def k_legal(i):
        _lib.check(L.aq_legal_mask_ws(P(batches[i % nb]), B, P(mask), P(pawn), P(lws), lws.numel(), st), "aq_legal_mask_ws")

    def k_trunk(i):
        _lib.check(L.aq_gcn_trunk_forward(P(flat), P(prep), P(batches[i % nb]), B, P(pooled), prec, st), "aq_gcn_trunk_forward")

    def k_heads(i):
        _lib.check(L.aq_heads_forward(P(flat), P(prep), P(pooled), B, P(priors), P(value), P(mask), prec, st), "aq_heads_forward")

    kms = {"legal_mask_kernels": timed(k_legal, K, 2)[0], "gcn_forward_kernel": timed(k_trunk, K, 2)[0],
           "heads_forward_kernel": timed(k_heads, K, 2)[0]}
    ksum = sum(kms.values())
    kinfo = {
        "legal_mask_kernels": {"bound": "hbm", "achieved": BYTES_PER_POSITION_LEGAL * B / (kms["legal_mask_kernels"] * 1e-3) / 1e9,
                              "peak": pk["hbm"], "unit": "GB/s"},
        "gcn_forward_kernel": {"bound": "tensor", "achieved": FLOP_PER_BOARD_FWD * B / (kms["gcn_forward_kernel"] * 1e-3) / 1e12,
                               "peak": pk["tensor"], "unit": "TFLOP/s"},
        "heads_forward_kernel": {"bound": "hbm", "achieved": BYTES_PER_BOARD_HEADS * B / (kms["heads_forward_kernel"] * 1e-3) / 1e9,
                                 "peak": pk["hbm"], "unit": "GB/s"},
    }
    for k, v in kinfo.items():
        v["ms"] = kms[k]
        v["share_of_step"] = kms[k] / ksum
        v["frac"] = v["achieved"] / v["peak"]
    dom = max(kms, key=kms.get)
    traffic = NCU_TRAFFIC.get((dom, prec, B), (None, "no ncu capture for this configuration"))
    roofline = {"kernel": dom, "bound": kinfo[dom]["bound"], "achieved": kinfo[dom]["achieved"], "peak": kinfo[dom]["peak"],
                "unit": kinfo[dom]["unit"], "frac": kinfo[dom]["frac"], "traffic": traffic[0], "traffic_source": traffic[1],
                "peak_source": pk["source"],
                "arith": "fp32 FFMA" if prec == 0 else "bf16 tcgen05 node transforms + fp16 tcgen05 aggregation, fp32 accumulate in TMEM",
                "kernel_symbol": "gcn_forward_fp32_kernel" if prec == 0 else "gcn_forward_tc2_kernel"}

    # ---- end to end through host buffers, every step: pinned packed states H2D, kernels, results D2H, one event wait ----
    hst = [torch.from_numpy(gl.pack_rows_host(*[t.cpu().numpy() for t in gl.unpack_rows(b)])).pin_memory() for b in batches]
    for h, b in zip(hst, batches):
        assert torch.equal(h, b.cpu())

    def e2e_pipelined(inflight, steps=None, **kw):
        """`inflight` evaluators (pools of games) used round-robin: while the host waits for one batch, the others' kernels run and
        their results cross PCIe.  Every step still moves its own states H2D and its own results D2H inside the timed region."""
        evs = [HostLeafEvaluator(net, B, **kw) for _ in range(inflight)]
        d2h = []

        def run(n):
            for j in range(min(inflight - 1, n)):
                evs[j].submit(B, states=hst[j % nb])
            for i in range(n):
                j = i + inflight - 1
                if j < n:
                    evs[j % inflight].submit(B, states=hst[j % nb])
                out = evs[i % inflight].wait()
                d2h.append(evs[i % inflight].d2h_bytes(out))

        n_timed = steps or K
        run(2 * inflight + 2)
        del d2h[:]
        barrier()
        t0 = time.perf_counter()
        run(n_timed)
        barrier()
        dt = reduce_max(time.perf_counter() - t0)
        short = sum(ev.stats()[0] for ev in evs)
        for ev in evs:
            ev.close()
        return world * B * n_timed / dt, int(sum(d2h) / len(d2h)), short

    def e2e_sync(dense):
        ev = HostLeafEvaluator(net, B, dense=dense)
        d2h = []
        for i in range(3):
            ev.evaluate(B, states=hst[i % nb])
        barrier()
        t0 = time.perf_counter()
        for i in range(K):
            d2h.append(ev.d2h_bytes(ev.evaluate(B, states=hst[i % nb])))  # synchronous: results are on the host when it returns
        barrier()
        dt = reduce_max(time.perf_counter() - t0)
        ev.close()
        return world * B * K / dt, int(sum(d2h) / len(d2h))

    def d2h_ceiling(nbytes, reps=300):
        """What this box's device -> host path gives one plain pinned cudaMemcpyAsync loop per rank, all ranks at once.  Long enough
        (about 1 GB per rank) that the ranks' loops really overlap: with 40 copies the eight-GPU figure came out a third too high."""
        src = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
        dst = torch.empty((nbytes,), dtype=torch.uint8).pin_memory()
        for _ in range(10):
            dst.copy_(src, non_blocking=True)
        barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            dst.copy_(src, non_blocking=True)
        barrier()
        return nbytes * reps / reduce_max(time.perf_counter() - t0) / 1e9

    wire = "f16" if prec == 1 else "f32"
    # How many batches to keep in flight is the caller's choice (one HostLeafEvaluator per pool of games).  More of them let the
    # legal-mask / heads / compaction kernels of neighbouring batches fill the ends of each other's trunk (6 in flight: +10 % on one
    # GPU); where the box's device -> host link is the limit (eight GPUs at once) more outstanding copies only contend (-6 %).  A
    # host would try both once; so does this: an untimed trial of each, then the K timed steps with the better one (the decision is
    # taken on the maximum over ranks, so every rank takes the same).
    est_d2h = B * (4 + 4 + 102 * (2 if wire == "f16" else 4))          # offsets + value + ~102 legal actions per board
    ceil_gbs = d2h_ceiling(max(1 << 20, est_d2h))
    trial = {n: e2e_pipelined(n, steps=max(12, K // 2), wire=wire, with_mask=False)[0] for n in (3, 6)}
    inflight = max(trial, key=trial.get)
    e2e_v, e2e_d2h, e2e_short = e2e_pipelined(inflight, wire=wire, with_mask=False)
    e2e = {"value": e2e_v, "unit": "board-evals/s", "h2d_bytes_per_step": B * 32, "d2h_bytes_per_step": e2e_d2h,
           "api": f"HostLeafEvaluator(wire='{wire}', with_mask=False).submit / wait -> aq_leaf_eval_host_compact_submit / _wait: what "
                  f"BaseNetwork.predict returns for a batch (ragged priors of the legal actions in legal_actions() order + value); "
                  f"{inflight} batches in flight ({inflight} evaluators used round-robin; the better of 3 and 6 in an untimed trial "
                  f"before the timed steps); one event wait per batch",
           "batches_in_flight": inflight, "trial_board_evals_per_sec": {str(n): v for n, v in trial.items()},
           "ragged_copies_completed_by_a_second_copy": e2e_short}
    e2e["d2h_ceiling_gbs_per_gpu"] = ceil_gbs
    e2e["d2h_achieved_gbs_per_gpu"] = e2e_d2h * (e2e_v / world / B) / 1e9
    extra = {}
    v32, d32, _ = e2e_pipelined(3, wire="f32", with_mask=True)
    extra["e2e_f32_wire_with_mask_and_pawn"] = {"value": v32, "unit": "board-evals/s", "d2h_bytes_per_step": d32,
                                                "api": "the round-1 result set (f32 ragged priors + value + legal mask + pawn list), three in flight"}
    sync_v, sync_d2h = e2e_sync(dense=False)
    dense_v, dense_d2h = e2e_sync(dense=True)
    extra["e2e_one_batch_in_flight"] = {"value": sync_v, "unit": "board-evals/s", "d2h_bytes_per_step": sync_d2h,
                                        "api": "HostLeafEvaluator.evaluate (synchronous, one caller): aq_leaf_eval_host_compact"}
    extra["e2e_dense_priors"] = {"value": dense_v, "unit": "board-evals/s", "d2h_bytes_per_step": dense_d2h,
                                 "api": "aq_leaf_eval_host (synchronous): dense priors [B,209]"}
    cpu_ok = rank == 0 and world == 1 and not args.skip_cpu

    if not args.skip_extra:
        # ---- the fp32 (FFMA) leaf evaluation beside the bf16 headline --------------------------------------------------------
        if prec == 1:
            ms32, _ = timed(lambda i: step(i, 0, None), max(3, K // 4), 2)
            extra["leaf_eval_fp32"] = {"value": world * B / (ms32 * 1e-3), "unit": "board-evals/s", "ms_per_step": ms32,
                                       "note": "the same step with precision fp32 (FFMA trunk and heads): the arithmetic of the reference"}
        # ---- legal mask, BASELINE configs[1]: 1M positions resident in HBM ----------------------------------------------------
        M = 1_000_000
        big = positions.random_positions(M, seed=101 + rank, games=16384, device=dev)
        bmask = torch.empty((M, 8), dtype=torch.int32, device=dev)
        bpawn = torch.empty((M, 8), dtype=torch.uint8, device=dev)
        bws = torch.empty((L.aq_legal_mask_ws_bytes(M),), dtype=torch.uint8, device=dev)
        ms, _ = timed(lambda i: _lib.check(L.aq_legal_mask_ws(P(big), M, P(bmask), P(bpawn), P(bws), bws.numel(), st), "aq_legal_mask_ws"), 5, 2)
        gbs = BYTES_PER_POSITION_LEGAL * M / (ms * 1e-3) / 1e9
        extra["legal_mask"] = {"value": world * M / (ms * 1e-3), "unit": "positions/s", "ms_per_1M": ms,
                               "config": "BASELINE configs[1]: 1,000,000 random legal positions per GPU (plies 0..61), two-phase kernel pair",
                               "roofline": {"bound": "hbm", "achieved": gbs, "peak": pk["hbm"], "unit": "GB/s", "frac": gbs / pk["hbm"],
                                            "note": "HBM by rule (72 B per position); the kernels are integer-issue bound (DESIGN.md section 4)"},
                               "cpu_baseline": time_cpu_legal_mask() if cpu_ok else None}
        del big, bmask, bpawn, bws

        # ---- training step through the public trainer (forward + loss + backward + gradient all-reduce + Adam), random targets ----
        def train_bench(TB, precision, collective="p2p"):
            torch.manual_seed(0)
            tnet = GNNNetwork().to(dev).train()
            trainer = train_network.FlatTrainer(tnet, rank=rank, world_size=world, precision=precision, collective=collective)
            tb = allpos[:TB].contiguous()
            torch.manual_seed(1)
            pt = torch.softmax(torch.randn(TB, 209, device=dev), 1)
            vt = torch.randint(-1, 2, (TB,), device=dev).float()
            ms, launches = timed(lambda i: trainer.step(tb, pt, vt, TB * world), 20, 5)
            trainer.check()
            # graph replays do not pass through the library's launch counter: the count of the last eagerly run step stands for them
            return ms, (trainer.kernels_per_step if trainer.kernels_per_step is not None else launches / 20)

        tr = {}
        for TB in (256, 4096):
            ms, launches = train_bench(TB, args.precision)
            tf = FLOP_PER_BOARD_FWDBWD * TB / (ms * 1e-3) / 1e12
            tr[f"B{TB}"] = {"value": world * TB / (ms * 1e-3), "unit": "samples/s", "ms_per_step": ms, "kernel_launches_per_step": launches,
                            "roofline": {"bound": "tensor", "achieved": tf, "peak": pk["tensor"], "unit": "TFLOP/s", "frac": tf / pk["tensor"]}}
        if prec == 1:
            ms, _ = train_bench(256, "fp32")
            tr["B256_fp32"] = {"value": world * 256 / (ms * 1e-3), "unit": "samples/s", "ms_per_step": ms}
        if world > 1:  # the checked alternative: same backward kernels, torch.distributed (NCCL) all-reduce + aq_adam_step
            for TB in (256, 4096):
                ms, launches = train_bench(TB, args.precision, "nccl")
                tr[f"B{TB}_nccl_allreduce"] = {"value": world * TB / (ms * 1e-3), "unit": "samples/s", "ms_per_step": ms,
                                               "kernel_launches_per_step": launches}
            # every rank pushes its flat gradient as {value, step tag} words of 8 bytes into its inbox on each of the other ranks
            tr["nvlink_bytes_per_step_per_gpu"] = {"sent": (world - 1) * 251 * 256 * 8, "received": (world - 1) * 251 * 256 * 8}
        tr["config"] = ("BASELINE configs[0] shape (B = 256 per GPU) and a throughput-sized batch (B = 4096 per GPU): FlatTrainer.step = "
                        "aq_gnn_forward(saved) + aq_train_backward_step (loss gradient + heads backward | trunk backward | head weight gradients "
                        "| slot reduction + peer-memory all-reduce + Adam), replayed as one CUDA graph")
        tr["cpu_baseline"] = time_cpu_train() if cpu_ok else None
        extra["train"] = tr

        # ---- lock-step PV-MCTS self-play, WHOLE games (BASELINE configs[3]) and training on that record (configs[4]) ----------
        try:
            G, SIMS = args.mcts_games, args.mcts_sims
            # warm-up = one untimed pass of the same work: module loads and the graph captures for the batch sizes a game passes through
            self_play.play_batch_device(net, G, dev, sims=SIMS, seed=4, policy_dtype=torch.float32)
            barrier()
            t0 = time.perf_counter()
            rec = self_play.play_batch_device(net, G, dev, sims=SIMS, seed=5 + rank, policy_dtype=torch.float32)
            barrier()
            dt = reduce_max(time.perf_counter() - t0)
            tot = torch.tensor([rec["sims"], rec["states"].shape[0], int((rec["flags"] & 1).sum()), int(rec["plies"].sum())],
                               dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tot)
            sims_s = float(tot[0]) / dt
            tf = sims_s * FLOP_PER_BOARD_FWD / 1e12
            extra["mcts"] = {"value": sims_s, "unit": "simulations/s", "seconds": dt, "games": G * world, "sims_per_move": SIMS,
                             "positions": int(tot[1]), "decided_games": int(tot[2]), "mean_plies_per_game": float(tot[3]) / (G * world),
                             "config": f"BASELINE configs[3]: {G} concurrent self-play games per GPU x {SIMS} simulations per move, whole games "
                                       "(start position to win / 116-ply draw), T = 1 sampling; every simulation = select + leaf evaluation "
                                       "(legal mask + GNN) + expand/backup, replayed as one CUDA graph",
                             "roofline": {"bound": "tensor", "achieved": tf, "peak": pk["tensor"], "unit": "TFLOP/s", "frac": tf / pk["tensor"],
                                          "note": "one leaf evaluation (5.79 MFLOP) per simulation; the tree kernels are HBM/latency work"},
                             "cpu_baseline": time_cpu_mcts(SIMS) if cpu_ok else None}
            # configs[4]: the buffer just produced -> one epoch of data-parallel training at the reference's batch size per GPU
            torch.manual_seed(0)
            tnet = GNNNetwork().to(dev).train()
            tnet.train_precision = args.precision
            Mrec = int(rec["states"].shape[0])
            Muse = Mrec // (128 * 1) * 128   # whole batches; every rank trains on its own record, gradients all-reduced (global batch 128 x world)
            if world > 1:
                mm = torch.tensor([Muse], device=dev)
                dist.all_reduce(mm, op=dist.ReduceOp.MIN)
                Muse = int(mm.item())
            trainer = train_network.FlatTrainer(tnet, rank=rank, world_size=world)
            perm = torch.randperm(Muse, device=dev)       # DataLoader(shuffle=True), train_network.py:49
            sp, pp, vv = rec["states"][:Muse], rec["policy"][:Muse], rec["value"][:Muse]
            bp, bt, bv = trainer.inputs(128)
            nsteps = min(Muse // 128, 400)

            def cycle_step(i):  # what train_network.train_on_buffer does per batch: gather into the persistent inputs, one step
                idx = perm[i * 128:(i + 1) * 128]
                torch.index_select(sp, 0, idx, out=bp)
                torch.index_select(pp, 0, idx, out=bt)
                torch.index_select(vv, 0, idx, out=bv)
                trainer.step(bp, bt, bv, 128 * world)

            for i in range(5):
                cycle_step(i)
            barrier()
            t0 = time.perf_counter()
            for i in range(nsteps):
                cycle_step(i)
            barrier()
            dt = reduce_max(time.perf_counter() - t0)
            trainer.check()
            extra["train_cycle"] = {"value": world * 128 * nsteps / dt, "unit": "samples/s", "steps": nsteps, "ms_per_step": dt / nsteps * 1e3,
                                    "config": "BASELINE configs[4]: the self-play record above (device-resident) -> data-parallel training, "
                                              "batch 128 per GPU (train_network.py:15), one all-reduce of the flat gradient per step, wall clock "
                                              "including the host loop"}
            del rec, sp, pp, vv
        except Exception as e:  # the callers of the hot path must not take the headline down with them
            extra["mcts"] = f"unavailable: {type(e).__name__}: {e}"

    if world > 1:
        extra["dp_check"] = dp_check(dev, rank, world)

    clocks = sampler.stop()

    cpu_baseline = None
    if cpu_ok:
        cpu_steps = 3
        v, sec, threads = time_cpu_leaf_eval(B, cpu_steps, 1)
        cpu_baseline = {"value": v, "unit": "board-evals/s", "cores": threads, "kind": "port",
                        "sample": f"{cpu_steps} steps (1 warm-up) of {B} positions: C oracle legal_actions (OpenMP, {threads} threads) + "
                                  f"torch CPU GNN forward + legal renorm; {sec:.1f} s per step"}

    if rank == 0:
        line = {
            "metric": "gnn_board_evals_per_sec", "value": value_main, "unit": "board-evals/s", "n_gpus": world,
            "steps": K, "warmup": Wm, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32" if prec == 0 else "bf16", "data": "synthetic",
            "config": {"workload": "leaf_eval: BASELINE configs[2], batched predict (legal mask + graph + GNN forward + legal "
                                   "renorm) on random legal 9x9 positions, random-init weights",
                       "batch_per_gpu": B, "precision": args.precision, "parallelism": f"independent leaf batches x{world}",
                       "l2": "flushed before every timed launch (256 MiB write, outside the per-launch CUDA events)",
                       "host_numa": numa},
            "roofline": roofline, "kernels": kinfo,
            # the kernels of a step are chained by programmatic dependent launches (prologues overlap the predecessor's tail), so the
            # step is shorter than the sum of its kernels timed alone
            "sum_of_kernels_timed_alone_ms": ksum,
            "cpu_baseline": cpu_baseline, "e2e": e2e,
            "gpu_launches": int(gpu_launches),  # counted by the library (aq_launch_count) over the K timed steps
            "clocks": clocks, "extra": extra,
        }
        print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=16384)
    ap.add_argument("--precision", default=os.environ.get("AQ_PRECISION", "bf16"), choices=["fp32", "bf16"],
                    help="GNN inference arithmetic: bf16 = tcgen05 tensor cores (default), fp32 = FFMA")
    ap.add_argument("--mcts-games", type=int, default=4096)
    ap.add_argument("--mcts-sims", type=int, default=200)
    ap.add_argument("--skip-extra", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last of them returned (priors, value, mask, pawn of rank 0's batch) "
                         "as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path; --impl reference has none")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
