#!/usr/bin/env python
"""PPO-update throughput of the B200 path (BASELINE.json metric: graph-samples/s + achieved HBM GB/s vs roofline).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

A "step" is one PPO minibatch update -- forward + backward of the SGNN policy/value net on 256 rollout graphs per
GPU, gradient reduction, (N>1: NCCL all-reduce of the 55 KB gradient buffer), clip + Adam -- on synthetic
HLG-shaped graphs (BASELINE.json configs[1]; SURVEY.md section 8(d) generator, seed 111).  Weak scaling: 256 graphs
per GPU, global minibatch 256*N.  One JSON line is printed by rank 0; see README/DESIGN.md for the fields.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "ppo_update_graph_samples_per_sec"
UNIT = "graph-samples/s"
BATCH = 256
SEED = 111


def read_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of one k_sgnn<TRAIN> launch from the committed `ncu --set full`
    capture of this workload (profiles/traffic.json; cannot be measured inside a timed run)."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return float(json.load(f)["k_sgnn_train_dram_bytes_per_launch"])
    except Exception:
        return None


def read_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


def dump_outputs(out_dir: str, params, grad, losses):
    """One timed step's results as float32 .npy files: the parameters after the step, the gradient, the loss
    statistics [0..7] of the gradient buffer (include/upb200.h) and the four logged losses."""
    from drl_urban_planning_b200 import _lib
    os.makedirs(out_dir, exist_ok=True)
    g = grad.cpu().numpy()
    arrays = {"params": params.cpu().numpy(), "grad": g[:_lib.UPB_NUM_PARAMS],
              "grad_stats": g[_lib.UPB_STAT_OFFSET:_lib.UPB_STAT_OFFSET + 8], "losses": np.asarray(losses)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


def workload_name(args):
    return "+".join(args.mixed.split(",")) + " mixed" if args.mixed else args.community


def workload_states(args, seed, distinct, pool_minibatches):
    return make_pool(seed, args.community, distinct, pool_minibatches, mixed=args.mixed)


def make_pool(seed: int, community: str, distinct: int, pool_minibatches: int, mixed: str = ""):
    """`pool_minibatches` x 256 states: `distinct` generated graphs tiled (duplicates occupy distinct HBM).
    `mixed` = "a,b": BASELINE.json configs[4], communities alternating inside every minibatch (variable node / edge
    counts, shared caps)."""
    from drl_urban_planning_b200 import synth
    if mixed:
        states, actions = synth.make_mixed_states(seed, mixed.split(","), distinct)
    else:
        states, actions = synth.make_states(seed, community, distinct)
    total = pool_minibatches * BATCH
    reps = (total + distinct - 1) // distinct
    order = np.random.default_rng(seed).permutation(distinct * reps)[:total] % distinct
    return [states[i] for i in order], actions[order]


def cpu_port_step_time(states, actions, flat, steps: int, warmup: int, threads: int):
    """Seconds per PPO minibatch step of the padded eager-PyTorch oracle port (the reference's CPU dataflow)."""
    import torch
    from oracle import torch_port as TP
    torch.set_num_threads(threads)
    n = len(states)
    rng = np.random.default_rng(5)
    adv = torch.tensor(rng.standard_normal((n, 1)).astype(np.float32))
    ret = torch.tensor(rng.standard_normal((n, 1)).astype(np.float32))
    fixed = torch.full((n, 1), -4.0)
    ind = torch.arange(n)
    agent = TP.PortAgent(flat)
    act = torch.tensor(actions)
    times = []
    for k in range(warmup + steps):
        t0 = time.perf_counter()
        b = TP.stack_states(states)                 # tensorfy + batch_data are inside the reference's timed region
        agent.step(b, act, adv, ret, fixed, ind)
        if k >= warmup:
            times.append(time.perf_counter() - t0)
    return float(np.mean(times))


def reference_kind():
    """"reference": the unmodified reference staged under oracle/_ref by oracle/stage_ref.py; "port": the pinned
    oracle restatement of its dataflow (fallback)."""
    try:
        from oracle import ref_runner
        return "reference" if ref_runner.available() else "port"
    except Exception:
        return "port"


def cpu_step_time(kind, states, actions, flat, steps, warmup, threads):
    """Seconds per PPO minibatch step of the CPU arm (tensorfy + losses + backward + clip + Adam, :327-337)."""
    if kind == "reference":
        from oracle import ref_runner
        n_cap, e_cap = states[0][1].shape[0], states[0][2].shape[0]
        return ref_runner.step_time(states, actions, flat, steps, warmup, threads, n_cap, e_cap)
    return cpu_port_step_time(states, actions, flat, steps, warmup, threads)


def best_cpu_threads(states, actions, flat, cores: int, kind: str = "port"):
    """The reference prescribes OMP_NUM_THREADS=1 (README.md:22-25) but the update path is faster with more threads;
    SURVEY 8(d): time several settings and use the fastest as "reference CPU".  Probe on 32 graphs."""
    cands = sorted({1, min(cores, 8), min(cores, 16), min(cores, 32), min(cores, 64), cores})
    best, best_t = cands[0], float("inf")
    for th in cands:
        t = cpu_step_time(kind, states[:32], actions[:32], flat, 1, 1, th)
        if t < best_t:
            best, best_t = th, t
    return best, best_t / 32


def run_reference(args):
    """--impl reference: the reference's own CPU PyTorch update step on the host cores, same metric / config: the
    UNMODIFIED reference staged under oracle/_ref (kind "reference"), else the pinned oracle port (kind "port")."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from drl_urban_planning_b200 import params as PL
    cores = os.cpu_count() or 1
    kind = reference_kind()
    states, actions = workload_states(args, SEED, min(args.distinct, BATCH), 1)
    flat = PL.default_init(SEED)
    # bounded sample: shrink the per-step sample so the whole run ends within a few minutes
    threads, per_graph = best_cpu_threads(states, actions, flat, cores, kind)
    budget = 150.0
    sample = int(max(16, min(BATCH, budget / max(per_graph * (args.steps + args.warmup), 1e-9))))
    t = cpu_step_time(kind, states[:sample], actions[:sample], flat, args.steps, args.warmup, threads)
    value = sample / t
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{workload_name(args)} PPO minibatch update, padded eager PyTorch on CPU ("
                               + ("unmodified reference staged under oracle/_ref" if kind == "reference" else
                                  "oracle port of the reference dataflow") + f"), {sample} graphs per step",
                   "global_batch": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind, "host_cores": cores,
                         "sample": f"{args.steps} steps x {sample} {args.community} graphs, torch threads={threads} "
                                   f"(fastest of 1/8/16/32/64/{cores})"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--community", default="hlg")
    ap.add_argument("--distinct", type=int, default=512, help="distinct generated graphs per rank (tiled to the pool)")
    ap.add_argument("--pool", type=int, default=16, help="minibatches resident in HBM (16 x 11.5 MB > 126 MB L2)")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--nccl-exchange", action="store_true", help="multi-GPU: all-reduce the gradients with NCCL instead of the in-kernel peer exchange")
    ap.add_argument("--mixed", default="", help='BASELINE configs[4]: "hlg_concept,dhm_concept" alternating in every minibatch')
    ap.add_argument("--mode", default="weak", choices=["weak", "strong", "buffer"],
                    help="weak: 256 graphs per GPU per step (global 256*N); strong: global minibatch 256 split over the "
                         "GPUs (the reference's update sequence); buffer: BASELINE configs[3], an 8192-graph buffer "
                         "sharded over the GPUs, walked in global minibatches of 256*N")
    ap.add_argument("--iter-states", type=int, default=25000,
                    help="e2e_iteration leg (N=1): rollout states of one whole update_params iteration (0 = skip)")
    ap.add_argument("--tiles", default="f32", choices=["f32", "bf16"],
                    help="bf16: the labelled NON-PARITY build with bf16-rounded single-pass tensor-core tiles (configs[2])")
    ap.add_argument("--padded-gpu", action="store_true",
                    help="also time the padded eager PyTorch dataflow (reference layout, oracle/_ref or port) on this GPU: "
                         "the padded-layout comparator of configs[4]")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write what the last timed step returned (parameters after the step, "
                         "gradient, loss statistics, losses) as DIR/<name>.npy; the inputs are seeded, so two builds "
                         "run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the B200 path (--impl b200)")
    args.warmup = max(args.warmup, 3)
    if args.tiles == "bf16":
        os.environ["UPB_LIB"] = os.path.join(ROOT, "drl_urban_planning_b200", "libupb200_bf16.so")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from drl_urban_planning_b200 import _lib, params as PL
    from drl_urban_planning_b200.engine import Engine
    from drl_urban_planning_b200.packing import pack_states

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    # host side of the end-to-end path: this rank's packer threads and pinned staging buffers on the GPU's NUMA node
    from drl_urban_planning_b200.engine import bind_host_to_gpu_node
    numa = bind_host_to_gpu_node(dev)

    # ---- workload: resident pool of minibatches, larger than L2
    t0 = time.time()
    global BATCH
    GLOBAL = BATCH * world if args.mode != "strong" else BATCH            # graphs per optimiser step, all GPUs
    if args.mode == "strong":
        BATCH = max(1, BATCH // world)                                    # per-GPU shard of the global 256
    if args.mode == "buffer":
        args.pool = max(1, 8192 // GLOBAL)                                # 8192 graphs in total, 8192/N per GPU
    states, actions = workload_states(args, SEED + rank, args.distinct, args.pool)
    total = len(states)
    blob = pack_states(states).to(dev)
    rng = np.random.default_rng(SEED + 1000 * rank)
    adv = torch.as_tensor(rng.standard_normal(total).astype(np.float32), device=dev)
    ret = torch.as_tensor(rng.standard_normal(total).astype(np.float32), device=dev)
    exps = torch.ones(total, dtype=torch.float32, device=dev)
    act = torch.as_tensor(actions, device=dev)
    flat = PL.default_init(SEED)
    eng = Engine(dev, blob.n_cap, blob.e_cap)
    params = torch.as_tensor(flat, device=dev).clone()
    # old log-probs from perturbed weights so that importance ratios straddle the clip range
    pert = params * (1.0 + 0.05 * torch.randn(params.shape, device=dev, generator=torch.Generator(dev).manual_seed(3)))
    _, fixed, _ = eng.forward(blob, pert, act)
    info = blob.info.astype(np.int64)
    cost = Engine.graph_cost(info)      # cycles model fitted to tools/phase_times.py
    mb_ids = []
    for m in range(args.pool):
        ids = np.arange(m * BATCH, (m + 1) * BATCH)
        ids = eng.balance_ids(ids, cost)                        # static schedule: long graph + short graph per CTA
        mb_ids.append(torch.as_tensor(ids.astype(np.int32), device=dev))
    balg_mb = np.array([(1208 * info[m * BATCH:(m + 1) * BATCH, 0] + 42 * info[m * BATCH:(m + 1) * BATCH, 1] + 1300).sum()
                        for m in range(args.pool)], dtype=np.float64)
    grad = eng.new_grad_buffer()
    gB, gI = GLOBAL, GLOBAL
    # multi-GPU: the ranks' gradient sums are exchanged inside the step kernel through peer memory (NVLink) when the
    # peers' buffers can be mapped; --nccl-exchange keeps one ncclAllReduce + upb_apply per step instead
    fused_exchange = world > 1 and not args.nccl_exchange and eng.connect_peers()
    setup_s = time.time() - t0

    def step(i):
        if world == 1:      # gradient + cross-CTA reduction + Adam in one launch
            eng.ppo_step(blob, params, act, adv, ret, fixed, exps, 1.0 / gB, 1.0 / gI, ids=mb_ids[i % args.pool], out=grad)
            return
        if fused_exchange and eng.next_step_fused():      # cross-rank sum inside the kernel (peer memory), one launch
            eng.ppo_step(blob, params, act, adv, ret, fixed, exps, 1.0 / gB, 1.0 / gI, ids=mb_ids[i % args.pool], out=grad)
            return
        eng.ppo_grad(blob, params, act, adv, ret, fixed, exps, 1.0 / gB, 1.0 / gI, ids=mb_ids[i % args.pool], out=grad)
        dist.all_reduce(grad, op=dist.ReduceOp.SUM)
        eng.apply(params, grad)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        step(i)
    barrier()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
        time.sleep(0.15)
    launches0 = eng.launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for i in range(args.steps):
        step(args.warmup + i)
    ev1.record()
    barrier()
    ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    total_ms = float(ms.item())
    launches = eng.launches - launches0
    losses = eng.read_losses(grad)          # of the last timed step
    # what the last timed step returned, kept before the steps below move the parameters on
    last = (params.clone(), grad.clone()) if args.dump_outputs else None
    # the timed region lasts a few ms, too short for nvidia-smi: keep the same load for ~1 s more (same count on every
    # rank) so the clock / throttle record describes this workload
    for i in range(int(min(20000, max(0.0, 1000.0 / max(total_ms / args.steps, 1e-3))))):
        step(args.warmup + i)
    torch.cuda.synchronize()
    clk = clocks.stop() if rank == 0 else None
    value = GLOBAL * args.steps / (total_ms * 1e-3)
    assert all(np.isfinite(losses)), losses

    # ---- N > 1: correctness of the exchange, visible in the bench line (not just finite losses).
    #  (a) parameters bit-identical on all ranks after the timed steps;
    #  (b) one more step on a 32-graph-per-rank check minibatch through the product path, against rank 0 recomputing
    #      the gradient of the SAME global minibatch alone (every rank's check blob gathered to rank 0, upb_ppo_grad on
    #      each with the global 1/B, summed).
    selfcheck = None
    if world > 1:
        flatp = params.clone()
        gathered = [torch.empty_like(flatp) for _ in range(world)]
        dist.all_gather(gathered, flatp)
        identical = all(torch.equal(gathered[0], g) for g in gathered)
        CK = min(32, BATCH)
        ck_states = states[:CK]
        ck_blob = pack_states(ck_states, blob.n_cap, blob.e_cap).to(dev)
        ck_side = torch.stack([adv[:CK], ret[:CK], fixed[:CK], exps[:CK]])
        ck_act = act[:CK].contiguous()
        p0 = params.clone()
        g_prod = eng.new_grad_buffer()
        if fused_exchange and eng.next_step_fused():
            eng.ppo_step(ck_blob, params, ck_act, ck_side[0], ck_side[1], ck_side[2], ck_side[3], 1.0 / (CK * world),
                         1.0 / (CK * world), out=g_prod)
        else:
            eng.ppo_grad(ck_blob, params, ck_act, ck_side[0], ck_side[1], ck_side[2], ck_side[3], 1.0 / (CK * world),
                         1.0 / (CK * world), out=g_prod)
            dist.all_reduce(g_prod, op=dist.ReduceOp.SUM)
            eng.apply(params, g_prod)
        nbmax = torch.tensor([ck_blob.nbytes], device=dev)
        dist.all_reduce(nbmax, op=dist.ReduceOp.MAX)
        pad = torch.zeros(int(nbmax.item()), dtype=torch.uint8, device=dev)
        pad[:ck_blob.nbytes] = ck_blob.dev[:ck_blob.nbytes]
        blobs = [torch.empty_like(pad) for _ in range(world)]
        sides = [torch.empty_like(ck_side) for _ in range(world)]
        acts = [torch.empty_like(ck_act) for _ in range(world)]
        dist.all_gather(blobs, pad); dist.all_gather(sides, ck_side); dist.all_gather(acts, ck_act)
        if rank == 0:
            from drl_urban_planning_b200.packing import PackedGraphs
            eng1 = Engine(dev, blob.n_cap, blob.e_cap)
            tot = torch.zeros(_lib.UPB_NUM_PARAMS, dtype=torch.float64, device=dev)
            for r in range(world):
                pb = PackedGraphs(None, int(blobs[r].numel()), CK, blob.n_cap, blob.e_cap)
                pb.dev = blobs[r]
                gr = eng1.ppo_grad(pb, p0, acts[r], sides[r][0], sides[r][1], sides[r][2], sides[r][3],
                                   1.0 / (CK * world), 1.0 / (CK * world))
                tot += gr[:_lib.UPB_NUM_PARAMS].double()
            got = g_prod[:_lib.UPB_NUM_PARAMS].double()
            err = float((got - tot).abs().max() / tot.abs().max().clamp_min(1e-30))
            selfcheck = {"ranks_identical": bool(identical), "grad_vs_single_rank_rel": err,
                         "check_minibatch": f"{CK} graphs per rank, global {CK * world}", "pass": bool(identical and err < 1e-4)}
            eng1.close()
        torch.cuda.synchronize()

    # ---- roofline of the dominant kernel (fused SGNN fwd+bwd), CUDA events on the launching stream
    eng.profile(True)
    for i in range(args.steps):
        step(args.warmup + i)
    kms, kn = eng.profile_read()
    eng.profile(False)
    k_avg_ms = kms / max(kn, 1)
    balg = float(balg_mb[[(args.warmup + i) % args.pool for i in range(args.steps)]].mean())
    peak, peak_src = read_peaks()
    achieved = balg / (k_avg_ms * 1e-3) / 1e9

    # ---- end to end: host states (reference layout) -> pack -> H2D -> step -> D2H losses, every step
    e2e = None
    if not args.skip_e2e:
        from drl_urban_planning_b200.packing import pack_states as pk
        host_adv = torch.as_tensor(rng.standard_normal(BATCH).astype(np.float32)).pin_memory()
        host_ret = torch.as_tensor(rng.standard_normal(BATCH).astype(np.float32)).pin_memory()
        host_fix = torch.full((BATCH,), -4.0).pin_memory()
        host_exp = torch.ones(BATCH).pin_memory()
        host_side = torch.cat([torch.zeros(BATCH * 2), host_adv, host_ret, host_fix, host_exp]).pin_memory()
        # Three-stage pipeline, one step deep per stage: the host packer (C, releases the GIL, persistent worker pool)
        # fills the pinned buffer of step i+2 while the copy stream uploads step i+1 and the GPU works on step i.
        # Every step's blob and per-sample arrays still cross PCIe inside the timed region and every step ends with a
        # D2H read of its losses.
        from concurrent.futures import ThreadPoolExecutor
        cap = int(blob.nbytes / args.pool * 1.3)
        host_bufs = [torch.empty(cap, dtype=torch.uint8).pin_memory() for _ in range(2)]
        side_bufs = [host_side.clone().pin_memory() for _ in range(2)]
        dev_bufs = [torch.empty(cap, dtype=torch.uint8, device=dev) for _ in range(2)]
        dev_sides = [torch.empty_like(host_side, device=dev) for _ in range(2)]
        copy_stream = torch.cuda.Stream(device=dev)
        ev_h2d = [torch.cuda.Event() for _ in range(2)]      # upload of the buffer pair finished
        ev_done = [torch.cuda.Event() for _ in range(2)]     # the step that read the device buffers finished
        for ev in ev_h2d + ev_done:
            ev.record()
        n_e2e = max(3, min(args.steps, 20))
        h2d = 0
        # the ranks of one node share its host cores: each packer gets its share (0 = all CPUs of this process, <= 32)
        local_world = int(os.environ.get("LOCAL_WORLD_SIZE", world))
        sharers = local_world if numa is None else -(-local_world // numa[2])       # ranks that share these CPUs
        pack_threads = 0 if sharers <= 1 else max(2, min(32, len(os.sched_getaffinity(0)) // sharers))
        pool_ex = ThreadPoolExecutor(1)

        def pack_job(i):
            j = i & 1
            ev_h2d[j].synchronize()                                  # the previous upload from this pinned buffer is over
            lo = (i % args.pool) * BATCH
            b = pk(states[lo:lo + BATCH], blob.n_cap, blob.e_cap, threads=pack_threads, out_host=host_bufs[j])
            side_bufs[j][:BATCH * 2].copy_(torch.from_numpy(actions[lo:lo + BATCH].reshape(-1)))
            return b

        def upload(i):
            j = i & 1
            b = pending.pop(i).result()
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(ev_done[j])                   # step i-2 no longer reads these device buffers
                b.to(dev, out=dev_bufs[j])
                dev_sides[j].copy_(side_bufs[j], non_blocking=True)  # actions | adv | ret | old log-probs | exps: one copy
                ev_h2d[j].record(copy_stream)
            return b

        pending = {0: pool_ex.submit(pack_job, 0)}
        uploaded = {0: upload(0)}
        pending[1] = pool_ex.submit(pack_job, 1)

        def e2e_step(i):
            nonlocal h2d
            j = i & 1
            pending[i + 2] = pool_ex.submit(pack_job, i + 2)          # host packing two steps ahead (queued behind i+1)
            uploaded[i + 1] = upload(i + 1)                           # H2D of the next step, on the copy stream
            b = uploaded.pop(i)
            side = dev_sides[j]
            d = [side[:BATCH * 2]] + [side[BATCH * (2 + q):BATCH * (3 + q)] for q in range(4)]
            torch.cuda.current_stream().wait_event(ev_h2d[j])
            if world == 1:
                eng.ppo_step(b, params, d[0], d[1], d[2], d[3], d[4], 1.0 / gB, 1.0 / gI, out=grad)
            else:
                if fused_exchange and eng.next_step_fused():
                    eng.ppo_step(b, params, d[0], d[1], d[2], d[3], d[4], 1.0 / gB, 1.0 / gI, out=grad)
                else:
                    eng.ppo_grad(b, params, d[0], d[1], d[2], d[3], d[4], 1.0 / gB, 1.0 / gI, out=grad)
                    dist.all_reduce(grad, op=dist.ReduceOp.SUM)
                    eng.apply(params, grad)
            ev_done[j].record()
            eng.read_losses(grad)                                     # D2H of the step's result (synchronises)
            h2d = b.nbytes + 4 * (BATCH * 2 + BATCH * 4)

        for i in range(2):
            e2e_step(i)
        barrier()
        t1 = time.perf_counter()
        for i in range(n_e2e):
            e2e_step(2 + i)
        barrier()
        dt = torch.tensor([time.perf_counter() - t1], device=dev)
        for f in pending.values():
            f.result()
        torch.cuda.synchronize()
        pool_ex.shutdown()
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        e2e = {"value": BATCH * world * n_e2e / float(dt.item()), "unit": UNIT, "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": 32, "steps": n_e2e,
               "path": "reference-layout host states -> upb_pack_fill -> pinned -> H2D (copy stream) -> upb_ppo_step (N > 1 without peer access: upb_ppo_grad, all-reduce, upb_apply) -> D2H losses; "
                       "packer, upload and step of consecutive minibatches overlap"}

    # ---- end to end, the case the product runs: ONE WHOLE update_params iteration (urban_planning_agent.py:248-361) from
    # reference-layout host lists: pack once, upload once, value / fixed-log-prob sweep, GAE, epochs x floor(T/B)
    # optimiser steps, loss read-back per epoch
    iteration = None
    if rank == 0 and world == 1 and args.iter_states > 0 and args.mode == "weak":
        from drl_urban_planning_b200.ppo import PPOUpdater
        T = args.iter_states
        reps = (T + len(states) - 1) // len(states)
        it_states = (states * reps)[:T]
        it_actions = np.concatenate([actions] * reps)[:T]
        rng_i = np.random.default_rng(9)
        rewards = rng_i.standard_normal(T).astype(np.float32)
        masks = np.ones(T, np.float32); masks[99::100] = 0.0
        up = PPOUpdater(flat, blob.n_cap, blob.e_cap, dev, opt_num_epochs=4, mini_batch_size=256,
                        clip_mode=_lib.CLIP_REFERENCE, process_group=None)
        np.random.seed(1)
        secs = []
        for k in range(2):                       # first pass allocates the pinned / device buffers; second is timed
            torch.cuda.synchronize(); t1 = time.perf_counter()
            res = up.update_params(it_states, it_actions, rewards, masks)
            torch.cuda.synchronize(); secs.append(time.perf_counter() - t1)
        nsteps = 4 * (T // 256)
        iteration = {"states": T, "epochs": 4, "mini_batch_size": 256, "optimiser_steps": nsteps, "seconds": secs[1],
                     "first_call_seconds": secs[0], "graph_samples_per_s": nsteps * 256 / secs[1],
                     "h2d_bytes": int(up.blob.nbytes), "total_loss": float(res["total_loss"]),
                     "path": "reference-layout host lists -> upb_pack_plan_fill chunk by chunk into pinned memory, each chunk's "
                             "H2D copies overlapping the next chunk's packing -> upb_forward sweep -> upb_gae -> "
                             "4 x floor(T/256) upb_ppo_step (next epoch's host work overlapped) -> loss statistics read back "
                             "once per epoch"}
        del up, it_states
        torch.cuda.empty_cache()

    # ---- CPU baseline beside it (rank 0, N=1): oracle port of the reference's padded eager dataflow
    cpu = None
    if rank == 0 and world == 1 and not args.skip_cpu:
        cores = os.cpu_count() or 1
        sample = BATCH
        kind = reference_kind()
        threads, _ = best_cpu_threads(states, actions, flat, cores, kind)
        tstep = cpu_step_time(kind, states[:sample], actions[:sample], flat, 3, 1, threads)
        cpu = {"value": sample / tstep, "unit": UNIT, "cores": threads, "kind": kind, "host_cores": cores,
               "sample": f"3 steps (after 1 warm-up) x {sample} {workload_name(args)} graphs padded to "
                         f"{blob.n_cap}/{blob.e_cap}, torch threads={threads} (fastest of 1/8/16/32/64/{cores})"}
        if iteration is not None:
            # the same whole iteration on the CPU arm: its minibatch steps at the measured step time plus its two
            # pre-pass sweeps (forward only ~ 1/3 of a step each) -- an estimate, a full run would take minutes
            nsteps = iteration["optimiser_steps"]
            iteration["cpu_arm_estimate_s"] = tstep * (nsteps + 2 * (iteration["states"] / BATCH) / 3.0)
            iteration["speedup_vs_cpu_arm_estimate"] = iteration["cpu_arm_estimate_s"] / iteration["seconds"]

    # ---- padded-layout comparator (configs[4] "padded-CSR vs segmented"): the reference's padded eager dataflow on THIS
    # GPU (what `train.py --use_nvidia_gpu` runs), measured as a baseline leg like cpu_baseline
    padded = None
    if rank == 0 and world == 1 and args.padded_gpu:
        from oracle import torch_port as TP
        n_p = min(BATCH, 128)
        agent = TP.PortAgent(flat, device=dev)
        if agent is not None:
            rngp = np.random.default_rng(5)
            tt = lambda x: torch.tensor(x, device=dev)
            adv_p = tt(rngp.standard_normal((n_p, 1)).astype(np.float32)); ret_p = tt(rngp.standard_normal((n_p, 1)).astype(np.float32))
            fix_p = torch.full((n_p, 1), -4.0, device=dev); ind_p = torch.arange(n_p, device=dev); act_p = tt(actions[:n_p])
            ts = []
            for k in range(5):
                torch.cuda.synchronize(); t1 = time.perf_counter()
                b = TP.stack_states(states[:n_p], device=dev)
                agent.step(b, act_p, adv_p, ret_p, fix_p, ind_p)
                torch.cuda.synchronize()
                if k >= 2:
                    ts.append(time.perf_counter() - t1)
            padded = {"value": n_p / float(np.mean(ts)), "unit": UNIT, "layout": f"padded (B, {blob.n_cap}, ...) / (B, {blob.e_cap}, ...) eager PyTorch on the GPU",
                      "sample": f"3 steps x {n_p} graphs", "segmented_over_padded": None}

    if rank == 0:
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "strong" if args.mode == "strong" else "weak", "vs_baseline": None,
            "dtype": "f32" if args.tiles == "f32" else "f32 with bf16-rounded single-pass tensor-core tiles (NOT parity-grade)",
            "data": "synthetic",
            "config": {"workload": f"{workload_name(args)} (cfg {workload_name(args)}), PPO minibatch update, {BATCH} rollout graphs per GPU "
                                   f"per step, caps {blob.n_cap}/{blob.e_cap}, mean n={info[:, 0].mean():.0f} e={info[:, 1].mean():.0f}"
                                   + (", 8192-graph buffer sharded over the GPUs" if args.mode == "buffer" else ""),
                       "mode": args.mode, "global_batch": GLOBAL, "parallelism": f"dp{world}",
                       "gradient_exchange": ("none (one GPU)" if world == 1 else
                                             "inside the step kernel, peer memory over NVLink" if fused_exchange else
                                             "ncclAllReduce of the 55 KB gradient buffer + upb_apply"),
                       "l2_policy": (f"inputs larger than L2: {args.pool} resident minibatches = {blob.nbytes / 1e6:.0f} MB cycled"
                                     if blob.nbytes > 130e6 else
                                     f"{args.pool} resident minibatches = {blob.nbytes / 1e6:.0f} MB per GPU cycled (this mode's "
                                     f"working set is smaller than L2 by definition)")},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": read_traffic(), "kernel": "k_sgnn<TRAIN>", "kernel_ms": k_avg_ms,
                         "algorithmic_bytes_per_launch": balg, "peak_source": peak_src,
                         "kernel_share_of_step": k_avg_ms / (total_ms / args.steps)},
            "cpu_baseline": cpu, "e2e": e2e, "e2e_iteration": iteration, "multi_gpu_selfcheck": selfcheck,
            "padded_comparator": padded, "gpu_launches": int(launches), "clocks": clk,
            "losses_last_step": [float(x) for x in losses], "setup_s": setup_s,
            "host_numa": None if numa is None else {"node": numa[0], "cpus": len(numa[1])},
        }
        if padded is not None:
            padded["segmented_over_padded"] = value / padded["value"]
        if last is not None:
            dump_outputs(args.dump_outputs, last[0], last[1], losses)
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
