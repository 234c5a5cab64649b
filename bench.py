#!/usr/bin/env python
"""bench.py -- placements/sec for the hot path named by BASELINE.json.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py --gpus N --steps K --warmup W --dump-outputs DIR   (also writes the last timed step's results: dump_outputs)

Workload (config.workload): BASELINE.json configs[3] -- weighted rendezvous placement of 10 M objects x 1024 nodes
(weights u32 in [1,16], seed 7; keys = splitmix stream), id-range sharded one shard per GPU, with the bounded-load
capacity check after ONE exchange of the per-node load counters (cap 1.25, <= 4 rounds).  Weak scaling: every rank
owns a 10 M-object shard, so N GPUs place N x 10 M objects per step.

Policy (config.policy): HRW2, the hierarchical weighted rendezvous with fan-out 2 (DESIGN.md 3.8; ~13 contests per
object, HBM / shared-memory bound).  The flat rendezvous (1024 pair hashes per object, integer-pipe bound by construction)
is timed beside it in `policies`.

A step  = one bounded-load assignment pass over the rank's resident shard (keys already in HBM, results stay in HBM):
          walk kernel with fused per-node histogram -> counter exchange + capacity check (one small kernel) -> 8 bytes to
          the host.
value   = objects placed by all ranks per second over K steps (CUDA events on the engine's stream, max over ranks).
e2e     = the SAME work through the host-buffer C-ABI call rio_cuda_assign_bounded_batch (pinned host keys in, pinned host
          node indices out, histogram + exchange + capacity check included, H2D + D2H inside the timed region).
roofline= the walk kernel alone: algorithmic HBM bytes (12 B/object) / its launch time against the measured HBM peak.
cpu_baseline = this repo's CPU port of the same policy (oracle/rio_oracle.c), all host cores, bounded sample.
--impl reference = the reference's own per-id CPU path (LocalObjectPlacement + Service::get_or_create_placement, restated
          in oracle/directory_model.cpp because rio-rs is Rust and no cargo exists here), all host threads.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_OBJECTS = 10_000_000
N_NODES = 1024
N_SETS = 4  # distinct resident key sets rotated step to step: 4 x 120 MB of traffic > 126 MB of L2
ALGO_BYTES_PER_OBJECT = 12  # 8 B key read + 4 B node index written (SURVEY 8d)
HBM_FALLBACK_GBS = 6650.0
TRIE_BITS = 12
STORM_EVENTS = [("leave", 17), ("join", 1024), ("leave", 3), ("join", 1025), ("leave", 900), ("join", 1026), ("leave", 64), ("join", 1027)]  # SURVEY 8d


def ncu_traffic(name):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of a kernel from the committed ncu capture."""
    p = os.path.join(ROOT, "profiles", name)
    try:
        return float(json.load(open(p))["dram_bytes_per_launch"]), os.path.relpath(p, ROOT)
    except Exception:
        return None, None


def measured(key, fallback):
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            if key in d:
                return float(d[key]), "measured"
        except Exception:
            pass
    return fallback, "fallback"


def bind_to_gpu_numa(local_rank):
    """Pin this rank's threads (and therefore its pinned allocations, first touch) to the CPUs of the NUMA node its GPU hangs
    off: eight ranks pushing 80 MB each across the socket interconnect cost 15 % of the end-to-end rate in round 1."""
    try:
        import torch

        bus = torch.cuda.get_device_properties(local_rank)
        pci = "%04x:%02x:%02x.0" % (getattr(bus, "pci_domain_id", 0), bus.pci_bus_id, bus.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % pci).read())
        if node < 0:
            return None
        cpus = []
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "cpus": len(cpus)}
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)}


def time_loop(p, fn, reps, slot=0):
    p.sync()
    p.event_record(slot)
    for i in range(reps):
        fn(i)
    p.event_record(slot + 1)
    p.sync()
    return p.event_elapsed_ms(slot, slot + 1) / reps


def extra_configs(p, O, n):
    """The other single-GPU configs of BASELINE.json, measured with the same event discipline (N = 1 only):
    C2 = 1 M x 64 weighted rendezvous; C3 = 10 M x 1024, 16-dim affinity cost + argmin on the tensor cores."""
    import rio_rs_b200 as R

    out = {}
    q = R.GpuObjectPlacement(device=p.device_info()["device"])
    addrs, seeds, w = O.synth_nodes(64)
    q.set_nodes(addrs, w)
    s = q.new_set(1 << 20)
    s.synth_keys(0, 1 << 20, 1)
    for solver in ("hrw2", "hrw"):
        q.set_solver(solver, TRIE_BITS)
        for _ in range(5):
            s.assign()
        ms = time_loop(q, lambda i: s.assign(), 50)
        ref = O.assign_hrw2(O.synth_keys(20000, 1), seeds, w, bits=TRIE_BITS) if solver == "hrw2" else O.assign_hrw(O.synth_keys(20000, 1), seeds, w)
        out["C2_rendezvous_1Mx64_" + solver] = {"ms": ms, "placements_per_s": (1 << 20) / (ms * 1e-3), "parity_vs_oracle_20k": bool((s.read(0, 20000) == ref).all()),
                                               "note": "resident keys, weights 1..16"}
    q.set_solver("hrw")
    del s
    M, K = 1024, 16
    addrs, _, _ = O.synth_nodes(M)
    fn = np.random.default_rng(13).uniform(-1, 1, (M, K)).astype(np.float32)
    q.set_nodes(addrs, None, fn)
    s = q.new_set(n)
    s.load_keys(np.arange(n, dtype=np.uint64))
    fo = np.random.default_rng(11).uniform(-1, 1, (n, K)).astype(np.float32)
    s.load_feats(fo)
    for _ in range(3):
        s.assign(True)
    ms = time_loop(q, lambda i: s.assign(True), 10)
    got = s.read(0, 20000)
    idx, cost, gap = O.assign_affinity(fo[:20000], fn, np.ones(M, dtype=np.uint32), threads=8)
    ok = bool(((got == idx) | (gap <= 1e-5 * np.abs(cost) + 1e-12)).all())
    peak, src = measured("bf16_tflops", 1590.0)
    algo = 2 * K * M * n / (ms * 1e-3) / 1e12
    out["C3_affinity_10Mx1024xK16"] = {
        "ms": ms, "placements_per_s": n / (ms * 1e-3), "kernels": "k_affinity_umma (tcgen05/TMEM, bf16x3 split) + k_affinity_resolve",
        "parity_vs_fp64_oracle_20k": ok,
        "roofline": {"bound": "tensor", "achieved": algo, "peak": peak, "unit": "TFLOP/s", "frac": algo / peak, "peak_source": src + " (burst figure: a 1-2 ms kernel timed alone)",
                     "issued_bf16_tflops": 6 * algo, "note": "achieved = ALGORITHMIC 2KM FLOP per object; the kernel issues 6 bf16 cross-term MMAs per product (issued = 6 x achieved)"},
    }
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_indices):
        self.idx = ",".join(str(i) for i in gpu_indices)
        self.proc = None
        self.lines = []

    def start(self):
        if os.environ.get("RIO_BENCH_NO_SMI"):
            return
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", self.idx, "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def mark(self):
        """Samples collected before this call (warm-up) are dropped."""
        self.lines = []

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


def pinned_array(p, nbytes, dtype):
    ptr = C.c_void_p()
    p._ck(p.L.rio_cuda_host_alloc(p.h, nbytes, C.byref(ptr)))
    n = nbytes // np.dtype(dtype).itemsize
    arr = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint8)), shape=(nbytes,)).view(dtype)[:n]
    return arr, ptr


DUMP_MAX_BYTES = 64 << 20   # all ranks' files together
DUMP_SEED = 20240917


def dump_outputs(out_dir, s, passes, rank, world):
    """What a caller of the timed step receives, as .npy files a second build's run can be compared with file for file:
    node_index (the node chosen for every object of the rank's shard, float32; 4294967296 = no node), load_counters (the global
    per-node loads the capacity check saw, float64) and passes (float64).  A shard whose node_index would not fit this rank's
    share of DUMP_MAX_BYTES is written as a seeded sample of it, the sampled object positions in node_index_position (float64).
    With world > 1 every name ends in _rank<r>."""
    os.makedirs(out_dir, exist_ok=True)
    sfx = "_rank%d" % rank if world > 1 else ""
    idx = s.read()
    counters = s.counters()
    budget = DUMP_MAX_BYTES // world - counters.size * 8 - 1024
    out = {"node_index": idx, "load_counters": counters.astype(np.float64), "passes": np.array([passes], dtype=np.float64)}
    if idx.size * 4 > budget:
        pos = np.unique(np.random.default_rng(DUMP_SEED).integers(0, idx.size, budget // 12))
        out["node_index"], out["node_index_position"] = idx[pos], pos.astype(np.float64)
    out["node_index"] = out["node_index"].astype(np.float32)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + sfx + ".npy"), a)


def run_reference(args, rank, world):
    """The reference's own CPU path for this metric: per-id Service::get_or_create_placement over LocalObjectPlacement
    (service.rs:193-254, local.rs:12-68), all host threads, bounded sample per step."""
    if rank != 0:
        return
    from oracle import pyoracle as O

    cores = os.cpu_count() or 1
    per_step = 400_000
    steps = min(args.steps, 50)   # bounded: the whole arm ends within a few minutes whatever K the caller passes
    O.bench_resolve(20_000, N_NODES, cores)  # warm caches / allocator
    for _ in range(max(min(args.warmup, 5), 0)):
        O.bench_resolve(per_step // 4, N_NODES, cores)
    tot_s, tot_n = 0.0, 0
    for k in range(steps):
        s, placed = O.bench_resolve(per_step, N_NODES, cores, first=k * per_step)
        tot_s += s
        tot_n += placed
    v = tot_n / tot_s
    sample = "%d steps x %d fresh ids ('Obj', decimal i) resolved per-id against a %d-member cluster" % (steps, per_step, N_NODES)
    line = {
        "impl": "reference", "metric": "placements/sec", "value": v, "unit": "placements/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * tot_s / max(steps, 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32", "data": "synthetic",
        "config": {"workload": "10M objects x 1024 nodes placement (BASELINE.json configs[3]); reference policy: first server to see the id claims it",
                   "objects_per_step": per_step, "nodes": N_NODES, "steps_run": steps},
        "cpu_baseline": {"value": v, "unit": "placements/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "placements/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "rio-rs is Rust; no cargo/rustc in this image, so this is the C++ restatement oracle/directory_model.cpp of local.rs + service.rs:193-254",
    }
    emit(line)


_JSON_FD = None


def claim_stdout():
    """stdout carries ONE JSON line.  Libraries print there too (NCCL's version banner when the box sets NCCL_DEBUG, nvcc
    notes, torch warnings), so file descriptor 1 is pointed at stderr for the rest of the run and the line is written to
    the original stdout at the end."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_JSON_FD, data)


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--objects", type=int, default=N_OBJECTS, help="objects per rank (default: the BASELINE size)")
    ap.add_argument("--nodes", type=int, default=N_NODES)
    ap.add_argument("--policy", default="hrw2", choices=["hrw2", "hrw"], help="headline solver policy (the other one is timed in `policies`)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the C2/C3/C4-strong/C5 side measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    import __graft_entry__ as G

    if rank == 0:
        G.build()
    if dist:
        dist.barrier()
    import rio_rs_b200 as R
    from rio_rs_b200 import parallel
    from oracle import pyoracle as O  # synthetic-input helpers, the in-bench parity checks and the cpu_baseline leg only

    n, M = args.objects, args.nodes
    p = R.GpuObjectPlacement(device=local_rank)
    info = p.device_info()
    addrs, seeds, w = O.synth_nodes(M)
    p.set_nodes(addrs, w)
    p.set_solver(args.policy, TRIE_BITS)
    if dist:
        parallel.init_comm(p, dist)
    n_global = n * world
    cores = os.cpu_count() or 1

    def oracle_assign(keys, solver, weights=w, threads=8):
        return O.assign_hrw2(keys, seeds, weights, bits=TRIE_BITS, threads=threads) if solver == "hrw2" else O.assign_hrw(keys, seeds, weights, threads=threads)

    def barrier_sync():
        p.sync()
        torch.cuda.synchronize()
        if dist:
            dist.barrier()

    def max_over_ranks(x):
        if not dist:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_ranks_ok(ok):
        if not dist:
            return bool(ok)
        t = torch.tensor([1 if ok else 0], dtype=torch.int32, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(t.item())

    # resident shards: id range [rank*n, (rank+1)*n) of N_SETS independent key streams
    sets = []
    for k in range(N_SETS):
        s = p.new_set(n)
        s.synth_keys(rank * n, n, 1 + k)
        sets.append(s)
    p.sync()

    def step(i):
        return sets[i % N_SETS].assign_bounded(n_global, 5, 4, 4)

    # Steps are issued through the two-halved form of the same call (rio_cuda_set_assign_bounded_begin / _end) with DEPTH passes
    # in flight on different resident sets: pass i+DEPTH is enqueued before pass i's capacity check is read, so the GPU never waits
    # for the host between steps.  Every step is still complete -- walk, histogram, exchange, check, and the spill rounds if the
    # check asks for them -- before its _end returns, and all K of them are inside the timed region.
    DEPTH = max(1, min(N_SETS - 1, int(os.environ.get("RIO_BENCH_DEPTH", "3"))))

    def run_steps(k0, k):
        """Steps k0 .. k0+k-1; returns the passes each one took, in step order."""
        passes = []
        for i in range(k0, k0 + k):
            sets[i % N_SETS].assign_bounded_begin(n_global, 5, 4, 4)
            if i - k0 >= DEPTH:
                passes.append(sets[(i - DEPTH) % N_SETS].assign_bounded_end())
        for i in range(max(k0, k0 + k - DEPTH), k0 + k):
            passes.append(sets[i % N_SETS].assign_bounded_end())
        return passes

    # ONE sampler for the whole job (rank 0 watches every GPU of the run): a poller per rank contends for the driver
    # and showed up as ~0.4 ms per step at N = 8 (profiles/r01_scale_n8.json vs r01_scale_n8_one_sampler.json)
    clocks = ClockSampler(range(world)) if rank == 0 else None
    if clocks:
        clocks.start()
    passes = max([1] + run_steps(0, args.warmup))
    barrier_sync()
    if clocks:
        time.sleep(0.25)   # make sure the sampler is producing before the timed region starts
        clocks.mark()
    barrier_sync()
    l0 = p.launch_count()
    p.event_record(0)
    timed_passes = run_steps(args.warmup, args.steps)
    p.event_record(1)
    barrier_sync()
    passes = max([passes] + timed_passes)
    if args.dump_outputs:   # before anything below reuses the resident sets
        dump_outputs(args.dump_outputs, sets[(args.warmup + args.steps - 1) % N_SETS], timed_passes[-1], rank, world)
    my_ms = p.event_elapsed_ms(0, 1)
    ms_total = max_over_ranks(my_ms)
    per_rank_ms = None
    if dist:   # diagnostics only: every rank's own device time for the same K steps (the line's value uses the max)
        t = torch.zeros(world, dtype=torch.float64, device="cuda")
        t[rank] = my_ms / args.steps
        dist.all_reduce(t)
        per_rank_ms = [round(float(x), 6) for x in t.tolist()]
    launches = p.launch_count() - l0
    ms_per_step = ms_total / args.steps
    value = n_global / (ms_per_step * 1e-3)

    # the dominant kernel alone (walk + fused histogram), same resident inputs, events on its stream
    kreps = max(20, min(args.steps, 2000))
    for i in range(5):
        sets[i % N_SETS].assign()
    kern_ms = time_loop(p, lambda i: sets[i % N_SETS].assign(), kreps, 2)
    if clocks and len(clocks.lines) < 3 * world:   # short runs: keep the same kernel running until a few samples exist
        t_end = time.perf_counter() + 0.5
        while time.perf_counter() < t_end:
            for i in range(50):
                sets[i % N_SETS].assign()
            p.sync()
    clk = clocks.stop() if clocks else None   # covers the timed steps, the kernel-only loop (and the burst above, if any)
    peak, peak_src = measured("hbm_gbs", HBM_FALLBACK_GBS)
    kernel_name = "k_assign_trie" if args.policy == "hrw2" else "k_assign_hrw_v2"
    traffic, traffic_src = ncu_traffic("r02_ncu_trie.json" if args.policy == "hrw2" else "r01_ncu_assign_v3.json") if (n == N_OBJECTS and M == N_NODES) else (None, None)
    achieved_gbs = ALGO_BYTES_PER_OBJECT * n / (kern_ms * 1e-3) / 1e9

    # the headline result against the oracle: the FIRST shard-local 200k objects of set 0 on every rank
    chk = sets[0].read(0, min(n, 200_000))
    parity_ok = all_ranks_ok((chk == oracle_assign(O.synth_keys(len(chk), 1, first=rank * n), args.policy)).all())
    assert parity_ok, "GPU result differs from the oracle"

    # both policies on the same resident inputs (kernel alone + full bounded step)
    policies = {}
    for solver in ("hrw2", "hrw"):
        p.set_solver(solver, TRIE_BITS)
        reps = kreps if solver == "hrw2" else 10
        for i in range(3):
            sets[i % N_SETS].assign()
        k_ms = time_loop(p, lambda i: sets[i % N_SETS].assign(), reps, 2)
        barrier_sync()
        s_ms = max_over_ranks(time_loop(p, lambda i: sets[i % N_SETS].assign_bounded(n_global, 5, 4, 4), reps, 4))   # one call at a time
        ok = bool((sets[0].read(0, 50_000) == oracle_assign(O.synth_keys(50_000, 1, first=rank * n), solver)).all())
        policies[solver] = {"kernel_ms": k_ms, "step_ms_one_call_at_a_time": s_ms, "placements_per_s_step": n_global / (s_ms * 1e-3), "hbm_frac_kernel": ALGO_BYTES_PER_OBJECT * n / (k_ms * 1e-3) / 1e9 / peak,
                            "contests_or_pair_hashes_per_object": (TRIE_BITS + 1) if solver == "hrw2" else M, "parity_vs_oracle_50k": ok}
        if solver == "hrw":
            mix_peak = max(p.bench_mix_rate(4000) for _ in range(3))
            policies[solver]["alu_roofline"] = {"bound": "int-alu", "achieved": n * M / (k_ms * 1e-3), "peak": mix_peak, "unit": "pair-hashes/s", "frac": n * M / (k_ms * 1e-3) / mix_peak,
                                                "peak_source": "rio_cuda_bench_mix_rate: register-only replay of the same IMAD/IMAD/VIMNMX3 mix, measured in this run"}
    p.set_solver(args.policy, TRIE_BITS)
    sets[0].assign_bounded(n_global, 5, 4, 4)   # set 0 holds the headline policy's result again (the e2e leg compares against it)

    # multi-rank bounded rounds where they actually fire: cap 101/100 on a 400k-object shard per rank (passes > 1), every
    # rank's result against the oracle run on the GLOBAL key set -- decisions taken on global counters must agree bit for bit
    multi_rank = None
    if world > 1:
        m_per = 400_000
        t = p.new_set(m_per)
        t.synth_keys(rank * m_per, m_per, 9)
        got_passes = t.assign_bounded(m_per * world, 101, 100, 4)
        gkeys = O.synth_keys(m_per * world, 9)
        if args.policy == "hrw2":
            widx, wcnt, wpass = O.assign_bounded_hrw2(gkeys, seeds, w, 101, 100, 4, bits=TRIE_BITS, threads=max(1, cores // world))
        else:
            widx, wcnt, wpass = O.assign_bounded(gkeys, seeds, w, 101, 100, 4, threads=max(1, cores // world))
        ok = bool((t.read() == widx[rank * m_per:(rank + 1) * m_per]).all() and got_passes == wpass and (t.counters() == wcnt).all())
        multi_rank = {"objects_per_rank": m_per, "cap": "101/100", "passes": got_passes, "oracle_passes": int(wpass), "all_ranks_equal_oracle": all_ranks_ok(ok)}
        del t

    # e2e: host buffers through the C ABI, same work as `value` (H2D + walk + histogram + exchange + check + D2H, chunk-pipelined)
    e2e = None
    if not args.no_e2e:
        hk, hk_ptr = pinned_array(p, n * 8, np.uint64)
        ho, ho_ptr = pinned_array(p, n * 4, np.uint32)
        hk[:] = O.synth_keys(n, 1, first=rank * n)
        ereps = max(5, min(args.steps, 50))
        for _ in range(3):
            p.assign_bounded_batch(hk, n_global, 5, 4, 4, out=ho)
        barrier_sync()
        t0 = time.perf_counter()
        for _ in range(ereps):
            p.assign_bounded_batch(hk, n_global, 5, 4, 4, out=ho)
        p.sync()
        dt = max_over_ranks(time.perf_counter() - t0)
        e2e_ms = 1e3 * dt / ereps
        # the PCIe floor of this box, measured: the 8n-byte key buffer alone, pinned host -> device, no compute
        dkeys = C.c_void_p()
        p._ck(p.L.rio_cuda_dev_alloc(p.h, n * 8, C.byref(dkeys)))
        for _ in range(2):
            p._ck(p.L.rio_cuda_memcpy_h2d(p.h, dkeys, hk_ptr, n * 8))
        p.sync()
        t0 = time.perf_counter()
        for _ in range(5):
            p._ck(p.L.rio_cuda_memcpy_h2d(p.h, dkeys, hk_ptr, n * 8))
        p.sync()
        h2d_ms = (time.perf_counter() - t0) * 1e3 / 5
        p._ck(p.L.rio_cuda_dev_free(p.h, dkeys))
        e2e = {"value": n_global / (e2e_ms * 1e-3), "unit": "placements/s", "h2d_bytes_per_step": 8 * n, "d2h_bytes_per_step": 4 * n,
               "ms_per_step": e2e_ms, "steps": ereps, "h2d_of_the_keys_alone_ms": h2d_ms, "h2d_GBps": 8 * n / (h2d_ms * 1e-3) / 1e9,
               "api": "rio_cuda_assign_bounded_batch (pinned host keys -> pinned host node indices; fused histogram, counter exchange and capacity check included)"}
        # the result that came back over PCIe is the resident result
        assert (ho[:200_000] == sets[0].read(0, 200_000)).all()
        if numa:
            e2e["cpu_binding"] = numa

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        ks = O.synth_keys(min(n, 10_000_000), 1)
        oracle_assign(ks[:200_000], args.policy, threads=cores)
        t0, done = time.perf_counter(), 0
        while time.perf_counter() - t0 < 10.0:   # ~10 s of CPU work on all cores
            oracle_assign(ks, args.policy, threads=cores)
            done += len(ks)
        dt = time.perf_counter() - t0
        cpu = {"value": done / dt, "unit": "placements/s", "cores": cores, "kind": "port",
               "sample": "%d passes over the first %d of the 10M objects x %d nodes, oracle/rio_oracle.c (%s), %d threads, %.1f s" % (
                   done // len(ks), len(ks), M, "orc_assign_hrw2" if args.policy == "hrw2" else "orc_assign_hrw", cores, dt)}
        if args.policy == "hrw2":   # the flat solver on the same cores, for context
            kf = ks[:400_000]
            t0 = time.perf_counter()
            O.assign_hrw(kf, seeds, w, threads=cores)
            cpu["flat_policy_value"] = len(kf) / (time.perf_counter() - t0)

    extra = None
    if not args.no_extra and n == N_OBJECTS:
        extra = {}
        try:
            # C4 as BASELINE.json words it: 10 M objects TOTAL, id-range sharded over the ranks (strong scaling)
            lo, hi = parallel.shard_range(N_OBJECTS, rank, world)
            ts = []
            for k in range(3):
                t = p.new_set(hi - lo)
                t.synth_keys(lo, hi - lo, 1 + k)
                ts.append(t)

            SD = min(DEPTH, len(ts) - 1)   # a set takes one bounded call at a time

            def strong_steps(k):
                for i in range(k):
                    ts[i % 3].assign_bounded_begin(N_OBJECTS, 5, 4, 4)
                    if i >= SD:
                        ts[(i - SD) % 3].assign_bounded_end()
                for i in range(max(0, k - SD), k):
                    ts[i % 3].assign_bounded_end()

            strong_steps(20)
            barrier_sync()
            sreps = max(20, min(args.steps, 2000))
            p.event_record(6)
            strong_steps(sreps)
            p.event_record(7)
            barrier_sync()
            ms = max_over_ranks(p.event_elapsed_ms(6, 7)) / sreps
            ok = all_ranks_ok((ts[0].read(0, min(hi - lo, 100_000)) == oracle_assign(O.synth_keys(min(hi - lo, 100_000), 1, first=lo), args.policy)).all())
            extra["C4_strong_10M_total"] = {"ms_per_step": ms, "placements_per_s": N_OBJECTS / (ms * 1e-3), "objects_per_rank": hi - lo, "steps": sreps, "parity_vs_oracle": ok,
                                            "note": "BASELINE configs[3] as worded: 10 M objects TOTAL, id-range sharded over the ranks; three resident key sets rotated (L2-resident at N >= 2), "
                                                    "%d passes in flight; strong-scaling efficiency = (this at N) / (N x this at N=1)" % SD}
            del ts, t
            # C5: 100 M objects total, the fixed list of 8 join/leave events, one exchange of the counters per event
            lo, hi = parallel.shard_range(100_000_000, rank, world)
            q = R.GpuObjectPlacement(device=local_rank)
            a5, s5, w5 = O.synth_nodes(M + 4)
            q.set_nodes(a5[:M], w5[:M])
            q.set_solver(args.policy, TRIE_BITS)
            if dist:
                parallel.init_comm(q, dist)
            t = q.new_set(hi - lo)
            t.synth_keys(lo, hi - lo, 1)
            t.assign()
            q.sync()
            wl = w5.copy()
            wl[M:] = 0
            if dist:
                dist.barrier()
            t0 = time.perf_counter()
            moved = []
            for ev, j in STORM_EVENTS:
                if ev == "leave":
                    q.node_set_active(j, False)
                    wl[j] = 0
                else:
                    q.node_upsert(a5[j], int(w5[j]))
                    wl[j] = w5[j]
                moved.append(t.rebalance(ev, j))
                t.counters()   # the one exchange of the event
            q.sync()
            wall = max_over_ranks(time.perf_counter() - t0)
            m5 = min(hi - lo, 100_000)
            ok = all_ranks_ok((t.read(0, m5) == (O.assign_hrw2(O.synth_keys(m5, 1, first=lo), s5, wl, bits=TRIE_BITS, threads=8) if args.policy == "hrw2"
                                                 else O.assign_hrw(O.synth_keys(m5, 1, first=lo), s5, wl, threads=8))).all())
            extra["C5_storm_100M_8_events"] = {"wall_ms": wall * 1e3, "objects_total": 100_000_000, "objects_per_rank": hi - lo, "moved_on_rank0": moved,
                                               "state_equals_fresh_assignment_sample": ok, "events": ["%s(%d)" % e for e in STORM_EVENTS]}
            del t, q
            if rank == 0 and world == 1:
                extra.update(extra_configs(p, O, n))
                sys.path.insert(0, os.path.join(ROOT, "tools"))
                import bench_c1

                extra["C1_per_id_lookup_1k_ids_4_nodes"] = bench_c1.run(R, O, device=local_rank)
        except Exception as e:  # the headline line must still be printed
            extra["error"] = repr(e)

    if rank == 0:
        line = {
            "metric": "placements/sec", "value": value, "unit": "placements/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": "10M objects x 1024 nodes weighted-rendezvous placement, id-range shard per GPU, bounded-load check after one exchange of load counters (BASELINE.json configs[3])",
                       "policy": ("hrw2: hierarchical weighted rendezvous, fan-out 2, trie_bits %d (DESIGN.md 3.8)" % TRIE_BITS) if args.policy == "hrw2" else "hrw: flat weighted rendezvous (DESIGN.md 3.4)",
                       "objects_per_gpu": n, "global_objects": n_global, "nodes": M, "weights": "u32 in [1,16], seed 7", "capacity": "1.25", "max_rounds": 4,
                       "passes_run": passes, "passes_in_flight": DEPTH, "l2": "inputs larger than L2: %d resident key sets rotated step to step" % N_SETS, "parallelism": "id-range shard x%d" % world,
                       "parity_vs_oracle_200k_per_rank": parity_ok, "multi_rank_parity": multi_rank, "per_rank_ms_per_step": per_rank_ms, "device": info["name"], "sms": info["sm_count"]},
            "roofline": {"bound": "hbm", "achieved": achieved_gbs, "peak": peak, "unit": "GB/s", "frac": achieved_gbs / peak, "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": kernel_name, "kernel_ms": kern_ms, "algorithmic_bytes_per_launch": ALGO_BYTES_PER_OBJECT * n, "peak_source": peak_src,
                         "note": "12 B/object (8 B key in, 4 B node index out); the walk is bound by the shared-memory data pipe (random trie gathers: 76 % of peak wavefronts over the launch, 83 % while the SMs are active) with the issue slots next (75 %), HBM third (profiles/r02_ncu_trie.json, DESIGN.md 5.4)"
                         if args.policy == "hrw2" else "integer-ALU bound by construction (1024 pair hashes per 12 B); see policies.hrw.alu_roofline"},
            "policies": policies,
            "cpu_baseline": cpu,
            "e2e": e2e,
            "gpu_launches": int(launches),
            "clocks": clk,
            "extra_configs": extra,
        }
        emit(line)
    if dist:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
