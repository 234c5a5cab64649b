"""C1 (BASELINE.json configs[0]): per-id lookups over 1 k synthetic ids, 4-node cluster.  The reference's per-id CPU path
(LocalObjectPlacement restated in C++, SqliteObjectPlacement restated over Python's sqlite3) beside the GPU provider's per-id
calls -- direct (one launch per call behind the handle's mutex), through the coalescing front end at 1 and 16 threads -- and
the batched call the north star adds.  Prints one JSON object.  Importable: run(p_factory) returns the dict."""
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def run(R, O, device=0, n=1000, M=4):
    from oracle.sqlite_model import SqliteDirectoryModel

    out = {"ids": n, "nodes": M}
    s, hits = O.bench_lookup(n, M, 200)
    out["cpu_local_restatement_ns_per_lookup"] = 1e9 * s / (n * 200)
    sm = SqliteDirectoryModel()
    sm.prepare()
    ids = [("Obj", str(i)) for i in range(n)]
    addrs = ["10.0.0.%d:5000" % j for j in range(M)]
    for k, (t, i) in enumerate(ids):
        sm.update(t, i, addrs[k % M])
    t0 = time.perf_counter()
    for _ in range(3):
        for t, i in ids:
            sm.lookup(t, i)
    out["cpu_sqlite_restatement_us_per_lookup"] = 1e6 * (time.perf_counter() - t0) / (3 * n)

    p = R.GpuObjectPlacement(device=device)
    p.set_nodes(addrs)
    keys = p.hash_ids(ids)
    p.update_many(keys, np.arange(n, dtype=np.uint32) % M)
    oids = [R.ObjectId(t, i) for t, i in ids]

    def timed_threads(fn, T, reps=1):
        def work(t):
            for _ in range(reps):
                for k in range(t, n, T):
                    fn(oids[k])
        th = [threading.Thread(target=work, args=(t,)) for t in range(T)]
        t0 = time.perf_counter()
        for x in th:
            x.start()
        for x in th:
            x.join()
        return 1e6 * (time.perf_counter() - t0) / (n * reps)

    p.lookup(oids[0])
    out["gpu_direct_lookup_us_1_thread"] = timed_threads(p.lookup, 1)
    out["gpu_direct_lookup_us_per_op_16_threads"] = timed_threads(p.lookup, 16)
    r = R.Resolver(p, policy="self", self_address=addrs[0], max_batch=256, max_wait_us=20)
    r.lookup(oids[0])
    out["gpu_coalesced_lookup_us_1_thread"] = timed_threads(r.lookup, 1)
    out["gpu_coalesced_lookup_us_per_op_16_threads"] = timed_threads(r.lookup, 16, 4)
    out["gpu_coalesced_lookup_us_per_op_64_threads"] = timed_threads(r.lookup, 64, 8)
    st = r.stats()
    out["coalescing"] = {"calls": st["calls"], "batches": st["batches"], "largest_batch": st["largest_batch"]}
    r.close()
    t0 = time.perf_counter()
    for _ in range(50):
        got = p.lookup_many(keys)
    out["gpu_batched_lookup_ns_per_id_1k_batch"] = 1e9 * (time.perf_counter() - t0) / (50 * n)
    big = np.tile(keys, 1000)
    p.lookup_many(big)
    t0 = time.perf_counter()
    p.lookup_many(big)
    out["gpu_batched_lookup_ns_per_id_1M_batch"] = 1e9 * (time.perf_counter() - t0) / len(big)
    assert (got == np.arange(n) % M).all()
    # the same calls from real threads through the C ABI (the Python threads above serialise on the interpreter lock); the
    # harness is compiled into a temporary directory so that a benchmark run leaves the source tree as it found it (it may be read-only)
    try:
        import subprocess
        import tempfile

        src = os.path.join(ROOT, "tools", "bench_c1.cpp")
        so_dir = os.path.join(ROOT, "rio_rs_b200")
        with tempfile.TemporaryDirectory() as tmp:
            exe = os.path.join(tmp, "bench_c1")
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-pthread", src, "-I" + os.path.join(ROOT, "include"), "-L" + so_dir, "-lrio_cuda",
                                   "-Wl,-rpath," + so_dir, "-o", exe])
            out["c_abi_threads"] = json.loads(subprocess.check_output([exe], timeout=300).decode().strip().splitlines()[-1])
    except Exception as e:  # noqa: BLE001
        out["c_abi_threads"] = {"error": repr(e)}
    out["note"] = ("a per-id call is one GPU round trip (H2D 8 B, launch, D2H, sync): latency-bound; the per-request call sites are meant to go "
                   "through the coalescing front end or the batched calls, where the cost per id falls with the batch size")
    return out


if __name__ == "__main__":
    import __graft_entry__ as G

    G.build()
    import rio_rs_b200 as R
    from oracle import pyoracle as O

    print(json.dumps(run(R, O), indent=1))
