"""GPU parity tests (run under gpurun): every call goes through the C ABI of librio_cuda.so and is compared with the
CPU oracle on the same seeded inputs.  Integer / index work is bit-exact; the float-cost path's contract (DESIGN.md 3.6) is
checked in tests/test_gpu_affinity.py, the affinity tests here are the older 1e-5-relative ones on well-conditioned inputs.

Directory tests restate the reference's own tests against the GPU provider, exactly as a `mod gpu { ... }` block in
rio-rs/tests/object_placement_backend.rs would.
"""
import os
import random

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

NONE = 0xFFFFFFFF


@pytest.fixture(scope="module")
def gp():
    from rio_rs_b200 import build

    build.build()
    import rio_rs_b200 as R

    return R


def provider(gp, **kw):
    return gp.GpuObjectPlacement(**kw)


# ---- directory semantics: the reference's known-answer tests ------------------------------------------------
def test_no_placement(gp):
    """rio-rs/tests/object_placement_backend.rs:11-16"""
    p = provider(gp)
    p.prepare()
    assert p.lookup(gp.ObjectId.new("obj", "1")) is None


def test_save_and_load(gp):
    """rio-rs/tests/object_placement_backend.rs:18-34"""
    p = provider(gp)
    p.prepare()
    p.update(gp.ObjectPlacementItem.new(gp.ObjectId.new("obj", "1"), "0.0.0.0:8888"))
    assert p.lookup(gp.ObjectId.new("obj", "1")) == "0.0.0.0:8888"
    p.clean_server("0.0.0.0:8888")
    assert p.lookup(gp.ObjectId.new("obj", "1")) is None


def test_provider_is_clonable(gp):
    """rio-rs/src/object_placement/local.rs:75-114"""
    p = provider(gp)
    q = p.clone()
    p.update(gp.ObjectPlacementItem.new(gp.ObjectId("test", "1"), "0.0.0.0:80"))
    assert p.lookup(gp.ObjectId("test", "1")) is not None
    assert q.lookup(gp.ObjectId("test", "1")) is not None
    q.clean_server("0.0.0.0:80")
    assert p.lookup(gp.ObjectId("test", "1")) is None
    assert q.lookup(gp.ObjectId("test", "1")) is None


def test_overwrite_then_clean(gp):
    """rio-rs/src/object_placement/sqlite.rs:149-193"""
    p = provider(gp)
    p.update(gp.ObjectPlacementItem(gp.ObjectId("Test", "1"), "0.0.0.0:5000"))
    p.update(gp.ObjectPlacementItem(gp.ObjectId("Test", "1"), "0.0.0.0:5001"))
    assert p.lookup(gp.ObjectId("Test", "1")) == "0.0.0.0:5001"
    p.clean_server("0.0.0.0:5000")
    assert p.lookup(gp.ObjectId("Test", "1")) == "0.0.0.0:5001"
    p.clean_server("0.0.0.0:5001")
    assert p.lookup(gp.ObjectId("Test", "1")) is None
    p.clean_server("1.2.3.4:1")  # never-seen address: no-op, not an error


def test_update_none_and_remove(gp):
    """local.rs:34-38 and :60-68"""
    p = provider(gp)
    oid = gp.ObjectId("obj", "1")
    p.update(gp.ObjectPlacementItem(oid, "0.0.0.0:1"))
    p.update(gp.ObjectPlacementItem(oid, None))
    assert p.lookup(oid) is None and p.directory_len()[0] == 0
    p.update(gp.ObjectPlacementItem(oid, "0.0.0.0:1"))
    p.remove(oid)
    p.remove(oid)
    assert p.lookup(oid) is None


def test_random_ops_match_directory_model(gp, oracle):
    """String-level provider vs the LocalObjectPlacement restatement on a random op sequence."""
    rng = random.Random(3)
    p, m = provider(gp), oracle.DirectoryModel()
    addrs = ["10.0.0.%d:5000" % j for j in range(5)]
    ids = [("T%d" % (i % 3), str(i)) for i in range(40)]
    for _ in range(600):
        op = rng.random()
        t, i = rng.choice(ids)
        if op < 0.45:
            a = rng.choice(addrs)
            p.update(gp.ObjectPlacementItem(gp.ObjectId(t, i), a))
            m.update(t, i, a)
        elif op < 0.55:
            p.remove(gp.ObjectId(t, i))
            m.remove(t, i)
        elif op < 0.62:
            a = rng.choice(addrs)
            p.clean_server(a)
            m.clean_server(a)
        else:
            assert p.lookup(gp.ObjectId(t, i)) == m.lookup(t, i)
    for t, i in ids:
        assert p.lookup(gp.ObjectId(t, i)) == m.lookup(t, i)
    assert p.directory_len()[0] == len(m)


def test_batched_directory_matches_model_with_growth_and_duplicates(gp, oracle):
    """Batched update/lookup/remove/clean_node vs the model; forces several table growths (initial capacity 1024),
    and checks the 'last one in array order wins' rule for duplicate keys inside one batch."""
    p, m = provider(gp, directory_capacity=1024), oracle.DirectoryModel()
    addrs = ["10.0.0.%d:5000" % j for j in range(7)]
    nidx = p.set_nodes(addrs)
    rng = np.random.default_rng(9)
    n = 50000
    ids = [("Obj", str(i)) for i in range(n)]
    keys = p.hash_ids(ids)
    assert keys.tolist() == [oracle.object_key(t, i) for t, i in ids[:]]  # device FNV == host helper == oracle
    assert len(set(keys.tolist())) == n
    for rnd in range(4):
        sel = rng.integers(0, n, 20000)
        # duplicates inside the batch on purpose
        sel[:2000] = sel[2000:4000]
        tgt = rng.integers(0, len(addrs), len(sel))
        rm = rng.random(len(sel)) < 0.1
        idx = np.where(rm, NONE, nidx[tgt]).astype(np.uint32)
        p.update_many(keys[sel], idx)
        for s, t, r in zip(sel.tolist(), tgt.tolist(), rm.tolist()):
            m.update("Obj", str(s), None if r else addrs[t])
        if rnd == 2:
            assert p.clean_node(int(nidx[3])) == sum(1 for i in range(n) if m.lookup("Obj", str(i)) == addrs[3])
            m.clean_server(addrs[3])
        if rnd == 3:
            dead = rng.integers(0, n, 3000)
            p.remove_many(keys[dead])
            for s in dead.tolist():
                m.remove("Obj", str(s))
    got = p.lookup_many(keys)
    want = []
    for i in range(n):
        a = m.lookup("Obj", str(i))
        want.append(NONE if a is None else int(nidx[addrs.index(a)]))
    assert got.tolist() == want
    placed, slots = p.directory_len()
    assert placed == len(m) and slots >= 2 * placed
    cnt = p.load_counters()
    assert cnt.sum() == placed and cnt.tolist() == [want.count(int(j)) for j in nidx]
    # empty batches are fine
    p.update_many(np.empty(0, np.uint64), np.empty(0, np.uint32))
    assert p.lookup_many(np.empty(0, np.uint64)).shape == (0,)


# ---- solver: weighted rendezvous, bit-exact --------------------------------------------------------------------
def _nodes(p, oracle, M, uniform=False):
    addrs, seeds, w = oracle.synth_nodes(M, uniform=uniform)
    idx = p.set_nodes(addrs, w)
    assert idx.tolist() == list(range(M))
    return addrs, seeds, w


@pytest.mark.parametrize("variant", ["2", "1"])
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_c2_weighted_rendezvous_1m_x_64(gp, oracle, seed, variant):
    """BASELINE.json configs[1]: 1M objects x 64 nodes, weights in [1,16]; both kernel variants."""
    os.environ["RIO_ASSIGN_VARIANT"] = variant
    try:
        p = provider(gp)
        _, seeds, w = _nodes(p, oracle, 64)
        keys = oracle.synth_keys(1 << 20, seed)
        got = p.assign_batch(keys)
    finally:
        os.environ.pop("RIO_ASSIGN_VARIANT", None)
    want = oracle.assign_hrw(keys, seeds, w, threads=8)
    assert (got == want).all()


@pytest.mark.parametrize("variant", ["2", "1"])
@pytest.mark.parametrize("M,uniform", [(1, True), (2, False), (3, True), (31, False), (33, False), (64, True), (257, False), (1024, False), (1024, True), (1500, False)])
def test_ragged_node_counts(gp, oracle, M, uniform, variant):
    os.environ["RIO_ASSIGN_VARIANT"] = variant
    try:
        p = provider(gp)
        _, seeds, w = _nodes(p, oracle, M, uniform)
        keys = oracle.synth_keys(40013, 2)  # ragged: not a multiple of any tile
        got = p.assign_batch(keys)
    finally:
        os.environ.pop("RIO_ASSIGN_VARIANT", None)
    assert (got == oracle.assign_hrw(keys, seeds, w, threads=8)).all()


@pytest.mark.parametrize("variant", ["2", "1"])
@pytest.mark.parametrize("M,n", [(9000, 6001), (70000, 1501)])
def test_node_tables_larger_than_one_shared_memory_chunk(gp, oracle, M, n, variant):
    """M = 9000: the table is streamed through shared memory in two chunks and the winner is re-hashed from global
    memory; M = 70000 exceeds the 16-bit positions of k_assign_hrw_v2, so the launcher must route to k_assign_hrw."""
    os.environ["RIO_ASSIGN_VARIANT"] = variant
    try:
        p = provider(gp)
        _, seeds, w = _nodes(p, oracle, M)
        keys = oracle.synth_keys(n, 5)
        got = p.assign_batch(keys)
    finally:
        os.environ.pop("RIO_ASSIGN_VARIANT", None)
    assert (got == oracle.assign_hrw(keys, seeds, w, threads=8)).all()


def test_many_weight_classes_and_big_weights(gp, oracle):
    p = provider(gp)
    addrs, seeds, _ = oracle.synth_nodes(300)
    rng = np.random.default_rng(4)
    w = rng.integers(1, 2**31, 300).astype(np.uint32)  # ~300 distinct classes
    w[7] = 0xFFFFFFFF
    w[8] = 1
    p.set_nodes(addrs, w)
    keys = oracle.synth_keys(30000, 3)
    assert (p.assign_batch(keys) == oracle.assign_hrw(keys, seeds, w, threads=8)).all()


def test_edge_cases_empty_dead_and_raw_keys(gp, oracle):
    p = provider(gp)
    addrs, seeds, w = oracle.synth_nodes(16)
    # no nodes at all -> NONE
    assert (p.assign_batch(oracle.synth_keys(100, 1)) == NONE).all()
    w2 = w.copy()
    w2[::2] = 0  # weight 0 == not live
    p.set_nodes(addrs, w2)
    p.node_set_active(1, False)  # set_inactive (peer_to_peer.rs:170-173)
    w2[1] = 0
    keys = np.concatenate([np.arange(0, 5000, dtype=np.uint64), np.array([2**64 - 1, 2**64 - 2, 0], dtype=np.uint64)])  # raw, unmixed keys
    got = p.assign_batch(keys)
    assert (got == oracle.assign_hrw(keys, seeds, w2)).all()
    assert p.assign_batch(np.empty(0, np.uint64)).shape == (0,)
    p.node_set_active(1, True)
    w2[1] = w[1]
    assert (p.assign_batch(keys) == oracle.assign_hrw(keys, seeds, w2)).all()


def test_golden_vectors_on_gpu(gp):
    import json

    g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "solver_hrw_v3.json")))
    p = provider(gp)
    p.set_nodes(g["hrw"]["addresses"], np.array(g["hrw"]["weights"], dtype=np.uint32))
    keys = np.array([int(k) for k in g["hrw"]["keys"]], dtype=np.uint64)
    assert p.assign_batch(keys).tolist() == g["hrw"]["idx"]
    s = p.new_set(len(keys))
    s.load_keys(keys)
    passes = s.assign_bounded(0, *g["bounded"]["cap"], g["bounded"]["max_rounds"])
    assert passes == g["bounded"]["passes"] and s.read().tolist() == g["bounded"]["idx"]
    assert s.counters().tolist() == g["bounded"]["counts"]


# ---- solver: affinity cost, 1e-5 relative ------------------------------------------------------------------------
@pytest.mark.parametrize("variant", ["umma", "ffma"])
@pytest.mark.parametrize("K,M,n", [(16, 1024, 60000), (16, 37, 5001), (16, 64, 999), (16, 65, 7000), (16, 300, 20000), (16, 2000, 4000), (8, 64, 3000), (5, 9, 1000)])
def test_affinity_cost_argmin(gp, oracle, K, M, n, variant):
    """cost = -dot, argmin (DESIGN.md 3.6).  K == 16 runs on the tensor cores (tcgen05, bf16x3 split) unless
    RIO_AFFINITY_VARIANT=ffma or more than 2048 nodes are live (M = 2000 still fits: 1998 live nodes pad to 2048); other K
    use CUDA cores.  tests/test_gpu_affinity.py holds the exact and error-bounded checks of every dispatch branch."""
    rng = np.random.default_rng(11)
    fo = rng.uniform(-1, 1, (n, K)).astype(np.float32)
    fn = np.random.default_rng(13).uniform(-1, 1, (M, K)).astype(np.float32)
    addrs, _, _ = oracle.synth_nodes(M)
    w = np.ones(M, dtype=np.uint32)
    if M > 4:
        w[3] = 0
        w[M - 1] = 0
    os.environ["RIO_AFFINITY_VARIANT"] = variant
    try:
        p = provider(gp)
        p.set_nodes(addrs, w, fn)
        got = p.assign_batch(obj_feats=fo)
        s = p.new_set(n)
        s.load_keys(np.arange(n, dtype=np.uint64))
        s.load_feats(fo)
        s.assign(True)
        assert (s.read() == got).all() and (s.counters() == np.bincount(got, minlength=M)).all()
    finally:
        os.environ.pop("RIO_AFFINITY_VARIANT", None)
    idx, cost, gap = oracle.assign_affinity(fo, fn, w, threads=8)
    # index must match unless the fp64 top-2 gap is below the tolerance (then either node is accepted);
    # in every case the fp64 cost of the chosen node is within 1e-5 relative of the optimum
    tol = 1e-5 * np.abs(cost) + 1e-12
    mism = got != idx
    assert (gap[mism] <= tol[mism]).all(), (int(mism.sum()), float(gap[mism].max()) if mism.any() else None)
    chosen = -(fo.astype(np.float64) * fn.astype(np.float64)[got]).sum(1)
    assert (np.abs(chosen - cost) <= tol).all()
    assert (w[got] > 0).all()


def test_affinity_bf16_exact_inputs_are_bit_stable(gp, oracle):
    """bf16-representable features (SURVEY 8d variant): every cross term is exact, so the tensor-core path and the
    CUDA-core path must pick identical nodes."""
    rng = np.random.default_rng(3)
    def bf16_round(x):
        u = x.astype(np.float32).view(np.uint32)
        return ((u + 0x8000) & 0xFFFF0000).astype(np.uint32).view(np.float32)
    fo = bf16_round(rng.uniform(-1, 1, (30000, 16)))
    fn = bf16_round(rng.uniform(-1, 1, (512, 16)))
    addrs, _, _ = oracle.synth_nodes(512)
    p = provider(gp)
    p.set_nodes(addrs, None, fn)
    res = {}
    for v in ("umma", "ffma"):
        os.environ["RIO_AFFINITY_VARIANT"] = v
        try:
            res[v] = p.assign_batch(obj_feats=fo)
        finally:
            os.environ.pop("RIO_AFFINITY_VARIANT", None)
    idx, cost, gap = oracle.assign_affinity(fo, fn, np.ones(512, dtype=np.uint32), threads=8)
    # bf16-exact inputs: every product is exact in fp32, the two paths differ only in the order of 16 additions
    same = res["umma"] == res["ffma"]
    assert same.mean() > 0.9999 and (gap[~same] <= 1e-5 * np.abs(cost[~same])).all()
    assert ((res["umma"] == idx) | (gap <= 1e-5 * np.abs(cost))).all()


# ---- resident sets: bounded-load rounds, rebalance storm ----------------------------------------------------------
def test_set_assign_and_bounded_rounds(gp, oracle):
    p = provider(gp)
    addrs, seeds, w = oracle.synth_nodes(64)
    p.set_nodes(addrs, w)
    n = 200000
    s = p.new_set(n)
    s.synth_keys(0, n, 1)
    keys = oracle.synth_keys(n, 1)
    k2, _ = s.read(want_keys=True)
    assert (k2 == keys).all()  # device key stream == oracle key stream
    s.assign()
    want = oracle.assign_hrw(keys, seeds, w, threads=8)
    assert (s.read() == want).all()
    assert (s.counters() == oracle.counts(want, 64)).all()
    for cap in [(5, 4), (101, 100), (1, 1)]:
        passes = s.assign_bounded(0, cap[0], cap[1], 4)
        widx, wcnt, wpass = oracle.assign_bounded(keys, seeds, w, cap[0], cap[1], 4, threads=8)
        assert passes == wpass, cap
        assert (s.read() == widx).all(), cap
        assert (s.counters() == wcnt).all(), cap


def test_rebalance_storm_matches_fresh_assignment(gp, oracle):
    """C5 at test scale: 8 join/leave events; after each one the incremental result must equal a from-scratch
    assignment over the new live set (rendezvous is history-free), and only the minimal set of objects moves."""
    M0 = 128
    p = provider(gp)
    addrs, seeds, w = oracle.synth_nodes(M0 + 4)
    w_live = w.copy()
    w_live[M0:] = 0
    p.set_nodes(addrs[:M0], w[:M0])
    n = 300000
    keys = oracle.synth_keys(n, 2)
    s = p.new_set(n)
    s.load_keys(keys)
    s.assign()
    s.commit()  # directory follows the same events through rio_cuda_rebalance
    events = [("leave", 17), ("join", M0), ("leave", 3), ("join", M0 + 1), ("leave", 100), ("join", M0 + 2), ("leave", 64), ("join", M0 + 3)]
    prev = s.read().copy()
    for ev, j in events:
        if ev == "leave":
            p.node_set_active(j, False)
            w_live[j] = 0
        else:
            assert p.node_upsert(addrs[j], int(w[j])) == j
            w_live[j] = w[j]
        moved = s.rebalance(ev, j)
        dmoved = p.rebalance(ev, j)
        want = oracle.assign_hrw(keys, seeds, w_live, threads=8)
        got = s.read()
        assert (got == want).all(), (ev, j)
        assert moved == int((prev != want).sum()) == dmoved, (ev, j)
        if ev == "leave":
            assert (prev[prev != want] == j).all()
        else:
            assert (want[prev != want] == j).all()
        assert (p.lookup_many(keys) == want).all(), (ev, j)
        assert (s.counters() == oracle.counts(want, M0 + 4)[: len(s.counters())]).all()
        prev = got.copy()


# ---- the per-request policy, batched (service.rs:193-254) -----------------------------------------------------------
def test_place_batch_self_policy_matches_service_model(gp, oracle):
    p, m = provider(gp), oracle.DirectoryModel()
    addrs = ["0.0.0.0:%d" % (5000 + j) for j in range(4)]
    p.set_nodes(addrs)
    for a in addrs:
        ip, port = a.split(":")
        m.member_push(ip, port, True)
    ids = [("MockService", str(i)) for i in range(3000)]
    keys = np.array([oracle.object_key(t, i) for t, i in ids], dtype=np.uint64)

    def both(sel, me):
        got = p.place_batch(keys[sel], "self", addrs[me])
        want = [m.get_or_create_placement(addrs[me], *ids[s]) for s in sel]
        assert [p.node_address(int(g)) for g in got] == want

    both(list(range(0, 2000)), 0)          # unallocated -> claimed by the serving node (service.rs:244-252)
    both(list(range(1000, 3000)), 1)       # half already owned by node 0 -> kept (-> Redirect upstream)
    p.node_set_active(0, False)            # owner dies (tests/object_allocation.rs:75-137)
    m.member_set_active("0.0.0.0", "5000", False)
    both(list(range(500, 1500)), 2)        # re-placed on the new serving node; clean_server drops node 0's other objects
    for s in list(range(0, 3000, 7)):
        a = m.lookup(*ids[s])
        g = p.lookup(gp.ObjectId(*ids[s]))
        assert g == a
    # malformed record (service.rs:213-222): dropped and re-placed
    p.update(gp.ObjectPlacementItem(gp.ObjectId("MockService", "bad"), "garbage"))
    m.update("MockService", "bad", "garbage")
    kb = np.array([oracle.object_key("MockService", "bad")], dtype=np.uint64)
    assert p.node_address(int(p.place_batch(kb, "self", addrs[3])[0])) == m.get_or_create_placement(addrs[3], "MockService", "bad")


def test_place_batch_hrw_policy(gp, oracle):
    p = provider(gp)
    addrs, seeds, w = oracle.synth_nodes(32)
    p.set_nodes(addrs, w)
    keys = oracle.synth_keys(20000, 3)
    want = oracle.assign_hrw(keys, seeds, w, threads=4)
    got = p.place_batch(keys, "hrw")
    assert (got == want).all() and (p.lookup_many(keys) == want).all()
    assert (p.place_batch(keys, "hrw") == want).all()  # idempotent: everything already placed on live nodes
    p.node_set_active(5, False)
    w2 = w.copy()
    w2[5] = 0
    got2 = p.place_batch(keys[:10000], "hrw")
    want2 = oracle.assign_hrw(keys[:10000], seeds, w2, threads=4)
    assert (got2 == want2).all()
    # node 5's objects outside the batch were unassigned by clean_server, the rest is untouched
    rest = p.lookup_many(keys[10000:])
    assert (rest[want[10000:] == 5] == NONE).all() and (rest[want[10000:] != 5] == want[10000:][want[10000:] != 5]).all()


# ---- full-size properties (BASELINE sizes; every object is checked against the oracle) -------------------------------------------------
def test_full_size_10m_x_1024_properties(gp, oracle):
    n, M = 10_000_000, 1024
    p = provider(gp)
    addrs, seeds, w = oracle.synth_nodes(M)
    p.set_nodes(addrs, w)
    s = p.new_set(n)
    s.synth_keys(0, n, 1)
    s.assign()
    idx = s.read()
    cnt = s.counters()
    assert cnt.sum() == n and (cnt == np.bincount(idx, minlength=M)).all()
    # EVERY object against the oracle (10 M x 1024 pair hashes each on all host cores: a few seconds on the GPU box)
    keys = oracle.synth_keys(n, 1)
    assert (idx == oracle.assign_hrw(keys, seeds, w, threads=os.cpu_count() or 8)).all()
    # weights respected: chi-square of counts against w/W
    e = n * w / w.sum()
    chi = ((cnt - e) ** 2 / e).sum()
    assert chi < (M - 1) + 6 * np.sqrt(2 * (M - 1)), chi
    # leave(17): only node 17's objects move and node 17 ends empty
    p.node_set_active(17, False)
    moved = s.rebalance("leave", 17)
    idx2 = s.read()
    ch = idx != idx2
    assert moved == ch.sum() == cnt[17] and (idx[ch] == 17).all() and (idx2 != 17).all()
    # join(17) back: the exact same objects come back (idempotent round trip)
    p.node_set_active(17, True)
    moved2 = s.rebalance("join", 17)
    assert moved2 == moved and (s.read() == idx).all()
    # same result through the host-buffer API (H2D/D2H pipelined path)
    assert (p.assign_batch(keys[:3_000_000]) == idx[:3_000_000]).all()


# ---- micro-batched per-request resolves (SURVEY 8f row 1) ------------------------------------------------------------
def test_resolver_coalesces_concurrent_per_id_calls(gp, oracle):
    """16 threads call get_or_create_placement per id, as Service does per request (service.rs:193-254, one task per
    connection server.rs:303); the resolver must coalesce them into few place_batch launches and give every caller the
    answer the restated reference policy gives."""
    import threading

    p, m = provider(gp), oracle.DirectoryModel()
    addrs = ["0.0.0.0:%d" % (5000 + j) for j in range(4)]
    p.set_nodes(addrs)
    for a in addrs:
        ip, port = a.split(":")
        m.member_push(ip, port, True)
    ids = [("MockService", str(i)) for i in range(4000)]
    r = gp.Resolver(p, policy="self", self_address=addrs[1], max_batch=512, max_wait_us=200)
    got = [None] * len(ids)

    def work(t):
        for k in range(t, len(ids), 16):
            got[k] = r.get_or_create_placement(*ids[k])

    th = [threading.Thread(target=work, args=(t,)) for t in range(16)]
    for x in th:
        x.start()
    for x in th:
        x.join()
    want = [m.get_or_create_placement(addrs[1], *i) for i in ids]
    assert got == want
    st = r.stats()
    assert st["calls"] == len(ids) and st["batches"] < st["calls"] // 2 and st["largest_batch"] > 1, st
    # second pass from another "server": every id is already placed -> same owner (-> Redirect upstream)
    r2 = gp.Resolver(p, policy="self", self_address=addrs[2])
    assert [r2.get_or_create_placement(*i) for i in ids[:50]] == want[:50]
    # rendezvous policy through the same front end
    p3 = provider(gp)
    a3, seeds, w = oracle.synth_nodes(32)
    p3.set_nodes(a3, w)
    r3 = gp.Resolver(p3, policy="hrw")
    keys = oracle.synth_keys(300, 2)
    assert [r3.resolve(int(k)) for k in keys] == oracle.assign_hrw(keys, seeds, w).tolist()
    r.close(); r2.close(); r3.close()


# ---- durable write-through into the reference's SQL schema (SURVEY 8f row 3) ----------------------------------------
def test_durable_write_through_and_recovery(gp, oracle, tmp_path):
    """Mutations go to the GPU directory AND the reference's sqlite table (sqlite.rs:68-126 statements); a fresh provider
    pointed at the same file recovers every placement (bulk path: device-side id hashing + batched upsert), and the
    table itself equals the SqliteObjectPlacement restatement fed the same ops."""
    from oracle.sqlite_model import SqliteDirectoryModel
    from rio_rs_b200.durable import DurableGpuObjectPlacement

    db = str(tmp_path / "placement.sqlite3")
    p = DurableGpuObjectPlacement(db)
    assert p.prepare() == 0
    m = SqliteDirectoryModel()
    m.prepare()
    addrs = ["10.0.0.%d:5000" % j for j in range(5)]
    ids = [("Obj", str(i)) for i in range(3000)]
    tgt = [addrs[i % 5] for i in range(3000)]
    p.update_many_ids(ids, tgt)
    for (t, i), a in zip(ids, tgt):
        m.update(t, i, a)
    p.update(gp.ObjectPlacementItem(gp.ObjectId("Obj", "7"), "10.0.0.4:5000"))
    m.update("Obj", "7", "10.0.0.4:5000")
    p.remove(gp.ObjectId("Obj", "8"))
    m.remove("Obj", "8")
    p.clean_server(addrs[2])
    m.clean_server(addrs[2])
    del p
    q = DurableGpuObjectPlacement(db)   # "restart"
    restored = q.prepare()
    want = {(t, i): m.lookup(t, i) for t, i in ids}
    assert restored == sum(1 for v in want.values() if v is not None)
    for k in range(0, 3000, 13):
        assert q.lookup(gp.ObjectId(*ids[k])) == want[ids[k]]
    assert q.lookup(gp.ObjectId("Obj", "7")) == "10.0.0.4:5000" and q.lookup(gp.ObjectId("Obj", "8")) is None
    assert q.directory_len()[0] == restored


# ---- device-side id hashing and the device-resident (_dev) entry points ---------------------------------------------
def test_hash_ids_ragged_lengths(gp, oracle):
    """FNV-1a over the joined "{type}.{id}" bytes on the GPU == rio_cuda_object_key == oracle, for empty, short and very
    long ids (longer than the kernel's shared-memory staging window)."""
    rng = random.Random(5)
    ids = [("", ""), ("a.b", "c"), ("a", "b.c"), ("T", "x" * 70000)]
    for _ in range(5000):
        ids.append(("T%d" % rng.randrange(5), "".join(rng.choice("abcdef0123456789-") for _ in range(rng.choice([0, 1, 3, 8, 13, 36, 200])))))
    p = provider(gp)
    got = p.hash_ids(ids)
    assert got.tolist() == [oracle.object_key(t, i) for t, i in ids]
    assert got[1] == got[2]   # the reference's own aliasing of ("a.b","c") and ("a","b.c") (local.rs:26-29)
    assert p.hash_ids([]).shape == (0,)


def test_device_resident_entry_points(gp, oracle):
    """rio_cuda_*_dev: inputs already in HBM, asynchronous on the engine stream (what bench.py's `value` path uses)."""
    import ctypes as C

    p = provider(gp)
    addrs, seeds, w = oracle.synth_nodes(50)
    p.set_nodes(addrs, w)
    n = 123457
    keys = oracle.synth_keys(n, 3)
    L, h = p.L, p.h
    dk, di, dl = C.c_void_p(), C.c_void_p(), C.c_void_p()
    for ptr, nbytes in ((dk, n * 8), (di, n * 4), (dl, n * 4)):
        p._ck(L.rio_cuda_dev_alloc(h, nbytes, C.byref(ptr)))
    p._ck(L.rio_cuda_memcpy_h2d(h, dk, keys.ctypes.data_as(C.c_void_p), n * 8))
    p._ck(L.rio_cuda_assign_batch_dev(h, dk, None, n, di))
    p._ck(L.rio_cuda_directory_reserve(h, n))
    p._ck(L.rio_cuda_upsert_batch_dev(h, dk, di, n))
    p._ck(L.rio_cuda_lookup_batch_dev(h, dk, n, dl))
    out_i, out_l = np.empty(n, dtype=np.uint32), np.empty(n, dtype=np.uint32)
    p._ck(L.rio_cuda_memcpy_d2h(h, out_i.ctypes.data_as(C.c_void_p), di, n * 4))
    p._ck(L.rio_cuda_memcpy_d2h(h, out_l.ctypes.data_as(C.c_void_p), dl, n * 4))
    p.sync()
    want = oracle.assign_hrw(keys, seeds, w, threads=4)
    assert (out_i == want).all() and (out_l == want).all()
    assert p.directory_len()[0] == n
    for ptr in (dk, di, dl):
        p._ck(L.rio_cuda_dev_free(h, ptr))
    # an undersized table is refused up front instead of overflowing asynchronously
    q = provider(gp, directory_capacity=1024)
    q.set_nodes(addrs, w)
    q._ck(L.rio_cuda_dev_alloc(q.h, n * 8, C.byref(dk)))
    q._ck(L.rio_cuda_dev_alloc(q.h, n * 4, C.byref(di)))
    with pytest.raises(gp.Unknown):
        q._ck(L.rio_cuda_upsert_batch_dev(q.h, dk, di, n))


# ---- the client side (SURVEY 8(f) row 2); last in the file on purpose ----------------------------------------------
def test_client_first_hop_reaches_the_owner_without_redirect(gp, oracle):
    """SURVEY 8(f) row 2: ids the servers placed with policy "hrw" are found by the client's own rendezvous hash
    (include/rio_client.h, librio_client.so): node index for node index, also after a node left."""
    from rio_rs_b200 import client as CL

    try:
        CL.lib()
    except Exception as e:  # the client library is plain C++ built with g++; its own CPU tests cover it
        pytest.skip("librio_client.so unavailable: %r" % (e,))
    p = provider(gp)
    addrs, seeds, w = oracle.synth_nodes(64)
    p.set_nodes(addrs, w)
    keys = oracle.synth_keys(30000, 6)
    owner = p.place_batch(keys, "hrw")
    fh = CL.FirstHop(addrs, w)
    assert (fh.first_hop_batch(keys) == owner).all()
    p.node_set_active(9, False)
    p.rebalance("leave", 9)
    w2 = w.copy()
    w2[9] = 0
    fh.set_active_servers(addrs, w2)
    assert (fh.first_hop_batch(keys) == p.lookup_many(keys)).all()


# ---- the second half of the per-request policy (service.rs:261-298) ------------------------------------------------
def test_check_address_mismatch_matches_service_model(gp, oracle):
    """Service::call runs get_or_create_placement then check_address_mismatch (service.rs:62-70); both halves batched,
    against the restated reference after membership changes: Ok / Redirect / clean_server + DeallocateServiceObject /
    Unknown(malformed), including the directory state the clean_server side effect leaves behind."""
    from rio_rs_b200 import _native as N

    p, m = provider(gp), oracle.DirectoryModel()
    addrs = ["0.0.0.0:%d" % (5000 + j) for j in range(6)]
    p.set_nodes(addrs)
    for a in addrs:
        ip, port = a.split(":")
        m.member_push(ip, port, True)
    ids = [("MockService", str(i)) for i in range(3000)]
    keys = np.array([oracle.object_key(t, i) for t, i in ids], dtype=np.uint64)
    # objects land on all six servers (each batch is resolved by "its" server, the reference's first-claim rule)
    for me in range(6):
        sel = list(range(me * 500, (me + 1) * 500))
        got = p.place_batch(keys[sel], "self", addrs[me])
        assert [p.node_address(int(g)) for g in got] == [m.get_or_create_placement(addrs[me], *ids[s]) for s in sel]
    # two servers die, one is removed from the membership altogether
    p.node_set_active(1, False)
    m.member_set_active("0.0.0.0", "5001", False)
    p.node_set_active(4, False)
    m.member_remove("0.0.0.0", "5004")
    # a request batch arrives at server 2 carrying the owners the directory recorded BEFORE the failure (the window between
    # the two calls of Service::call); the verdict and the clean_server side effect must match, id for id
    owner = p.lookup_many(keys)
    verdict, cleaned = p.check_address_batch(owner, addrs[2])
    want = [m.check_address_mismatch(addrs[2], p.node_address(int(o))) for o in owner]
    assert verdict.tolist() == want
    assert set(want) == {N.ADDR_LOCAL, N.ADDR_REDIRECT, N.ADDR_DEALLOCATE}
    assert cleaned == 1000                                         # every object of the two dead servers was unassigned
    for s in range(0, 3000, 3):
        assert p.lookup(gp.ObjectId(*ids[s])) == m.lookup(*ids[s])
    assert p.directory_len()[0] == len(m)
    # per-request form, malformed and three-piece addresses (split(':') keeps the first two pieces)
    for addr in ("garbage", "0.0.0.0:5003:x", "0.0.0.0:5001:x", "7.7.7.7:1", addrs[2], addrs[3]):
        p.update(gp.ObjectPlacementItem(gp.ObjectId("E", addr), addr))
        m.update("E", addr, addr)
        assert p.check_address_mismatch(addrs[2], addr) == m.check_address_mismatch(addrs[2], addr), addr
        assert p.lookup(gp.ObjectId("E", addr)) == m.lookup("E", addr), addr
    assert p.check_address_mismatch("0.0.0.0:5003", "0.0.0.0:5003") == N.ADDR_LOCAL


def test_draining_node_keeps_its_objects(gp, oracle):
    """is_active looks at the membership flag only (storage/mod.rs:102-110): an active node of weight 0 is not a solver target
    but objects recorded on it are NOT cleaned by the policy."""
    p = provider(gp)
    addrs, seeds, w = oracle.synth_nodes(8)
    p.set_nodes(addrs, w)
    keys = oracle.synth_keys(4000, 2)
    owner = p.place_batch(keys, "hrw")
    w2 = w.copy()
    w2[3] = 0
    p.set_nodes(addrs, w2)                                       # node 3 drains: still active, no longer a target
    assert (p.place_batch(keys, "hrw") == owner).all()           # nothing is re-placed, nothing is cleaned
    fresh = oracle.synth_keys(4000, 3)
    assert (p.place_batch(fresh, "hrw") == oracle.assign_hrw(fresh, seeds, w2)).all() and (p.place_batch(fresh, "hrw") != 3).all()


# ---- exact ties (DESIGN.md 3.4 tie rules), forced with duplicated node seeds through the dev hook -------------------
@pytest.mark.parametrize("variant", ["2", "1"])
@pytest.mark.parametrize("mode", ["within_group", "across_groups", "across_classes", "across_classes_chunked"])
def test_exact_ties_go_to_the_lowest_index_on_the_gpu(gp, oracle, variant, mode):
    """Two or more nodes with the SAME seed hash every object alike: u ties exactly, and with equal weights so does the 64-bit
    score.  The spec sends the object to the lowest node index.  within_group: the twins sit inside one 32-node group of a
    class; across_groups: in different groups of one class; across_classes: the table is built with one class per node
    (dev option), so equal scores meet on the kernels' between-class path (`equal_score_takes` in k_assign_hrw_v2);
    across_classes_chunked: the same with a table larger than one shared-memory chunk (winner re-hashed from global)."""
    from rio_rs_b200 import _native as N

    M = {"within_group": 96, "across_groups": 200, "across_classes": 150, "across_classes_chunked": 9000}[mode]
    os.environ["RIO_ASSIGN_VARIANT"] = variant
    try:
        p = provider(gp)
        addrs, seeds, w = oracle.synth_nodes(M, uniform=True)
        seeds = seeds.copy()
        p.set_nodes(addrs, w)
        if mode == "within_group":
            twins = [(3, 4), (10, 17), (40, 41), (70, 95)]
        elif mode == "across_groups":
            twins = [(3, 44), (10, 170), (64, 199), (31, 32)]
        else:
            twins = [(3, 44), (10, 11), (100, 149), (0, M - 1)]
        for a, b in twins:
            seeds[b] = seeds[a]
            p.dev_set_node_seed(b, int(seeds[a]))
        # a triple, and a tie whose lowest index is NOT the first one met in the class-sorted table order
        seeds[7] = seeds[5] = seeds[6]
        p.dev_set_node_seed(5, int(seeds[6]))
        p.dev_set_node_seed(7, int(seeds[6]))
        if mode.startswith("across_classes"):
            p.dev_set_table_options(N.DEV_SPLIT_CLASSES)
        keys = oracle.synth_keys(300_000 if M < 1000 else 60_000, 7)
        got = p.assign_batch(keys)
        want = oracle.assign_hrw(keys, seeds, w, threads=8)
        assert (got == want).all()
        # the ties really happened: the upper twin never wins although it scores exactly like the lower one (twins hash alike, so
        # the pair wins as often as ONE node does)
        for a, b in twins:
            assert (want != b).all() and (want == a).sum() > (0.6 * len(keys) / M if M < 1000 else 0)
        assert (want != 6).all() and (want != 7).all()
    finally:
        os.environ.pop("RIO_ASSIGN_VARIANT", None)


def test_per_id_trait_calls_through_the_coalescing_front_end(gp, oracle):
    """lookup / update / remove per id (mod.rs:46-55) from 16 threads through the resolver: every thread owns a slice of the
    ids and replays a random op sequence on it; results must equal the LocalObjectPlacement restatement replaying the same
    sequence, and the calls must have been coalesced into far fewer engine batches."""
    import threading

    p, m = provider(gp), oracle.DirectoryModel()
    addrs = ["10.0.0.%d:5000" % j for j in range(4)]
    p.set_nodes(addrs)
    r = gp.Resolver(p, policy="self", self_address=addrs[0], max_batch=256, max_wait_us=100)
    T, per = 16, 60
    errors = []

    def work(t):
        rng = random.Random(100 + t)
        ids = [("T%d" % t, str(i)) for i in range(per)]
        local = {}
        try:
            for _ in range(300):
                oid = rng.choice(ids)
                x = rng.random()
                if x < 0.4:
                    a = rng.choice(addrs)
                    r.update(gp.ObjectPlacementItem(gp.ObjectId(*oid), a))
                    local[oid] = a
                elif x < 0.5:
                    r.remove(gp.ObjectId(*oid))
                    local.pop(oid, None)
                else:
                    got = r.lookup(gp.ObjectId(*oid))
                    if got != local.get(oid):
                        errors.append((oid, got, local.get(oid)))
            for oid, a in local.items():
                m.update(oid[0], oid[1], a)
        except Exception as e:  # noqa: BLE001
            errors.append(repr(e))

    th = [threading.Thread(target=work, args=(t,)) for t in range(T)]
    for x in th:
        x.start()
    for x in th:
        x.join()
    assert not errors, errors[:3]
    for t in range(T):
        for i in range(per):
            assert p.lookup(gp.ObjectId("T%d" % t, str(i))) == m.lookup("T%d" % t, str(i))
    assert p.directory_len()[0] == len(m)
    st = r.stats()
    assert st["calls"] == T * 300 and st["batches"] < st["calls"] and st["largest_batch"] > 1, st
    r.close()
