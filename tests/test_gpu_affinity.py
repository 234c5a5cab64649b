"""Affinity cost (DESIGN.md 3.6) on every dispatch branch, against two oracles.

`cost_ij = -sum_k Fobj[i,k] * Fnode[j,k]`, argmin over the live nodes, ties -> lowest j.  The engine has three kernels for it:
k_affinity_umma + k_affinity_resolve (K = 16 on the tensor cores: bf16x3 split, six MMAs, the best GROUP of 8 columns, then an
fp32 re-score of those 8 nodes), k_assign_affinity (K = 16 on CUDA cores, node rows in 2048-node shared-memory chunks) and
k_assign_affinity_generic (any other K).  Acceptance rules, one per kind of path:

* CUDA-core paths (RIO_AFFINITY_VARIANT=ffma, more than affinity_umma_max_nodes() live nodes, K != 16): the index equals
  `oracle.assign_affinity_f32` exactly -- the specified fp32 arithmetic (fmaf over k ascending, strict < in node order).
* Tensor-core path: (a) the returned node is the fp32 argmin (lowest index on ties) over the live nodes of its own group of 8
  compacted positions -- this pins the resolve exactly; (b) c64(j') - c64(j*) <= TAU * S_i, where c64 is the fp64 cost,
  j* the fp64 oracle's node and S_i = sum_k |Fobj[i,k]| * max_j |Fnode[j,k]| (an upper bound of sum_k |a_k b_k| over the live
  nodes).  TAU = 2^-15: dropped cross terms <= 2^-23 S, six fp32 MMA accumulations ~2^-20 S, fp32 re-score <= 2 gamma_16 S ~ 2^-19 S.
* Every path: where the fp64 top-2 gap exceeds TAU * S_i the index equals the fp64 oracle's.

Input families: A exact small integers (every path equals the fp64 oracle index for index, ties included; duplicated node rows
force ties at every boundary the kernels have), B general fp32 (uniform / normal / log-uniform magnitudes, with near-duplicate
nodes so that hundreds of objects sit within TAU * S of a tie), C cancellation (|cost| << sum |a b|), D power-of-two scaling
(each path's indices must not change).  Every case runs through assign_batch (host buffers, 1 Mi-object chunks), a resident set
(new_set + load_feats + assign(True), twice, counters against bincount) and rio_cuda_assign_batch_dev, which must agree.

The largest observed (c64(j') - c64(j*)) / S per family and path is printed at the end of the module (pytest -s).
"""
import ctypes as C
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

NONE = 0xFFFFFFFF
TAU = 2.0 ** -15
UMMA_MAX_LIVE = 2048      # affinity_umma_max_nodes(): (227 KiB - 2176 - 24576) / 96 B per node, rounded down to 256
CHUNK = 2048              # k_assign_affinity: node rows per shared-memory chunk
VARIANTS = ["umma", "ffma"]
THREADS = min(8, os.cpu_count() or 1)

_max_err = {}


@pytest.fixture(scope="module")
def gp():
    from rio_rs_b200 import build

    build.build()
    import rio_rs_b200 as R

    return R


@pytest.fixture(scope="module", autouse=True)
def error_report():
    yield
    if _max_err:
        print("\nlargest (c64(j') - c64(j*)) / S, TAU = 2^-15 = %.3g:" % TAU)
        for (fam, path), e in sorted(_max_err.items()):
            print("  family %-14s %-12s %.3g  (%.2g TAU)" % (fam, path, e, e / TAU))


# ---- running the engine ------------------------------------------------------------------------------------------------------
def addresses(M, port=7000):
    return ["10.1.%d.%d:%d" % (j >> 8, j & 255, port) for j in range(M)]


def is_tensor_core(variant, K, n_live):
    return variant == "umma" and K == 16 and 1 <= n_live <= UMMA_MAX_LIVE


def assign_dev(p, fo):
    """rio_cuda_assign_batch_dev: features already in device memory, one launch, no chunking."""
    L, h = p.L, p.h
    n = fo.shape[0]
    df, di = C.c_void_p(), C.c_void_p()
    p._ck(L.rio_cuda_dev_alloc(h, fo.nbytes, C.byref(df)))
    p._ck(L.rio_cuda_dev_alloc(h, n * 4, C.byref(di)))
    try:
        p._ck(L.rio_cuda_memcpy_h2d(h, df, fo.ctypes.data_as(C.c_void_p), fo.nbytes))
        p._ck(L.rio_cuda_assign_batch_dev(h, None, df, n, di))
        out = np.empty(n, dtype=np.uint32)
        p._ck(L.rio_cuda_memcpy_d2h(h, out.ctypes.data_as(C.c_void_p), di, n * 4))
        p.sync()
    finally:
        p._ck(L.rio_cuda_dev_free(h, df))
        p._ck(L.rio_cuda_dev_free(h, di))
    return out


def run(p, fo, variant, resident=True, dev=True):
    """The indices of every entry point (which must agree) for one variant; resident-set counters against bincount."""
    fo = np.ascontiguousarray(fo, dtype=np.float32)
    n = fo.shape[0]
    os.environ["RIO_AFFINITY_VARIANT"] = variant
    try:
        got = p.assign_batch(obj_feats=fo)
        if resident:
            s = p.new_set(n)
            s.load_keys(np.arange(n, dtype=np.uint64))
            s.load_feats(fo)
            total = p.node_count()[0]
            want_counts = np.bincount(got[got != NONE], minlength=total)
            for _ in range(2):   # the second call must reset the counters, not add to them
                s.assign(True)
                assert (s.read() == got).all()
                assert (s.counters() == want_counts).all()
        if dev:
            assert (assign_dev(p, fo) == got).all()
    finally:
        os.environ.pop("RIO_AFFINITY_VARIANT", None)
    return got


# ---- the oracles and the acceptance rules ------------------------------------------------------------------------------------
class Ref:
    """fp64 spec oracle + fp32 CUDA-core restatement for one (objects, node table, live mask)."""

    def __init__(self, oracle, fo, fn, live):
        self.oracle, self.fo, self.fn = oracle, np.ascontiguousarray(fo, np.float32), np.ascontiguousarray(fn, np.float32)
        self.live = np.ascontiguousarray(live, dtype=np.uint32)
        self.live_idx = np.flatnonzero(self.live)
        self.idx64, self.c64, self.gap = oracle.assign_affinity(self.fo, self.fn, self.live, threads=THREADS)
        self.idx32 = oracle.assign_affinity_f32(self.fo, self.fn, self.live, threads=THREADS)
        fmax = np.abs(self.fn[self.live_idx].astype(np.float64)).max(0)
        self.S = np.abs(self.fo.astype(np.float64)) @ fmax
        self.K = self.fo.shape[1]

    def cost64(self, idx):
        return -np.einsum("ik,ik->i", self.fo.astype(np.float64), self.fn[idx].astype(np.float64))

    def near_ties(self):
        return int((self.gap <= TAU * self.S).sum())

    def check(self, got, variant, family):
        """Apply the rule of the path `variant` takes; record the normalised fp64 error."""
        n = len(got)
        path = "tensor-core" if is_tensor_core(variant, self.K, len(self.live_idx)) else ("cuda-core" if self.K == 16 else "generic-K")
        assert got.shape == (n,) and (got != NONE).all() and (self.live[got] > 0).all(), (family, path)
        if path != "tensor-core":
            bad = np.flatnonzero(got != self.idx32)
            assert bad.size == 0, (family, path, bad.size, bad[:5], got[bad[:5]], self.idx32[bad[:5]])
        else:
            # (a) the resolve: fp32 argmin, lowest index, over the live nodes of the returned node's group of 8 positions
            pos = np.searchsorted(self.live_idx, got)
            cand_pos = (pos // 8)[:, None] * 8 + np.arange(8)
            valid = cand_pos < len(self.live_idx)
            cand = self.live_idx[np.minimum(cand_pos, len(self.live_idx) - 1)]
            c32 = self.oracle.affinity_pair_cost_f32(self.fo, self.fn, np.repeat(np.arange(n), 8), cand.ravel(), threads=THREADS).reshape(n, 8)
            c32[~valid] = np.inf
            want = cand[np.arange(n), np.argmin(c32, axis=1)]
            bad = np.flatnonzero(got != want)
            assert bad.size == 0, (family, path, "resolve", bad.size, bad[:5], got[bad[:5]], want[bad[:5]])
        # (b) the selection bound (the CUDA-core paths meet it with room to spare), and the fp64 index wherever the gap is clear
        err = (self.cost64(got) - self.c64) / np.where(self.S > 0, self.S, 1.0)
        worst = int(np.argmax(err))
        assert err[worst] <= TAU, (family, path, "bound", worst, err[worst] / TAU)
        clear = self.gap > TAU * self.S
        bad = np.flatnonzero(clear & (got != self.idx64))
        assert bad.size == 0, (family, path, "clear gap", bad.size, bad[:5])
        key = (family, path)
        _max_err[key] = max(_max_err.get(key, 0.0), float(max(err[worst], 0.0)))
        return path


# ---- input families ----------------------------------------------------------------------------------------------------------
def exact_ints(rng, shape):
    """Family A: integers in [-4, 4]: every product and partial sum is exact in bf16 pieces and in fp32, in any order."""
    return rng.integers(-4, 5, shape).astype(np.float32)


def general(rng, dist, shape):
    """Family B: general fp32 values with mixed signs."""
    if dist == "uniform":
        x = rng.uniform(-1, 1, shape)
    elif dist == "normal":
        x = rng.standard_normal(shape)
    else:   # log-uniform magnitudes over 2^-10 .. 2^10
        x = rng.choice([-1.0, 1.0], shape) * 2.0 ** rng.uniform(-10, 10, shape)
    return x.astype(np.float32)


def add_near_twins(rng, fn, live_idx, pairs):
    """Overwrite `pairs` live rows with copies of other live rows perturbed by 2^-24 .. 2^-12 relative: objects won by either
    row sit within rounding of a tie, in the same group of 8, across groups or across tiles (random positions)."""
    pick = rng.choice(live_idx, 2 * pairs, replace=False)
    src, dst = pick[:pairs], pick[pairs:]
    rel = rng.choice([-1.0, 1.0], (pairs, fn.shape[1])) * 2.0 ** rng.uniform(-24, -12, (pairs, fn.shape[1]))
    fn[dst] = (fn[src].astype(np.float64) * (1 + rel)).astype(np.float32)


def provider_with(gp, fn, live):
    p = gp.GpuObjectPlacement()
    p.set_nodes(addresses(len(fn)), np.asarray(live, dtype=np.uint32), fn)
    return p


# ---- family A over every node-count branch, with ties forced at each boundary ---------------------------------------------------
# name -> (live nodes, interned nodes, dead node indices)
SHAPES = {
    "live1": (1, 1, []),
    "live8": (8, 8, []),
    "live9": (9, 9, []),
    "live63": (63, 64, [4]),
    "live64": (64, 65, [4]),
    "live65": (65, 66, [4]),
    "live255": (255, 256, [4]),
    "live257": (257, 258, [4]),
    "live768": (768, 769, [4]),
    "live1280": (1280, 1281, [4]),
    "live1792": (1792, 1793, [4]),
    "live2048": (2048, 2049, [4]),         # the tensor cores' full capacity
    "live2049": (2049, 2050, [4]),         # one over: CUDA-core fallback, two shared-memory chunks
    "live4100": (4100, 6149, [4] + list(range(2048, 4096))),   # fallback, three chunks, the middle one entirely dead
    "sparse9000": (2000, 9000, None),      # compacted tensor-core operands + global-atomic histogram; ffma: 5 mostly dead chunks
}


def twin_pairs(live_idx, dead):
    """Node pairs (lower, upper) given identical rows.  Positions are compacted live positions (what the tensor-core kernel
    sees); the chunk pair straddles node index 2048 (what the CUDA-core kernel sees)."""
    nl = len(live_idx)
    at = lambda q: int(live_idx[q])   # noqa: E731
    pairs = []
    used = set()

    def add(a, b):
        if a not in used and b not in used:
            pairs.append((a, b))
            used.update((a, b))
    if nl >= 8:
        add(at(1), at(6))                   # inside one group of 8
    if nl >= 24:
        add(at(10), at(21))                 # two groups
    if nl >= 40:
        add(at(31), at(32))                 # the column halves of the 64-node tile
    if nl >= 130:
        add(at(127), at(128))               # the column halves of a 256-node tile
    if nl >= 400:
        add(at(200), at(300))               # two tiles
    if nl >= 1500:
        add(at(nl - 700), at(nl - 1))       # first and last tile region, last live node
    lo, hi = live_idx[live_idx < CHUNK], live_idx[live_idx >= CHUNK]
    if len(lo) > 64 and len(hi):
        add(int(lo[-2]), int(hi[0]))        # across the CUDA-core chunk boundary
    if dead:
        d = min(dead)
        add(d, int(live_idx[np.searchsorted(live_idx, d) + 3]))   # lower twin dead: the upper one must win
    return pairs


@pytest.mark.parametrize("shape", list(SHAPES))
def test_exact_arithmetic_every_node_count_branch(gp, oracle, shape):
    nl, total, dead = SHAPES[shape]
    rng = np.random.default_rng(100 + nl)
    live = np.ones(total, dtype=np.uint32)
    if dead is None:
        live[:] = 0
        live[np.sort(rng.choice(np.arange(5, total), nl, replace=False))] = 1
        dead = [4]
    live[dead] = 0
    live_idx = np.flatnonzero(live)
    assert len(live_idx) == nl
    fn = exact_ints(rng, (total, 16))
    pairs = twin_pairs(live_idx, dead)
    for a, b in pairs:
        fn[a] = fn[b] = rng.choice([-4, -3, 3, 4], 16)   # strong rows: each pair wins a fair share of the objects
    n = 3000 if total > 4000 else 6000
    fo = exact_ints(rng, (n, 16))
    ref = Ref(oracle, fo, fn, live)
    p = provider_with(gp, fn, live)
    for v in VARIANTS:
        got = run(p, fo, v)
        ref.check(got, v, "A")
        bad = np.flatnonzero(got != ref.idx64)
        assert bad.size == 0, (shape, v, bad.size, bad[:5], got[bad[:5]], ref.idx64[bad[:5]])
    # the ties really happened
    if nl >= 8:
        assert (ref.gap == 0).mean() > 0.1, (ref.gap == 0).mean()   # 11-21 % at these seeds
    for a, b in pairs:
        if live[a]:
            assert (ref.idx64 == a).sum() >= 5 and (ref.idx64 != b).all(), (a, b)
        else:
            assert (ref.idx64 == b).sum() >= 5, (a, b)


@pytest.mark.parametrize("n", [1, 127, 128, 129, 40013])
def test_exact_arithmetic_partial_row_blocks(gp, oracle, n):
    """Object counts around the 128-object row block of the tensor-core kernel (one partial block, n < 128)."""
    rng = np.random.default_rng(n)
    total = 301
    live = np.ones(total, dtype=np.uint32)
    live[4] = 0
    fn = exact_ints(rng, (total, 16))
    for a, b in twin_pairs(np.flatnonzero(live), [4]):
        fn[a] = fn[b] = rng.choice([-4, -3, 3, 4], 16)
    fo = exact_ints(rng, (n, 16))
    ref = Ref(oracle, fo, fn, live)
    p = provider_with(gp, fn, live)
    for v in VARIANTS:
        got = run(p, fo, v)
        ref.check(got, v, "A")
        assert (got == ref.idx64).all(), v


def test_host_chunk_boundary_matches_the_device_entry_point(gp, oracle):
    """(1 << 20) + 77 objects: assign_batch cuts host buffers into 1 Mi-object chunks; the _dev entry point runs one launch."""
    rng = np.random.default_rng(77)
    n = (1 << 20) + 77
    fn = exact_ints(rng, (10, 16))
    live = np.ones(10, dtype=np.uint32)
    live[4] = 0
    fn[2] = fn[7] = rng.choice([-4, 4], 16)
    fo = exact_ints(rng, (n, 16))
    ref = Ref(oracle, fo, fn, live)
    p = provider_with(gp, fn, live)
    for v in VARIANTS:
        got = run(p, fo, v, resident=False)
        ref.check(got, v, "A")
        assert (got == ref.idx64).all(), v


# ---- generic K: exact integers and general fp32 --------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [1, 2, 3, 15, 17, 32, 64])
def test_generic_k(gp, oracle, K):
    rng = np.random.default_rng(K)
    M = 150
    live = np.ones(M, dtype=np.uint32)
    live[[4, M - 1]] = 0
    live_idx = np.flatnonzero(live)
    # A: exact, with twins inside a group, across groups, and a dead lower twin
    fn = exact_ints(rng, (M, K))
    for a, b in ((1, 6), (10, 90), (4, 20)):
        fn[a] = fn[b] = rng.choice([-4, -3, 3, 4], K)
    fo = exact_ints(rng, (4000, K))
    ref = Ref(oracle, fo, fn, live)
    p = provider_with(gp, fn, live)
    got = run(p, fo, "umma")   # the variant does not matter for K != 16
    ref.check(got, "umma", "A")
    assert (got == ref.idx64).all()
    # B: general fp32 with near-twins (summation order decides many of them)
    fn = general(rng, "uniform", (M, K))
    add_near_twins(rng, fn, live_idx, 40)
    fo = general(rng, "uniform", (6000, K))
    ref = Ref(oracle, fo, fn, live)
    p = provider_with(gp, fn, live)
    got = run(p, fo, "ffma")
    ref.check(got, "ffma", "B")
    if K > 1:
        assert ref.near_ties() >= 100, ref.near_ties()


# ---- family B: general fp32 on the K = 16 paths ---------------------------------------------------------------------------------
@pytest.mark.parametrize("dist", ["uniform", "normal", "loguniform"])
@pytest.mark.parametrize("nl", [1024, 2200])
def test_general_fp32(gp, oracle, dist, nl):
    rng = np.random.default_rng(["uniform", "normal", "loguniform"].index(dist) * 10000 + nl)
    total = nl + 1
    live = np.ones(total, dtype=np.uint32)
    live[4] = 0
    fn = general(rng, dist, (total, 16))
    add_near_twins(rng, fn, np.flatnonzero(live), nl // 8)
    fo = general(rng, dist, (8000 if nl <= UMMA_MAX_LIVE else 4000, 16))
    ref = Ref(oracle, fo, fn, live)
    assert ref.near_ties() >= 100, ref.near_ties()   # the bound check is not vacuous
    p = provider_with(gp, fn, live)
    for v in VARIANTS:
        ref.check(run(p, fo, v), v, "B-" + dist)


# ---- family C: cancellation --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K,nl", [(16, 512), (16, 2100), (17, 300)])
def test_cancellation(gp, oracle, K, nl):
    """Objects [L, -L, x2 ...] against nodes [1 + d, 1 + d', y2 ...] with L ~ 1e4, |d| <= 1e-5: |cost| ~ 0.2 while
    sum |a b| ~ 2.5e4.  The fp32 rounding of L (1 + d) alone is ~5e-4, so no fp32 implementation meets an error bound stated
    against |cost|: the old rule (index equal unless the gap is <= 1e-5 |cost|) rejects even the exact-order fmaf argmin for
    1-2 % of the objects, checked below.  The rules of this module hold."""
    rng = np.random.default_rng(K * 1000 + nl)
    total = nl + 1
    live = np.ones(total, dtype=np.uint32)
    live[4] = 0
    n = 12000 if nl <= UMMA_MAX_LIVE else 6000
    L = rng.uniform(0.5e4, 2e4, n)
    fo = np.concatenate([L[:, None], -L[:, None], rng.uniform(-0.01, 0.01, (n, K - 2))], axis=1).astype(np.float32)
    fn = np.concatenate([1 + rng.uniform(-1e-5, 1e-5, (total, 2)), rng.uniform(-1, 1, (total, K - 2))], axis=1).astype(np.float32)
    ref = Ref(oracle, fo, fn, live)
    # the old rule (index equal unless gap <= 1e-5 |cost|, chosen cost within 1e-5 |cost|) fails the exact-order fp32 argmin
    old_tol = 1e-5 * np.abs(ref.c64) + 1e-12
    old_ok = ((ref.idx32 == ref.idx64) | (ref.gap <= old_tol)) & (np.abs(ref.cost64(ref.idx32) - ref.c64) <= old_tol)
    assert (~old_ok).sum() >= 50, (~old_ok).sum()
    assert ref.near_ties() >= 100, ref.near_ties()
    p = provider_with(gp, fn, live)
    for v in VARIANTS if K == 16 else ["ffma"]:
        ref.check(run(p, fo, v), v, "C")


# ---- family D: power-of-two scaling --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K,nl", [(16, 512), (16, 48), (16, 2100), (5, 100)])
def test_power_of_two_scaling_changes_no_index(gp, oracle, K, nl):
    """|x| in [2^-4, 1] or 0; objects scaled by 2^s, nodes by 2^t with s + t in [-40, 60]: every bf16 piece and product stays
    normal and nothing overflows, so each path's indices must equal its own unscaled run (no absolute epsilon, no narrower type)."""
    rng = np.random.default_rng(K * 7 + nl)
    total = nl + 1
    live = np.ones(total, dtype=np.uint32)
    live[4] = 0

    def feats(shape):
        x = rng.choice([-1.0, 1.0], shape) * 2.0 ** rng.uniform(-4, 0, shape)
        return np.where(rng.random(shape) < 0.1, 0.0, x).astype(np.float32)

    fn, fo = feats((total, K)), feats((6000 if nl <= UMMA_MAX_LIVE else 2000, K))
    base_ref = Ref(oracle, fo, fn, live)
    p = provider_with(gp, fn, live)
    base = {v: run(p, fo, v, resident=False) for v in VARIANTS}
    for v in VARIANTS:
        base_ref.check(base[v], v, "D")
    for s, t in ((-20, -20), (30, 30), (0, 60), (-40, 0), (50, -45)):
        q = provider_with(gp, fn * np.float32(2.0 ** t), live)
        for v in VARIANTS:
            got = run(q, fo * np.float32(2.0 ** s), v, resident=(s, t) == (30, 30))
            bad = np.flatnonzero(got != base[v])
            assert bad.size == 0, (s, t, v, bad.size, bad[:5])


# ---- membership changes rebuild the compacted operands ---------------------------------------------------------------------------
def test_membership_sequence(gp, oracle):
    """Leave, join with features, join without features (zero row), crossing the tensor cores' capacity both ways, and a second
    set_nodes with new features; after every step both variants against the oracles on the new live set (family A: exact)."""
    rng = np.random.default_rng(5)
    K = 16
    M0 = 2040
    fn_all = np.zeros((4096, K), dtype=np.float32)   # by interned node index
    live = np.zeros(4096, dtype=np.uint32)
    fn_all[:M0] = exact_ints(rng, (M0, K))
    p = gp.GpuObjectPlacement()
    idx = p.set_nodes(addresses(M0), None, fn_all[:M0])
    assert (idx == np.arange(M0)).all()
    live[:M0] = 1
    fo = exact_ints(rng, (1500, K))
    n_next = [M0]

    def join(feat):
        j = p.node_upsert(addresses(1, port=8000 + n_next[0])[0], 1, feat)
        assert j == n_next[0]
        n_next[0] += 1
        fn_all[j] = 0 if feat is None else feat
        live[j] = 1
        return j

    def leave(j):
        p.node_set_active(j, False)
        live[j] = 0

    def check(step):
        total = n_next[0]
        ref = Ref(oracle, fo, fn_all[:total], live[:total])
        for v in VARIANTS:
            got = run(p, fo, v)
            ref.check(got, v, "A")
            bad = np.flatnonzero(got != ref.idx64)
            assert bad.size == 0, (step, v, bad.size, bad[:5])

    check("start")
    leave(5)
    check("leave")
    j = join(fn_all[700].copy())        # a twin of a live node, joined at a higher index: never wins
    check("join with features")
    assert p.node_count()[0] == j + 1
    join(None)                          # no features: a zero row, cost 0 for every object
    check("join without features")
    for _ in range(8):
        join(exact_ints(rng, K))        # 2049 live: the CUDA-core fallback
    assert live.sum() == 2049
    check("over capacity")
    leave(0)
    leave(j)
    check("back under capacity")
    # a second set_nodes replaces every feature row and deactivates the nodes it does not list
    keep = np.arange(100, 1100)
    new = exact_ints(rng, (len(keep), K))
    p.set_nodes([addresses(M0)[i] for i in keep], None, new)
    fn_all[:] = 0
    live[:] = 0
    fn_all[keep] = new
    live[keep] = 1
    check("second set_nodes")
