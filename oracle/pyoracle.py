"""ctypes/numpy wrappers around the CPU oracle libraries (test infrastructure).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import
this module; the product package rio_rs_b200 never does.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_BUILD = os.path.join(_HERE, "_build")
NONE = 0xFFFFFFFF


def build(force=False):
    """Compile the oracle libraries (plain gcc/g++, seconds)."""
    so1 = os.path.join(_BUILD, "librio_oracle.so")
    so2 = os.path.join(_BUILD, "librio_dirmodel.so")
    srcs = [os.path.join(_HERE, "rio_oracle.c"), os.path.join(_HERE, "directory_model.cpp")]
    fresh = all(os.path.exists(s) for s in (so1, so2)) and min(os.path.getmtime(so1), os.path.getmtime(so2)) >= max(
        os.path.getmtime(s) for s in srcs
    )
    if force or not fresh:
        env = dict(os.environ)
        # the image exports CC=/opt/gcc/bin/gcc; either compiler works (no OpenMP needed)
        subprocess.check_call(["make", "-C", _HERE, "-s"] + (["-B"] if force else []), env=env)
    return so1, so2


_lib = None
_dm = None


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t)) if a is not None else None


def lib():
    global _lib
    if _lib is None:
        so1, _ = build()
        L = C.CDLL(so1)
        u64p, u32p, f32p, f64p = (C.POINTER(C.c_uint64), C.POINTER(C.c_uint32), C.POINTER(C.c_float), C.POINTER(C.c_double))
        L.orc_mix64.restype = C.c_uint64
        L.orc_mix64.argtypes = [C.c_uint64]
        L.orc_fnv1a64.restype = C.c_uint64
        L.orc_fnv1a64.argtypes = [C.c_char_p, C.c_size_t]
        L.orc_object_key.restype = C.c_uint64
        L.orc_object_key.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t]
        L.orc_node_seed.restype = C.c_uint64
        L.orc_node_seed.argtypes = [C.c_char_p, C.c_size_t]
        L.orc_log2frac.restype = C.c_uint32
        L.orc_log2frac.argtypes = [C.c_uint32]
        L.orc_elog.restype = C.c_uint32
        L.orc_elog.argtypes = [C.c_uint32]
        L.orc_pair_hash.restype = C.c_uint32
        L.orc_pair_hash.argtypes = [C.c_uint64, C.c_uint64]
        L.orc_inv_weight.restype = C.c_uint32
        L.orc_inv_weight.argtypes = [C.c_uint32]
        L.orc_spill_hash.restype = C.c_uint32
        L.orc_spill_hash.argtypes = [C.c_uint64, C.c_uint32]
        L.orc_capacity.restype = C.c_uint32
        L.orc_capacity.argtypes = [C.c_uint64, C.c_uint32, C.c_uint64, C.c_uint32, C.c_uint32]
        L.orc_assign_hrw.restype = None
        L.orc_assign_hrw.argtypes = [u64p, C.c_size_t, u64p, u32p, u32p, C.c_uint32, u32p, u64p, u32p, C.c_int]
        L.orc_assign_bounded.restype = C.c_uint32
        L.orc_assign_bounded.argtypes = [u64p, C.c_size_t, u64p, u32p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, u32p, u32p, C.c_int]
        L.orc_assign_affinity.restype = None
        L.orc_assign_affinity.argtypes = [f32p, f32p, u32p, C.c_size_t, C.c_uint32, C.c_uint32, u32p, f64p, f64p, C.c_int]
        L.orc_assign_affinity_f32.restype = None
        L.orc_assign_affinity_f32.argtypes = [f32p, f32p, u32p, C.c_size_t, C.c_uint32, C.c_uint32, u32p, C.c_int]
        L.orc_affinity_pair_cost_f32.restype = None
        L.orc_affinity_pair_cost_f32.argtypes = [f32p, f32p, u32p, u32p, C.c_size_t, C.c_uint32, f32p, C.c_int]
        L.orc_assign_hrw2.restype = None
        L.orc_assign_hrw2.argtypes = [u64p, C.c_size_t, u64p, u32p, u32p, C.c_uint32, C.c_uint32, u32p, C.c_int]
        L.orc_assign_bounded_hrw2.restype = C.c_uint32
        L.orc_assign_bounded_hrw2.argtypes = [u64p, C.c_size_t, u64p, u32p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, u32p, u32p, C.c_int]
        L.orc_hrw2_v.restype = C.c_uint32
        L.orc_hrw2_v.argtypes = [C.c_uint64, C.c_uint64]
        L.orc_hrw2_pos.restype = C.c_uint64
        L.orc_hrw2_pos.argtypes = [C.c_uint64]
        L.orc_hrw2_level_seed.restype = C.c_uint64
        L.orc_hrw2_level_seed.argtypes = [C.c_uint32]
        L.orc_hrw2_threshold.restype = C.c_uint32
        L.orc_hrw2_threshold.argtypes = [C.c_uint64, C.c_uint64]
        L.orc_synth_keys.restype = None
        L.orc_synth_keys.argtypes = [u64p, C.c_size_t, C.c_uint64, C.c_uint64]
        L.orc_counts.restype = None
        L.orc_counts.argtypes = [u32p, C.c_size_t, C.c_uint32, u32p]
        _lib = L
    return _lib


# ---- solver oracle --------------------------------------------------------------------------------
def object_key(type_, id_):
    t, i = type_.encode(), id_.encode()
    return lib().orc_object_key(t, len(t), i, len(i))


def node_seed(address):
    a = address.encode()
    return lib().orc_node_seed(a, len(a))


def synth_keys(n, seed, first=0):
    out = np.empty(n, dtype=np.uint64)
    lib().orc_synth_keys(_p(out, C.c_uint64), n, first, seed)
    return out


def synth_nodes(M, weight_seed=7, uniform=False):
    """SURVEY 8d: addresses "10.0.(j>>8).(j&255):5000", weights u32 in [1,16] (seed 7) or all ones."""
    addrs = ["10.0.%d.%d:5000" % (j >> 8, j & 255) for j in range(M)]
    seeds = np.array([node_seed(a) for a in addrs], dtype=np.uint64)
    if uniform:
        w = np.ones(M, dtype=np.uint32)
    else:
        L = lib()
        w = np.array([1 + (L.orc_mix64((j + 1) * 0x9E3779B97F4A7C15 % 2**64 ^ weight_seed) % 16) for j in range(M)], dtype=np.uint32)
    return addrs, seeds, w


def assign_hrw(keys, seeds, weights, mask=None, threads=1, want_score=False):
    keys = np.ascontiguousarray(keys, dtype=np.uint64)
    seeds = np.ascontiguousarray(seeds, dtype=np.uint64)
    weights = np.ascontiguousarray(weights, dtype=np.uint32)
    n, M = len(keys), len(seeds)
    idx = np.empty(n, dtype=np.uint32)
    sc = np.empty(n, dtype=np.uint64) if want_score else None
    uu = np.empty(n, dtype=np.uint32) if want_score else None
    if mask is not None:
        mask = np.ascontiguousarray(mask, dtype=np.uint32)
    lib().orc_assign_hrw(_p(keys, C.c_uint64), n, _p(seeds, C.c_uint64), _p(weights, C.c_uint32), _p(mask, C.c_uint32), M,
                         _p(idx, C.c_uint32), _p(sc, C.c_uint64), _p(uu, C.c_uint32), threads)
    return (idx, sc, uu) if want_score else idx


HRW2_DEFAULT_BITS = 12


def assign_hrw2(keys, seeds, weights, mask=None, bits=HRW2_DEFAULT_BITS, threads=1):
    """Hierarchical weighted rendezvous with fan-out 2 (DESIGN.md 3.8)."""
    keys = np.ascontiguousarray(keys, dtype=np.uint64)
    seeds = np.ascontiguousarray(seeds, dtype=np.uint64)
    weights = np.ascontiguousarray(weights, dtype=np.uint32)
    n, M = len(keys), len(seeds)
    idx = np.empty(n, dtype=np.uint32)
    if mask is not None:
        mask = np.ascontiguousarray(mask, dtype=np.uint32)
    lib().orc_assign_hrw2(_p(keys, C.c_uint64), n, _p(seeds, C.c_uint64), _p(weights, C.c_uint32), _p(mask, C.c_uint32), M, bits,
                          _p(idx, C.c_uint32), threads)
    return idx


def assign_bounded(keys, seeds, weights, cap_num=5, cap_den=4, max_rounds=4, threads=1):
    keys = np.ascontiguousarray(keys, dtype=np.uint64)
    seeds = np.ascontiguousarray(seeds, dtype=np.uint64)
    weights = np.ascontiguousarray(weights, dtype=np.uint32)
    n, M = len(keys), len(seeds)
    idx = np.empty(n, dtype=np.uint32)
    counts = np.zeros(M, dtype=np.uint32)
    passes = lib().orc_assign_bounded(_p(keys, C.c_uint64), n, _p(seeds, C.c_uint64), _p(weights, C.c_uint32), M, cap_num, cap_den,
                                      max_rounds, _p(idx, C.c_uint32), _p(counts, C.c_uint32), threads)
    return idx, counts, passes


def assign_bounded_hrw2(keys, seeds, weights, cap_num=5, cap_den=4, max_rounds=4, bits=HRW2_DEFAULT_BITS, threads=1):
    keys = np.ascontiguousarray(keys, dtype=np.uint64)
    seeds = np.ascontiguousarray(seeds, dtype=np.uint64)
    weights = np.ascontiguousarray(weights, dtype=np.uint32)
    n, M = len(keys), len(seeds)
    idx = np.empty(n, dtype=np.uint32)
    counts = np.zeros(M, dtype=np.uint32)
    passes = lib().orc_assign_bounded_hrw2(_p(keys, C.c_uint64), n, _p(seeds, C.c_uint64), _p(weights, C.c_uint32), M, bits, cap_num,
                                           cap_den, max_rounds, _p(idx, C.c_uint32), _p(counts, C.c_uint32), threads)
    return idx, counts, passes


def assign_affinity(fobj, fnode, weights, threads=1):
    fobj = np.ascontiguousarray(fobj, dtype=np.float32)
    fnode = np.ascontiguousarray(fnode, dtype=np.float32)
    weights = np.ascontiguousarray(weights, dtype=np.uint32)
    n, K = fobj.shape
    M = fnode.shape[0]
    idx = np.empty(n, dtype=np.uint32)
    cost = np.empty(n, dtype=np.float64)
    gap = np.empty(n, dtype=np.float64)
    lib().orc_assign_affinity(_p(fobj, C.c_float), _p(fnode, C.c_float), _p(weights, C.c_uint32), n, M, K, _p(idx, C.c_uint32),
                              _p(cost, C.c_double), _p(gap, C.c_double), threads)
    return idx, cost, gap


def assign_affinity_f32(fobj, fnode, weights, threads=1):
    """Implementation restatement, not spec: the CUDA-core kernels' fp32 arithmetic (fmaf over k ascending, strict < in node
    order).  Their indices must equal this exactly."""
    fobj = np.ascontiguousarray(fobj, dtype=np.float32)
    fnode = np.ascontiguousarray(fnode, dtype=np.float32)
    weights = np.ascontiguousarray(weights, dtype=np.uint32)
    n, K = fobj.shape
    idx = np.empty(n, dtype=np.uint32)
    lib().orc_assign_affinity_f32(_p(fobj, C.c_float), _p(fnode, C.c_float), _p(weights, C.c_uint32), n, fnode.shape[0], K, _p(idx, C.c_uint32),
                                  threads)
    return idx


def affinity_pair_cost_f32(fobj, fnode, obj, node, threads=1):
    """fp32 fmaf cost -sum_k fobj[obj[q],k] * fnode[node[q],k] for each pair q, with the arithmetic of assign_affinity_f32."""
    fobj = np.ascontiguousarray(fobj, dtype=np.float32)
    fnode = np.ascontiguousarray(fnode, dtype=np.float32)
    obj = np.ascontiguousarray(obj, dtype=np.uint32)
    node = np.ascontiguousarray(node, dtype=np.uint32)
    assert obj.shape == node.shape and (obj < fobj.shape[0]).all() and (node < fnode.shape[0]).all()
    out = np.empty(obj.shape, dtype=np.float32)
    lib().orc_affinity_pair_cost_f32(_p(fobj, C.c_float), _p(fnode, C.c_float), _p(obj, C.c_uint32), _p(node, C.c_uint32), obj.size, fobj.shape[1],
                                     _p(out, C.c_float), threads)
    return out


def counts(idx, M):
    idx = np.ascontiguousarray(idx, dtype=np.uint32)
    out = np.zeros(M, dtype=np.uint32)
    lib().orc_counts(_p(idx, C.c_uint32), len(idx), M, _p(out, C.c_uint32))
    return out


# ---- directory / service-policy oracle -----------------------------------------------------------
def dm():
    global _dm
    if _dm is None:
        _, so2 = build()
        D = C.CDLL(so2)
        D.dm_new.restype = C.c_void_p
        D.dm_free.argtypes = [C.c_void_p]
        D.dm_update.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.c_char_p]
        D.dm_lookup.restype = C.c_int64
        D.dm_lookup.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.c_char_p, C.c_size_t]
        D.dm_clean_server.argtypes = [C.c_void_p, C.c_char_p]
        D.dm_remove.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p]
        D.dm_len.restype = C.c_uint64
        D.dm_len.argtypes = [C.c_void_p]
        D.dm_member_push.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.c_int]
        D.dm_member_remove.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p]
        D.dm_member_set_active.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.c_int]
        D.dm_member_is_active.restype = C.c_int
        D.dm_member_is_active.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p]
        D.dm_get_or_create_placement.restype = C.c_int64
        D.dm_get_or_create_placement.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.c_char_p, C.c_char_p, C.c_size_t]
        D.dm_check_address_mismatch.restype = C.c_int
        D.dm_check_address_mismatch.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p]
        D.dm_bench_resolve.restype = C.c_double
        D.dm_bench_resolve.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32, C.c_int, C.POINTER(C.c_uint64)]
        D.dm_bench_lookup.restype = C.c_double
        D.dm_bench_lookup.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint64)]
        _dm = D
    return _dm


class DirectoryModel:
    """LocalObjectPlacement restatement (local.rs:12-68) + membership + service policy."""

    def __init__(self):
        self._d = dm()
        self._h = C.c_void_p(self._d.dm_new())
        self._buf = C.create_string_buffer(256)

    def __del__(self):
        try:
            self._d.dm_free(self._h)
        except Exception:
            pass

    def prepare(self):
        return None

    def update(self, type_, id_, address):
        self._d.dm_update(self._h, type_.encode(), id_.encode(), None if address is None else address.encode())

    def lookup(self, type_, id_):
        n = self._d.dm_lookup(self._h, type_.encode(), id_.encode(), self._buf, 256)
        return None if n < 0 else self._buf.raw[:n].decode()

    def clean_server(self, address):
        self._d.dm_clean_server(self._h, address.encode())

    def remove(self, type_, id_):
        self._d.dm_remove(self._h, type_.encode(), id_.encode())

    def __len__(self):
        return int(self._d.dm_len(self._h))

    # membership (cluster/storage/local.rs)
    def member_push(self, ip, port, active=True):
        self._d.dm_member_push(self._h, ip.encode(), port.encode(), int(active))

    def member_remove(self, ip, port):
        self._d.dm_member_remove(self._h, ip.encode(), port.encode())

    def member_set_active(self, ip, port, active):
        self._d.dm_member_set_active(self._h, ip.encode(), port.encode(), int(active))

    def member_is_active(self, ip, port):
        return bool(self._d.dm_member_is_active(self._h, ip.encode(), port.encode()))

    def get_or_create_placement(self, self_address, type_, id_):
        n = self._d.dm_get_or_create_placement(self._h, self_address.encode(), type_.encode(), id_.encode(), self._buf, 256)
        return self._buf.raw[:n].decode()


ADDR_LOCAL, ADDR_REDIRECT, ADDR_DEALLOCATE, ADDR_MALFORMED = 0, 1, 2, 3


def _dm_check_address_mismatch(self, self_address, server_address):
    """service.rs:261-298 -> ADDR_LOCAL (Ok) | ADDR_REDIRECT | ADDR_DEALLOCATE (clean_server applied) | ADDR_MALFORMED"""
    return int(self._d.dm_check_address_mismatch(self._h, self_address.encode(), server_address.encode()))


DirectoryModel.check_address_mismatch = _dm_check_address_mismatch


def bench_resolve(n, M, threads, first=0):
    placed = C.c_uint64(0)
    s = dm().dm_bench_resolve(first, n, M, threads, C.byref(placed))
    return s, int(placed.value)


def bench_lookup(n, M, reps):
    hits = C.c_uint64(0)
    s = dm().dm_bench_lookup(n, M, reps, C.byref(hits))
    return s, int(hits.value)
