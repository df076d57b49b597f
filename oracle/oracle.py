"""ctypes binding of oracle/libkroracle.so — TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this
(see oracle/kr_oracle.h).  The product package kuberay_b200/ never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from kuberay_b200 import abi

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
INDEXED, NS_SCAN = 0, 1


def build(force: bool = False) -> str:
    so = os.path.join(_HERE, "libkroracle.so")
    srcs = [os.path.join(_HERE, f) for f in ("kr_oracle.c", "kr_oracle.h")] + [os.path.join(_HERE, "..", "include", "kr_engine.h")]
    stale = force or not os.path.exists(so) or any(os.path.exists(s) and os.path.getmtime(s) > os.path.getmtime(so) for s in srcs)
    if stale:
        subprocess.check_call(["make", "-s", "-C", _HERE, "-B", "libkroracle.so"])
    return so


def build_native(out_dir: str) -> str:
    """The CPU arm's build: same source, -O3 -march=native for the host it runs on, into out_dir (bench.py only; never shipped)."""
    so = os.path.join(out_dir, "libkroracle_native.so")
    subprocess.check_call(["make", "-s", "-C", _HERE, "-B", "native", "NATIVE=" + so])
    return so


def _bind(L: C.CDLL) -> C.CDLL:
    L.kr_oracle_run.argtypes = [C.POINTER(abi.kr_snapshot_bufs), C.POINTER(abi.kr_sizes), C.POINTER(abi.kr_flags),
                                C.POINTER(abi.kr_oracle_out), C.c_int, C.c_int]
    L.kr_oracle_run.restype = C.c_int
    L.kr_oracle_run_range.argtypes = L.kr_oracle_run.argtypes + [C.c_uint32, C.c_uint32]
    L.kr_oracle_run_range.restype = C.c_int
    L.kr_oracle_ctx_create.argtypes = [C.POINTER(abi.kr_snapshot_bufs), C.POINTER(abi.kr_sizes), C.POINTER(C.c_void_p)]
    L.kr_oracle_ctx_create.restype = C.c_int
    L.kr_oracle_ctx_run.argtypes = [C.c_void_p, C.POINTER(abi.kr_flags), C.POINTER(abi.kr_oracle_out), C.c_int, C.c_int]
    L.kr_oracle_ctx_run.restype = C.c_int
    L.kr_oracle_ctx_run_range.argtypes = L.kr_oracle_ctx_run.argtypes + [C.c_uint32, C.c_uint32, C.c_int]
    L.kr_oracle_ctx_run_range.restype = C.c_int
    L.kr_oracle_ctx_destroy.argtypes = [C.c_void_p]
    L.kr_oracle_ctx_destroy.restype = None
    L.kr_oracle_sha1_impl.restype = C.c_int
    L.kr_oracle_hash32.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p]
    L.kr_oracle_sha1.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p]
    L.kr_oracle_desired_replicas.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_uint32]
    L.kr_oracle_desired_replicas.restype = C.c_int32
    L.kr_oracle_should_delete.argtypes = [C.c_uint32]
    L.kr_oracle_should_delete.restype = C.c_int
    return L


def load(path: str) -> C.CDLL:
    """Load another build of the oracle (bench.py: the -march=native CPU arm)."""
    return _bind(C.CDLL(path))


class Context:
    """One snapshot's shared index (kr_oracle_ctx): built once, reused by every run — as controller-runtime's informer cache
    is between reconciles.  Keeps the snapshot's arrays and one preallocated result set alive."""

    def __init__(self, snap, L: C.CDLL | None = None, create_cap: int = 1 << 20):
        self.L = L or lib()
        self.snap = snap
        self.sizes = snap.sizes()
        self.bufs = snap.bufs()
        self.res = abi.Results(self.sizes, create_cap)
        self.out = _out_struct(self.res)
        self.h = C.c_void_p()
        rc = self.L.kr_oracle_ctx_create(C.byref(self.bufs), C.byref(self.sizes), C.byref(self.h))
        if rc != 0:
            raise RuntimeError(f"kr_oracle_ctx_create failed: {rc}")

    def run_range(self, flags: abi.kr_flags, c0: int, c1: int, list_mode: int = NS_SCAN, threads: int = 1, reps: int = 1) -> abi.Results:
        rc = self.L.kr_oracle_ctx_run_range(self.h, C.byref(flags), C.byref(self.out), list_mode, threads, c0, c1, reps)
        if rc != 0:
            raise RuntimeError(f"kr_oracle_ctx_run_range failed: {rc}")
        return self.res

    def run(self, flags: abi.kr_flags, list_mode: int = INDEXED, threads: int = 1) -> abi.Results:
        rc = self.L.kr_oracle_ctx_run(self.h, C.byref(flags), C.byref(self.out), list_mode, threads)
        if rc != 0:
            raise RuntimeError(f"kr_oracle_ctx_run failed: {rc}")
        self.res.n_create_total, self.res.n_orphans, self.res.n_actions = self.out.n_create_total, self.out.n_orphans, self.out.n_actions
        return self.res

    def close(self):
        if self.h:
            self.L.kr_oracle_ctx_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def lib() -> C.CDLL:
    global _LIB
    if _LIB is None:
        L = _bind(C.CDLL(os.environ.get("KR_ORACLE_LIB") or build()))  # KR_ORACLE_LIB: e.g. the ASan/UBSan build (make -C oracle asan)
        _LIB = L
    return _LIB


def _out_struct(res: abi.Results) -> abi.kr_oracle_out:
    o = abi.kr_oracle_out()
    for name in abi.Results.FIELDS:
        setattr(o, name, getattr(res, name).ctypes.data)
    o.create_cap = res.create_idx.size
    return o


def default_create_cap(snap) -> int:
    """Upper bound on sum(n_create): sum over groups of max(expected, 0) — computed with the oracle's own scalar."""
    L = lib()
    tot = 0
    for g in range(snap.dims["groups"]):
        e = L.kr_oracle_desired_replicas(int(snap.g_replicas[g]), int(snap.g_min[g]), int(snap.g_max[g]), int(snap.g_num_hosts[g]), int(snap.g_flags[g]))
        tot += max(e, 0)
    return tot + 1


def run(snap, flags: abi.kr_flags, list_mode: int = INDEXED, threads: int = 1, create_cap: int | None = None) -> abi.Results:
    sizes = snap.sizes()
    if create_cap is None:
        create_cap = min(default_create_cap(snap), 1 << 27)
    res = abi.Results(sizes, create_cap)
    o = _out_struct(res)
    bufs = snap.bufs()
    rc = lib().kr_oracle_run(C.byref(bufs), C.byref(sizes), C.byref(flags), C.byref(o), list_mode, threads)
    if rc != 0:
        raise RuntimeError(f"kr_oracle_run failed: {rc}")
    res.n_create_total, res.n_orphans, res.n_actions = o.n_create_total, o.n_orphans, o.n_actions
    return res


def run_range(snap, flags: abi.kr_flags, c0: int, c1: int, list_mode: int = NS_SCAN, threads: int = 1, res: abi.Results | None = None) -> abi.Results:
    sizes = snap.sizes()
    if res is None:
        res = abi.Results(sizes, 1 << 20)
    o = _out_struct(res)
    bufs = snap.bufs()
    rc = lib().kr_oracle_run_range(C.byref(bufs), C.byref(sizes), C.byref(flags), C.byref(o), list_mode, threads, c0, c1)
    if rc != 0:
        raise RuntimeError(f"kr_oracle_run_range failed: {rc}")
    return res


def hash32(data: bytes) -> str:
    out = C.create_string_buffer(32)
    buf = C.create_string_buffer(data, len(data)) if data else C.create_string_buffer(1)
    lib().kr_oracle_hash32(buf, len(data), out)
    return out.raw.decode("ascii")


def sha1(data: bytes) -> bytes:
    out = C.create_string_buffer(20)
    buf = C.create_string_buffer(data, len(data)) if data else C.create_string_buffer(1)
    lib().kr_oracle_sha1(buf, len(data), out)
    return out.raw


def desired_replicas(replicas, min_, max_, num_hosts, suspend=False) -> int:
    gf = (abi.GF_SUSPEND if suspend else 0) | (abi.GF_REPLICAS_NIL if replicas is None else 0) | \
         (abi.GF_MIN_NIL if min_ is None else 0) | (abi.GF_MAX_NIL if max_ is None else 0)
    return lib().kr_oracle_desired_replicas(replicas or 0, min_ or 0, max_ or 0, num_hosts, gf)
