"""certificate_stark_b200 -- B200-native proving backend for the STARK prover of toposware/certificate-stark.

The product is ``lib/libcsg.so`` (hand-written sm_100a CUDA kernels + a C++ host driver) behind the C ABI declared in
``include/csg.h``.  This module is the thin host-side mirror of the reference's example/prover interface
(``TransactionExample::{new, prove}`` at /root/reference/src/lib.rs:75-141, ``ProofOptions`` at src/lib.rs:78-86, and the
five sub-AIR examples), implemented over that C ABI with ctypes.  There is no CPU fallback: if the shared library is
missing or no CUDA device can be opened, every entry point raises.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional
import os
import subprocess
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get("CSG_LIB", ROOT / "lib" / "libcsg.so"))
P = 0x4180000000000001  # f63 modulus (/root/reference/src/range/tests.rs:59)

AIR_TRANSACTION, AIR_MERKLE_UPDATE, AIR_MERKLE_INIT, AIR_SCHNORR, AIR_RANGE, AIR_RESCUE = range(6)
HASH_BLAKE3_256, HASH_SHA3_256 = 2, 3
FIELD_EXTENSION_NONE, FIELD_EXTENSION_QUADRATIC, FIELD_EXTENSION_CUBIC = 1, 2, 3
REPR_CANONICAL, REPR_MONTGOMERY = 0, 1   # csg.h: representation of the trace words crossing the boundary
TRACE_WIDTH = {AIR_TRANSACTION: 94, AIR_MERKLE_UPDATE: 65, AIR_MERKLE_INIT: 58, AIR_SCHNORR: 56, AIR_RANGE: 2, AIR_RESCUE: 14}
_ERRORS = {1: "invalid argument", 2: "CUDA error", 3: "call out of order", 4: "unsupported", 5: "random coin failure"}


class CsgError(RuntimeError):
    pass


class ProofOptions(C.Structure):
    """ProofOptions::new(num_queries, blowup_factor, grinding_factor, hash_fn, field_extension, fri_folding_factor,
    fri_max_remainder_size) -- same argument order as the reference (src/lib.rs:78-86)."""
    _fields_ = [(n, C.c_uint32) for n in ("num_queries", "blowup_factor", "grinding_factor", "hash_fn", "field_extension",
                                          "fri_folding_factor", "fri_max_remainder_size")]

    def __init__(self, num_queries=42, blowup_factor=8, grinding_factor=0, hash_fn=HASH_BLAKE3_256,
                 field_extension=FIELD_EXTENSION_NONE, fri_folding_factor=4, fri_max_remainder_size=256):
        super().__init__(num_queries, blowup_factor, grinding_factor, hash_fn, field_extension, fri_folding_factor, fri_max_remainder_size)


class ShardPlan(C.Structure):
    """csg_shard_plan: what one rank of a coset-sharded proof owns"""
    _fields_ = [(n, C.c_uint32) for n in ("first_coset", "num_cosets", "first_ce_coset", "num_ce_cosets", "first_column", "num_columns", "columns_per_rank")]


class Timings(C.Structure):
    _fields_ = [(n, C.c_float) for n in ("h2d", "lde", "commit_trace", "constraints", "composition", "ood_deep", "fri", "queries", "total")] + \
               [("kernel_launches", C.c_uint64)] + [(n, C.c_float) for n in ("cons_rescue", "cons_ecc_banks", "cons_ecc_final", "cons_rest", "comm", "cons_ecc_low")] + \
               [("stage_launches", C.c_uint32 * 7), ("batch_build", C.c_float)]
    STAGES = ("lde", "commit_trace", "constraints", "composition", "ood_deep", "fri", "queries")

    def as_dict(self):
        d = {n: getattr(self, n) for n, _ in self._fields_ if n != "stage_launches"}
        d["stage_launches"] = dict(zip(self.STAGES, [int(v) for v in self.stage_launches]))
        return d


def build(force: bool = False) -> Path:
    """Compile lib/libcsg.so for sm_100a (nvcc cross-compiles without a GPU)."""
    if force:
        subprocess.check_call(["make", "-C", str(ROOT / "csrc"), "clean"], stdout=subprocess.DEVNULL)
    subprocess.check_call(["make", "-C", str(ROOT / "csrc"), "-j", str(min(8, os.cpu_count() or 1))], stdout=subprocess.DEVNULL)
    return LIB_PATH


_lib = None
_u64p, _u8p, _szp = C.POINTER(C.c_uint64), C.POINTER(C.c_uint8), C.POINTER(C.c_size_t)


def lib() -> C.CDLL:
    """The loaded C-ABI library.  Raises if it has not been built: there is no other implementation to fall back to."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise CsgError(f"{LIB_PATH} is missing: run certificate_stark_b200.build() (needs nvcc); there is no CPU fallback")
    L = C.CDLL(str(LIB_PATH))
    vp, opt = C.c_void_p, C.POINTER(ProofOptions)
    sig = {
        "csg_create": (vp, [C.c_int]), "csg_destroy": (None, [vp]), "csg_last_error": (C.c_char_p, [vp]), "csg_free": (None, [vp]),
        "csg_prove": (C.c_int, [vp, C.c_int, _u64p, C.c_int, C.c_size_t, _u64p, C.c_size_t, opt, C.POINTER(_u8p), _szp]),
        "csg_prove_many": (C.c_int, [vp, C.c_int, C.c_size_t, C.POINTER(_u64p), C.c_int, C.c_size_t, _u64p, C.c_size_t, opt, C.POINTER(_u8p), _szp]),
        "csg_prove_many_device": (C.c_int, [vp, C.c_int, C.c_size_t, vp, C.c_int, C.c_size_t, _u64p, C.c_size_t, opt, C.POINTER(_u8p), _szp]),
        "csg_build_traces_many_rescue": (C.c_int, [vp, _u64p, C.c_size_t, C.c_size_t, vp, _u64p]),
        "csg_build_traces_many_schnorr": (C.c_int, [vp, vp, vp, _u64p]), "csg_build_traces_many_merkle_update": (C.c_int, [vp, vp, vp, _u64p]),
        "csg_build_traces_many_transaction": (C.c_int, [vp, vp, vp, _u64p]),
        "csg_prove_columns": (C.c_int, [vp, C.c_int, C.POINTER(_u64p), C.c_int, C.c_size_t, _u64p, C.c_size_t, opt, C.POINTER(_u8p), _szp]),
        "csg_set_air": (C.c_int, [vp, C.c_int, C.c_size_t, opt, _u64p, C.c_size_t]),
        "csg_load_trace": (C.c_int, [vp, _u64p, C.c_int]), "csg_reload_resident_trace": (C.c_int, [vp]),
        "csg_prove_loaded": (C.c_int, [vp, C.POINTER(_u8p), _szp]),
        "csg_prove_trace": (C.c_int, [vp, _u64p, C.c_int, C.POINTER(_u8p), _szp]),
        "csg_prefetch_trace": (C.c_int, [vp, _u64p, C.c_int]),
        "csg_prove_prefetched": (C.c_int, [vp, _u64p, C.c_int, C.POINTER(_u8p), _szp]),
        "csg_host_alloc": (vp, [C.c_size_t]), "csg_host_free": (None, [vp]), "csg_host_register": (C.c_int, [vp, C.c_size_t]),
        "csg_host_unregister": (C.c_int, [vp]),
        "csg_extend_and_commit_trace": (C.c_int, [vp, _u8p]), "csg_eval_constraints": (C.c_int, [vp, _u64p, _u64p]),
        "csg_commit_composition": (C.c_int, [vp, _u8p]), "csg_ood": (C.c_int, [vp, C.c_uint64, _u64p, _u64p, _u64p]),
        "csg_deep": (C.c_int, [vp, _u64p, _u64p, _u64p]), "csg_fri_commit_layer": (C.c_int, [vp, _u8p]),
        "csg_fri_fold": (C.c_int, [vp, C.c_uint64]), "csg_fri_fold_ext": (C.c_int, [vp, _u64p]),
        "csg_ood_ext": (C.c_int, [vp, _u64p, _u64p, _u64p, _u64p]), "csg_fri_remainder": (C.c_int, [vp, _u64p, C.c_size_t, _szp]),
        "csg_open_trace": (C.c_int, [vp, _u64p, C.c_size_t, _u64p, _u8p, C.c_size_t, _szp]),
        "csg_open_composition": (C.c_int, [vp, _u64p, C.c_size_t, _u64p, _u8p, C.c_size_t, _szp]),
        "csg_open_fri_layer": (C.c_int, [vp, C.c_size_t, _u64p, C.c_size_t, _u64p, _u8p, C.c_size_t, _szp]),
        "csg_verify": (C.c_int, [C.c_int, _u64p, C.c_size_t, _u8p, C.c_size_t]),
        "csg_verify_with_options": (C.c_int, [C.c_int, _u64p, C.c_size_t, _u8p, C.c_size_t, opt]),
        "csg_get_timings": (C.c_int, [vp, C.POINTER(Timings)]),
        "csg_dist_unique_id": (C.c_int, [_u8p]), "csg_dist_init": (C.c_int, [vp, C.c_int, C.c_int, _u8p]),
        "csg_dist_plan": (C.c_int, [C.c_int, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(ShardPlan)]),
        "csg_dist_trace_chunks": (C.c_int, [C.c_int, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.POINTER(C.c_uint32), C.c_size_t, C.POINTER(C.c_size_t)]),
        "csg_dist_init_local": (C.c_int, [C.POINTER(vp), C.c_int]), "csg_dist_info": (C.c_int, [vp, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
        "csg_timer_start": (C.c_int, [vp]), "csg_timer_stop": (C.c_int, [vp, C.POINTER(C.c_float)]),
        "csg_tx_batch_new": (vp, [C.c_uint64, C.c_size_t, C.c_uint]), "csg_tx_batch_free": (None, [vp]), "csg_tx_batch_size": (C.c_size_t, [vp]),
        "csg_tx_batch_roots": (None, [vp, _u64p, _u64p]),
        "csg_build_trace_transaction": (C.c_int, [vp, _u64p, _u64p]),
        "csg_build_trace_transaction_device": (C.c_int, [vp, vp]), "csg_download_trace": (C.c_int, [vp, _u64p]),
        "csg_tx_batch_build_device": (C.c_int, [vp, C.c_uint64, C.c_size_t, C.c_uint, _u64p]),
        "csg_build_trace_transaction_resident": (C.c_int, [vp]), "csg_download_batch_records": (C.c_int, [vp, _u64p, C.c_size_t]),
        "csg_tx_batch_pack": (C.c_size_t, [vp, _u64p]), "csg_sig_batch_pack": (C.c_size_t, [vp, _u64p]),
        "csg_build_trace_merkle_update_device": (C.c_int, [vp, vp]), "csg_build_trace_schnorr_device": (C.c_int, [vp, vp]), "csg_tx_batch_depth": (C.c_uint, [vp]), "csg_build_trace_merkle_update": (C.c_int, [vp, _u64p, _u64p]),
        "csg_build_trace_merkle_init": (C.c_int, [_u64p, _u64p, C.c_uint64, _u64p, _u64p]),
        "csg_sig_batch_new": (vp, [C.c_uint64, C.c_size_t]), "csg_sig_batch_free": (None, [vp]), "csg_sig_batch_size": (C.c_size_t, [vp]),
        "csg_build_trace_schnorr": (C.c_int, [vp, _u64p, _u64p]), "csg_build_trace_range": (C.c_int, [C.c_uint64, _u64p, _u64p]),
        "csg_build_trace_rescue": (C.c_int, [_u64p, C.c_size_t, _u64p, _u64p]),
        "csg_k_lde": (C.c_int, [vp, _u64p, C.c_size_t, C.c_size_t, C.c_size_t, _u64p]),
        "csg_k_hash_rows": (C.c_int, [vp, C.c_int, _u64p, C.c_size_t, C.c_size_t, _u8p]),
        "csg_k_merkle": (C.c_int, [vp, C.c_int, _u8p, C.c_size_t, _u8p]),
        "csg_k_fri_fold4": (C.c_int, [vp, _u64p, C.c_size_t, C.c_uint64, _u64p]),
        "csg_k_sweep": (C.c_int, [vp, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.POINTER(C.c_float)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args
    _lib = L
    return L


def _p64(a):
    return a.ctypes.data_as(_u64p)


def _p8(a):
    return a.ctypes.data_as(_u8p)


VERIFY_ERRORS = {16: "malformed proof", 17: "inconsistent out-of-domain constraint evaluations", 18: "proof of work check failed",
                 19: "trace query does not match the commitment", 20: "constraint query does not match the commitment", 21: "FRI verification failed",
                 22: "proof options weaker than the verifier's"}


def verify(air_id: int, pub: np.ndarray, proof: bytes, min_options: "ProofOptions | None" = None) -> int:
    """winterfell::verify::<Air>(proof, pub_inputs): 0 when the proof is accepted, else a key of VERIFY_ERRORS.  Host-only.
    With min_options the proof's own ProofOptions must be at least as strong (csg_verify_with_options)."""
    pub = np.ascontiguousarray(pub, dtype=np.uint64)
    buf = np.frombuffer(proof, dtype=np.uint8)
    if min_options is not None:
        return lib().csg_verify_with_options(air_id, _p64(pub), pub.size, _p8(buf), buf.size, C.byref(min_options))
    return lib().csg_verify(air_id, _p64(pub), pub.size, _p8(buf), buf.size)


class Context:
    """One proving context = one CUDA device + one stream; owns all device memory (csg_create / csg_destroy)."""

    def __init__(self, device: int = 0):
        self._h = lib().csg_create(device)
        self.device = device
        if not self._h:
            raise CsgError(f"cannot open CUDA device {device}: the CUDA backend is required, there is no CPU fallback")

    def close(self):
        if getattr(self, "_h", None):
            lib().csg_destroy(self._h)
            self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _check(self, rc):
        if rc != 0:
            msg = lib().csg_last_error(self._h)
            raise CsgError(f"{_ERRORS.get(rc, rc)}: {msg.decode() if msg else ''}")

    def _take_proof(self, out, n):
        proof = C.string_at(out, n.value)
        lib().csg_free(out)
        return proof

    # ---- one proof sharded over several GPUs by LDE coset (csg.h, csg_dist_*)
    def dist_init(self, rank: int, world: int, unique_id: bytes):
        """attach to a group of `world` contexts in `world` processes (NCCL); unique_id from dist_unique_id() on rank 0"""
        buf = np.frombuffer(unique_id, dtype=np.uint8).copy()
        if buf.size != 128:
            raise CsgError("an NCCL unique id has 128 bytes")
        self._check(lib().csg_dist_init(self._h, rank, world, _p8(buf)))

    def dist_init_torch(self):
        """attach to the torch.distributed world: rank 0 creates the NCCL id, broadcast through the default process group"""
        import torch.distributed as dist
        rank, world = dist.get_rank(), dist.get_world_size()
        box = [None]
        if rank == 0:
            try:
                box = [dist_unique_id()]
            except CsgError:
                pass                      # every rank learns about it through the broadcast and raises together
        dist.broadcast_object_list(box, src=0)
        if box[0] is None:
            raise CsgError("NCCL is not available on rank 0 (libnccl.so.2 could not be loaded)")
        self.dist_init(rank, world, box[0])

    def dist_info(self):
        r, w = C.c_int(), C.c_int()
        lib().csg_dist_info(self._h, C.byref(r), C.byref(w))
        return r.value, w.value

    # ---- level 1: Prover::prove(trace)
    def prove(self, air_id: int, trace: np.ndarray, pub: np.ndarray, options: ProofOptions, repr: int = REPR_CANONICAL) -> bytes:
        """trace: (width, n) uint64 column-major table (TraceTable's layout) in HOST memory -> StarkProof bytes."""
        trace = np.ascontiguousarray(trace, dtype=np.uint64)
        pub = np.ascontiguousarray(pub, dtype=np.uint64)
        if trace.ndim != 2 or trace.shape[0] != TRACE_WIDTH[air_id]:
            raise CsgError(f"trace must be ({TRACE_WIDTH[air_id]}, n)")
        out, n = _u8p(), C.c_size_t()
        self._check(lib().csg_prove(self._h, air_id, _p64(trace), repr, trace.shape[1], _p64(pub), pub.size, C.byref(options), C.byref(out), C.byref(n)))
        return self._take_proof(out, n)

    def prove_many(self, air_id: int, traces, pubs, options: ProofOptions, repr: int = REPR_CANONICAL) -> list:
        """csg_prove_many: K independent proofs of one AIR, trace length and options in one pass.  traces: a (K, width, n) array or
        a list of K (width, n) arrays in HOST memory; pubs: (K, npub).  Returns the K proofs, each identical to prove() of its trace."""
        traces = [np.ascontiguousarray(t, dtype=np.uint64) for t in traces]
        pubs = np.ascontiguousarray(pubs, dtype=np.uint64)
        if pubs.ndim == 1:
            pubs = pubs.reshape(len(traces), -1)
        if not traces or pubs.ndim != 2 or pubs.shape[0] != len(traces):
            raise CsgError("one row of public inputs per trace expected")
        if any(t.ndim != 2 or t.shape != traces[0].shape for t in traces) or traces[0].shape[0] != TRACE_WIDTH[air_id]:
            raise CsgError(f"every trace must be ({TRACE_WIDTH[air_id]}, n)")
        k = len(traces)
        ptrs = (_u64p * k)(*[_p64(t) for t in traces])
        outs, lens = (_u8p * k)(), (C.c_size_t * k)()
        self._check(lib().csg_prove_many(self._h, air_id, k, ptrs, repr, traces[0].shape[1], _p64(pubs), pubs.shape[1], C.byref(options), outs, lens))
        proofs = [C.string_at(outs[i], lens[i]) for i in range(k)]
        for i in range(k):
            lib().csg_free(outs[i])
        return proofs

    def prove_many_device(self, air_id: int, traces, pubs, options: ProofOptions, repr: int = REPR_CANONICAL) -> list:
        """csg_prove_many_device: prove_many of K traces already in device memory.  traces: a contiguous int64 / uint64 torch CUDA
        tensor (K, width, n) on this context's device, read in place and never written.  Torch's current stream is synchronised
        first, so work queued on it that writes the tensor has finished."""
        import torch
        if not isinstance(traces, torch.Tensor) or traces.device.type != "cuda":
            raise CsgError("traces must be a torch CUDA tensor (K, width, n)")
        if traces.dtype not in (torch.int64, torch.uint64) or not traces.is_contiguous():
            raise CsgError("traces must be a contiguous int64 or uint64 tensor")
        if traces.ndim != 3 or traces.shape[1] != TRACE_WIDTH[air_id]:
            raise CsgError(f"traces must be (K, {TRACE_WIDTH[air_id]}, n)")
        k = traces.shape[0]
        pubs = np.ascontiguousarray(pubs, dtype=np.uint64).reshape(k, -1)
        torch.cuda.current_stream(traces.device).synchronize()
        outs, lens = (_u8p * max(k, 1))(), (C.c_size_t * max(k, 1))()
        self._check(lib().csg_prove_many_device(self._h, air_id, k, traces.data_ptr(), repr, traces.shape[2], _p64(pubs), pubs.shape[1],
                                                C.byref(options), outs, lens))
        proofs = [C.string_at(outs[i], lens[i]) for i in range(k)]
        for i in range(k):
            lib().csg_free(outs[i])
        return proofs

    def _device_traces(self, count: int, width: int, rows: int):
        import torch
        return torch.empty((count, width, rows), dtype=torch.uint64, device=f"cuda:{self.device}")

    def build_many_rescue(self, seeds, chain_length: int):
        """csg_build_traces_many_rescue: K Rescue chains on the device.  seeds: (K, 7) words -> (uint64 CUDA tensor (K, 14, 8 *
        chain_length), pubs (K, 14)), each equal to build_rescue_trace(seeds[k], chain_length)"""
        seeds = np.ascontiguousarray(seeds, dtype=np.uint64).reshape(-1, 7)
        k = seeds.shape[0]
        if chain_length < 1 or chain_length & (chain_length - 1) or chain_length > 8192:
            raise CsgError("invalid argument: chain_length must be a power of two of at most 8192")
        out, pubs = self._device_traces(k, 14, 8 * chain_length), np.zeros((k, 14), dtype=np.uint64)
        self._check(lib().csg_build_traces_many_rescue(self._h, _p64(seeds), k, chain_length, out.data_ptr(), _p64(pubs)))
        return out, pubs

    def build_many_schnorr(self, batch: "SignatureBatch"):
        """csg_build_traces_many_schnorr: one trace per signature on the device -> (uint64 CUDA tensor (K, 56, 512), pubs (K, 38))"""
        out, pubs = self._device_traces(batch.num_sig, 56, 512), np.zeros((batch.num_sig, 38), dtype=np.uint64)
        self._check(lib().csg_build_traces_many_schnorr(self._h, batch._h, out.data_ptr(), _p64(pubs)))
        return out, pubs

    def build_many_merkle_update(self, batch: "TransactionBatch"):
        """csg_build_traces_many_merkle_update: one trace per transfer -> (uint64 CUDA tensor (K, 65, 512), pubs (K, 14))"""
        out, pubs = self._device_traces(batch.num_tx, 65, 512), np.zeros((batch.num_tx, 14), dtype=np.uint64)
        self._check(lib().csg_build_traces_many_merkle_update(self._h, batch._h, out.data_ptr(), _p64(pubs)))
        return out, pubs

    def build_many_transaction(self, batch: "TransactionBatch"):
        """csg_build_traces_many_transaction: one trace per transfer -> (uint64 CUDA tensor (K, 94, 1024), pubs (K, 14))"""
        out, pubs = self._device_traces(batch.num_tx, 94, 1024), np.zeros((batch.num_tx, 14), dtype=np.uint64)
        self._check(lib().csg_build_traces_many_transaction(self._h, batch._h, out.data_ptr(), _p64(pubs)))
        return out, pubs

    def prove_columns(self, air_id: int, columns, pub: np.ndarray, options: ProofOptions, repr: int = REPR_CANONICAL) -> bytes:
        """csg_prove_columns: one separately allocated array per trace column (how a winterfell TraceTable holds them)"""
        columns = [np.ascontiguousarray(c, dtype=np.uint64) for c in columns]
        if len(columns) != TRACE_WIDTH[air_id] or len({c.size for c in columns}) != 1:
            raise CsgError(f"{TRACE_WIDTH[air_id]} columns of equal length expected")
        pub = np.ascontiguousarray(pub, dtype=np.uint64)
        ptrs = (_u64p * len(columns))(*[_p64(c) for c in columns])
        out, n = _u8p(), C.c_size_t()
        self._check(lib().csg_prove_columns(self._h, air_id, ptrs, repr, columns[0].size, _p64(pub), pub.size, C.byref(options), C.byref(out), C.byref(n)))
        return self._take_proof(out, n)

    # ---- level 2 pieces used by benchmarks: trace resident in HBM, proved repeatedly
    def set_air(self, air_id, trace_len, pub, options):
        pub = np.ascontiguousarray(pub, dtype=np.uint64)
        self._check(lib().csg_set_air(self._h, air_id, trace_len, C.byref(options), _p64(pub), pub.size))

    def load_trace(self, trace, repr: int = REPR_CANONICAL):
        trace = np.ascontiguousarray(trace, dtype=np.uint64)
        self._check(lib().csg_load_trace(self._h, _p64(trace), repr))

    def load_trace_ptr(self, host_ptr: int, repr: int = REPR_CANONICAL):
        """same, from a raw host pointer (e.g. a HostBuffer's ptr)"""
        self._check(lib().csg_load_trace(self._h, C.cast(host_ptr, _u64p), repr))

    def prove_trace_ptr(self, host_ptr: int, repr: int = REPR_CANONICAL) -> bytes:
        """proof of the trace at a raw HOST pointer for the AIR already set: pinned memory (HostBuffer) is copied at link speed
        under the extension, pageable memory is staged through the library's own pinned buffers"""
        out, n = _u8p(), C.c_size_t()
        self._check(lib().csg_prove_trace(self._h, C.cast(host_ptr, _u64p), repr, C.byref(out), C.byref(n)))
        return self._take_proof(out, n)

    def prefetch_trace_ptr(self, host_ptr: int, repr: int = REPR_CANONICAL):
        """start the copy of a trace at a raw HOST pointer (keep it alive until the prove_prefetched_ptr that proves it has
        started); returns at once for page-locked memory"""
        self._check(lib().csg_prefetch_trace(self._h, C.cast(host_ptr, _u64p), repr))

    def prove_prefetched_ptr(self, next_host_ptr: Optional[int] = None, repr: int = REPR_CANONICAL) -> bytes:
        """proof of the prefetched trace; the copy of the trace at next_host_ptr (if any) runs under it"""
        out, n = _u8p(), C.c_size_t()
        nxt = C.cast(next_host_ptr, _u64p) if next_host_ptr else C.cast(None, _u64p)
        self._check(lib().csg_prove_prefetched(self._h, nxt, repr, C.byref(out), C.byref(n)))
        return self._take_proof(out, n)

    def reload_resident_trace(self):
        self._check(lib().csg_reload_resident_trace(self._h))

    def prove_loaded(self) -> bytes:
        out, n = _u8p(), C.c_size_t()
        self._check(lib().csg_prove_loaded(self._h, C.byref(out), C.byref(n)))
        return self._take_proof(out, n)

    def build_transaction_trace(self, batch: "TransactionBatch"):
        """TransactionProver::build_trace on the device (witness_gen.cu): the trace never exists in host memory"""
        self._check(lib().csg_build_trace_transaction_device(self._h, batch._h))

    def build_batch(self, seed: int, num_tx: int, tree_depth: int = 15) -> np.ndarray:
        """TransactionMetadata::build_random on the device (batch_gen.cu): returns the public inputs; the packed records stay in HBM"""
        pub = np.zeros(14, dtype=np.uint64)
        self._check(lib().csg_tx_batch_build_device(self._h, seed, num_tx, tree_depth, _p64(pub)))
        return pub

    def build_transaction_trace_resident(self):
        """build_trace on the device from the records left by build_batch"""
        self._check(lib().csg_build_trace_transaction_resident(self._h))

    def download_batch_records(self, num_tx: int) -> np.ndarray:
        out = np.zeros((num_tx, 278), dtype=np.uint64)
        self._check(lib().csg_download_batch_records(self._h, _p64(out), out.size))
        return out

    def build_merkle_update_trace(self, batch: "TransactionBatch"):
        """MerkleProver::build_trace on the device (after set_air(AIR_MERKLE_UPDATE, 512 * num_tx, ...))"""
        self._check(lib().csg_build_trace_merkle_update_device(self._h, batch._h))

    def build_schnorr_trace(self, batch: "SignatureBatch"):
        """SchnorrProver::build_trace on the device (after set_air(AIR_SCHNORR, 512 * num_sig, ...))"""
        self._check(lib().csg_build_trace_schnorr_device(self._h, batch._h))

    def download_trace(self, width: int, trace_len: int) -> np.ndarray:
        out = np.empty((width, trace_len), dtype=np.uint64)
        self._check(lib().csg_download_trace(self._h, _p64(out)))
        return out

    def timer_start(self):
        """CUDA event on the proving stream"""
        self._check(lib().csg_timer_start(self._h))

    def timer_stop(self) -> float:
        """milliseconds of device time since timer_start (CUDA events on the proving stream)"""
        ms = C.c_float()
        self._check(lib().csg_timer_stop(self._h, C.byref(ms)))
        return float(ms.value)

    def timings(self) -> dict:
        t = Timings()
        self._check(lib().csg_get_timings(self._h, C.byref(t)))
        return t.as_dict()

    # ---- kernel-level entry points (parity tests, kernel sweep); canonical values in host arrays
    def lde(self, cols: np.ndarray, blowup: int) -> np.ndarray:
        cols = np.ascontiguousarray(cols, dtype=np.uint64)
        out = np.empty((cols.shape[0], cols.shape[1] * blowup), dtype=np.uint64)
        self._check(lib().csg_k_lde(self._h, _p64(cols), cols.shape[0], cols.shape[1], blowup, _p64(out)))
        return out

    def hash_rows(self, cols: np.ndarray, hash_fn: int = HASH_BLAKE3_256) -> np.ndarray:
        cols = np.ascontiguousarray(cols, dtype=np.uint64)
        out = np.empty((cols.shape[1], 32), dtype=np.uint8)
        self._check(lib().csg_k_hash_rows(self._h, hash_fn, _p64(cols), cols.shape[0], cols.shape[1], _p8(out)))
        return out

    def merkle(self, leaves: np.ndarray, hash_fn: int = HASH_BLAKE3_256) -> np.ndarray:
        leaves = np.ascontiguousarray(leaves, dtype=np.uint8).reshape(-1, 32)
        out = np.empty((2 * leaves.shape[0], 32), dtype=np.uint8)
        self._check(lib().csg_k_merkle(self._h, hash_fn, _p8(leaves), leaves.shape[0], _p8(out)))
        return out

    def fri_fold4(self, evals: np.ndarray, alpha: int) -> np.ndarray:
        evals = np.ascontiguousarray(evals, dtype=np.uint64)
        out = np.empty(evals.size // 4, dtype=np.uint64)
        self._check(lib().csg_k_fri_fold4(self._h, _p64(evals), evals.size, alpha, _p64(out)))
        return out

    def sweep(self, width: int, n: int, blowup: int, hash_fn: int = HASH_BLAKE3_256, iters: int = 3) -> dict:
        ms = (C.c_float * 4)()
        self._check(lib().csg_k_sweep(self._h, width, n, blowup, hash_fn, iters, ms))
        return dict(zip(("lde_ms", "hash_rows_ms", "merkle_ms", "fri_fold_ms"), [float(v) for v in ms]))


class HostBuffer:
    """page-locked host memory from csg_host_alloc, viewed as a (width, n) uint64 array: where a caller builds a trace it is
    going to prove more than once or wants copied at link speed"""

    def __init__(self, width: int, n: int):
        self.nbytes = width * n * 8
        self.ptr = lib().csg_host_alloc(self.nbytes)
        if not self.ptr:
            raise CsgError("csg_host_alloc failed (no CUDA device, or out of page-locked memory)")
        self.array = np.ctypeslib.as_array(C.cast(self.ptr, _u64p), shape=(width, n))

    def close(self):
        if getattr(self, "ptr", None):
            self.array = None
            lib().csg_host_free(self.ptr)
            self.ptr = None

    __del__ = close


def dist_plan(rank: int, world: int, blowup: int, ce_blowup: int, width: int) -> ShardPlan:
    """ownership of rank `rank` in a `world`-way sharded proof (csg_dist_plan); host-only"""
    p = ShardPlan()
    if lib().csg_dist_plan(rank, world, blowup, ce_blowup, width, C.byref(p)):
        raise CsgError("world must be a power of two dividing the blowup factor, rank below it")
    return p


def dist_trace_chunks(rank: int, world: int, blowup: int, ce_blowup: int, width: int, from_host: bool) -> list:
    """column chunks in which that rank copies / extends its column block in stage 1 (csg_dist_trace_chunks); host-only"""
    sizes = (C.c_uint32 * max(1, width))()
    count = C.c_size_t(0)
    if lib().csg_dist_trace_chunks(rank, world, blowup, ce_blowup, width, int(bool(from_host)), sizes, width, C.byref(count)):
        raise CsgError("world must be a power of two dividing the blowup factor, rank below it")
    return [int(sizes[k]) for k in range(count.value)]


def dist_unique_id() -> bytes:
    """ncclGetUniqueId through the library (rank 0 of a sharded proof calls it and hands the bytes to the other ranks)"""
    buf = np.zeros(128, dtype=np.uint8)
    if lib().csg_dist_unique_id(_p8(buf)):
        raise CsgError("NCCL is not available (libnccl.so.2 could not be loaded)")
    return buf.tobytes()


class LocalGroup:
    """`world` contexts of THIS process proving one trace together (csg_dist_init_local): one host thread per context, the
    exchanges are peer copies.  devices: one CUDA device per context; they may repeat (all ranks on one GPU is how the
    tests cover the sharded path on a single-GPU box)."""

    def __init__(self, world: int, devices=None):
        devices = list(devices) if devices is not None else [0] * world
        if len(devices) != world:
            raise CsgError("one device per context")
        self.ctxs = [Context(d) for d in devices]
        arr = (C.c_void_p * world)(*[c._h for c in self.ctxs])
        if lib().csg_dist_init_local(arr, world):
            raise CsgError("cannot form a local group: " + lib().csg_last_error(self.ctxs[0]._h).decode())
        self.world = world

    def run(self, fn):
        """fn(ctx, rank) on every context concurrently (the library calls block until the peers arrive); results by rank"""
        import threading
        out, err = [None] * self.world, [None] * self.world

        def work(r):
            try:
                out[r] = fn(self.ctxs[r], r)
            except BaseException as e:   # noqa: BLE001 - re-raised below
                err[r] = e
        ts = [threading.Thread(target=work, args=(r,)) for r in range(self.world)]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        for e in err:
            if e is not None:
                raise e
        return out

    def prove(self, air_id, trace, pub, options):
        """every context's proof bytes (all equal to the single-GPU proof)"""
        return self.run(lambda ctx, r: ctx.prove(air_id, trace, pub, options))

    def close(self):
        for c in self.ctxs:
            c.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


# ---------------------------------------------------------------------------------------------- witness builders (host)
def build_rescue_trace(seed, chain_length):
    """RescueProver::build_trace (benches/rescue.rs:279-321) -> (trace (14, 8*len), pub = seed[7] result[7])"""
    seed = np.ascontiguousarray(seed, dtype=np.uint64)
    trace, pub = np.zeros((14, 8 * chain_length), dtype=np.uint64), np.zeros(14, dtype=np.uint64)
    if lib().csg_build_trace_rescue(_p64(seed), chain_length, _p64(trace), _p64(pub)):
        raise CsgError("chain length must be a power of two")
    return trace, pub


def build_range_trace(number):
    """RangeProver::build_trace (src/range/prover.rs:36-56)"""
    trace, pub = np.zeros((2, 64), dtype=np.uint64), np.zeros(1, dtype=np.uint64)
    lib().csg_build_trace_range(number, _p64(trace), _p64(pub))
    return trace, pub


def build_merkle_init_trace(s_inputs, r_inputs, delta):
    """PreMerkleProver::build_trace (src/merkle/init/prover.rs:35-53)"""
    s, r = np.ascontiguousarray(s_inputs, dtype=np.uint64), np.ascontiguousarray(r_inputs, dtype=np.uint64)
    trace, pub = np.zeros((58, 16), dtype=np.uint64), np.zeros(29, dtype=np.uint64)
    lib().csg_build_trace_merkle_init(_p64(s), _p64(r), delta, _p64(trace), _p64(pub))
    return trace, pub


class TransactionBatch:
    """Seeded stand-in for TransactionMetadata::build_random (src/lib.rs:235-464): accounts in a Rescue Merkle tree,
    num_tx signed transfers.  The reference draws from OsRng; here everything derives from `seed`."""

    def __init__(self, seed: int, num_tx: int, tree_depth: int = 15):
        self._h = lib().csg_tx_batch_new(seed, num_tx, tree_depth)
        if not self._h:
            raise CsgError("bad transaction batch parameters")
        self.num_tx = num_tx

    def __del__(self):
        if getattr(self, "_h", None):
            lib().csg_tx_batch_free(self._h)
            self._h = None

    def public_inputs(self) -> np.ndarray:
        """initial_root[7] final_root[7]: TransactionProver::get_pub_inputs without building the trace"""
        pub = np.zeros(14, dtype=np.uint64)
        lib().csg_tx_batch_roots(self._h, _p64(pub[:7]), _p64(pub[7:]))
        return pub

    def transaction_trace(self, out: np.ndarray | None = None):
        """TransactionProver::build_trace (src/prover.rs:37-98) -> (trace (94, 1024*num_tx), pub[14])"""
        trace = out if out is not None else np.zeros((94, 1024 * self.num_tx), dtype=np.uint64)
        pub = np.zeros(14, dtype=np.uint64)
        if lib().csg_build_trace_transaction(self._h, _p64(trace), _p64(pub)):
            raise CsgError("number of transactions must be a power of two")
        return trace, pub

    def packed_records(self) -> np.ndarray:
        """the per-transfer records the device witness builder consumes (csg_tx_batch_pack): (num_tx, 278) words"""
        out = np.zeros((self.num_tx, 278), dtype=np.uint64)
        lib().csg_tx_batch_pack(self._h, _p64(out))
        return out

    def merkle_update_trace(self):
        """MerkleProver::build_trace (src/merkle/update/prover.rs:37-80) -> (trace (65, 512*num_tx), pub[14])"""
        trace, pub = np.zeros((65, 512 * self.num_tx), dtype=np.uint64), np.zeros(14, dtype=np.uint64)
        if lib().csg_build_trace_merkle_update(self._h, _p64(trace), _p64(pub)):
            raise CsgError("number of transactions must be a power of two")
        return trace, pub


class SignatureBatch:
    """Seeded stand-in for SchnorrExample::new's random messages and signatures (src/schnorr/mod.rs:79-141)."""

    def __init__(self, seed: int, num_sig: int):
        self._h = lib().csg_sig_batch_new(seed, num_sig)
        if not self._h:
            raise CsgError("bad signature batch parameters")
        self.num_sig = num_sig

    def __del__(self):
        if getattr(self, "_h", None):
            lib().csg_sig_batch_free(self._h)
            self._h = None

    def schnorr_trace(self):
        """SchnorrProver::build_trace (src/schnorr/prover.rs:52-80) -> (trace (56, 512*num_sig), pub[38*num_sig])"""
        trace, pub = np.zeros((56, 512 * self.num_sig), dtype=np.uint64), np.zeros(38 * self.num_sig, dtype=np.uint64)
        if lib().csg_build_trace_schnorr(self._h, _p64(trace), _p64(pub)):
            raise CsgError("number of signatures must be a power of two")
        return trace, pub


# ---------------------------------------------------------------------------------------------- the reference's example façade
def get_example(num_transactions: int, seed: int = 1, device: int = 0) -> "TransactionExample":
    """get_example() of the reference (src/lib.rs:75-89): default options 42 queries, blowup 8, Blake3_256, no extension,
    FRI folding 4, max remainder 256."""
    return TransactionExample(ProofOptions(), num_transactions, seed=seed, device=device)


class TransactionExample:
    """TransactionExample::{new, prove} (src/lib.rs:92-141): a batch of transactions and the proof of their state transition.
    `verify` runs on the host, as winterfell::verify does for the reference (src/lib.rs:144-150)."""

    def __init__(self, options: ProofOptions, num_transactions: int, seed: int = 1, device: int = 0, batch_on_device: bool = False):
        if num_transactions < 1 or num_transactions & (num_transactions - 1):
            raise CsgError("number of transactions must be a power of 2")  # src/lib.rs:100-103
        self.options, self.seed, self.num_transactions = options, seed, num_transactions
        # TransactionMetadata::build_random (src/lib.rs:111): on the host (OpenMP, seconds for large batches) or by kernels at prove() time
        self.batch = None if batch_on_device else TransactionBatch(seed, num_transactions)
        self.ctx = Context(device)
        self.pub_inputs = None

    def verify(self, proof: bytes) -> bool:
        """TransactionExample::verify (src/lib.rs:144-150)"""
        pub = self.pub_inputs if self.batch is None else self.batch.public_inputs()
        return verify(AIR_TRANSACTION, pub, proof, self.options) == 0

    def verify_with_wrong_inputs(self, proof: bytes) -> bool:
        """TransactionExample::verify_with_wrong_inputs (src/lib.rs:152-161): every limb of the final root replaced by its first"""
        pub = np.array(self.pub_inputs if self.batch is None else self.batch.public_inputs())
        pub[7:] = pub[7]
        return verify(AIR_TRANSACTION, pub, proof, self.options) == 0

    def prove(self, witness_on_device: bool = True) -> bytes:
        if self.batch is None:                               # metadata, witness and proof all on the device
            self.pub_inputs = pub = self.ctx.build_batch(self.seed, self.num_transactions)
            self.ctx.set_air(AIR_TRANSACTION, 1024 * self.num_transactions, pub, self.options)
            self.ctx.build_transaction_trace_resident()
            return self.ctx.prove_loaded()
        if not witness_on_device:
            trace, pub = self.batch.transaction_trace()      # prover.build_trace(&tx_metadata)   src/lib.rs:130  (host)
            self.pub_inputs = pub
            return self.ctx.prove(AIR_TRANSACTION, trace, pub, self.options)   # prover.prove(trace)   src/lib.rs:140
        self.pub_inputs = pub = self.batch.public_inputs()
        self.ctx.set_air(AIR_TRANSACTION, 1024 * self.batch.num_tx, pub, self.options)
        self.ctx.build_transaction_trace(self.batch)         # build_trace on the device (witness_gen.cu)
        return self.ctx.prove_loaded()
