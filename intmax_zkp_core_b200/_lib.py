"""Loader for the C-ABI shared library (include/b200zkp.h).

The library is built in-tree by `build()` (nvcc, sm_100a only) and loaded with ctypes.  There is no CPU
fallback: if the library is missing and cannot be built, or no CUDA device is present, every compute call
raises — the product path never routes through oracle/.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
# B200ZKP_LIB selects an alternative build of the same library (kernel tuning experiments only)
LIB_PATH = os.environ.get("B200ZKP_LIB") or os.path.join(_HERE, "libb200zkp.so")
SRC = os.path.join(_HERE, "csrc", "b200zkp.cu")
HEADER = os.path.join(os.path.dirname(_HERE), "include", "b200zkp.h")
TEST_HEADER = os.path.join(os.path.dirname(_HERE), "include", "b200zkp_test.h")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-shared", "-Xcompiler", "-fPIC", "-ldl",
]

u64p = C.POINTER(C.c_uint64)
u32p = C.POINTER(C.c_uint32)


class B200ZkpError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"b200zkp status {code}: {msg}")
        self.code = code


def _sources():
    d = os.path.join(_HERE, "csrc")
    return [os.path.join(d, f) for f in sorted(os.listdir(d))] + [HEADER, TEST_HEADER]


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(s) > t for s in _sources())


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/b200zkp.cu for sm_100a into libb200zkp.so (in-tree, so it travels with the repo).

    Safe under concurrent callers (the ranks of a torchrun launch, pytest-xdist workers): one process holds the lock and
    compiles into a temporary file that is renamed into place, the others wait and re-check."""
    if not force and not needs_build():
        return LIB_PATH
    import fcntl
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: cannot build libb200zkp.so (there is no CPU fallback)")
    with open(LIB_PATH + ".lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not needs_build():      # another process built it while we waited
                return LIB_PATH
            tmp = f"{LIB_PATH}.{os.getpid()}.tmp"
            cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", tmp, SRC]
            try:
                subprocess.check_call(cmd)
                os.replace(tmp, LIB_PATH)
            finally:
                if os.path.exists(tmp):
                    os.remove(tmp)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return LIB_PATH


_lib = None

_SIGS = {
    "b200zkp_version": (C.c_char_p, []),
    "b200zkp_device_count": (C.c_int, []),
    "b200zkp_ctx_create": (C.c_int, [C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]),
    "b200zkp_ctx_destroy": (None, [C.c_void_p]),
    "b200zkp_last_error": (C.c_char_p, [C.c_void_p]),
    "b200zkp_ctx_synchronize": (C.c_int, [C.c_void_p]),
    "b200zkp_ctx_launch_count": (C.c_uint64, [C.c_void_p]),
    "b200zkp_ctx_trim": (C.c_int, [C.c_void_p]),
    "b200zkp_ctx_set_pool_limit": (C.c_int, [C.c_void_p, C.c_uint64]),
    "b200zkp_ctx_set_timing": (C.c_int, [C.c_void_p, C.c_int]),
    "b200zkp_ctx_stage_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), u32p]),
    "b200zkp_host_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p)]),
    "b200zkp_host_free": (None, [C.c_void_p]),
    "b200zkp_commit_from_values": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.POINTER(C.c_void_p)]),
    "b200zkp_commit_from_coeffs": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.POINTER(C.c_void_p)]),
    "b200zkp_commit_copy_back": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    "b200zkp_batch_from_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p,
                                            C.POINTER(C.c_void_p)]),
    "b200zkp_batch_free": (None, [C.c_void_p]),
    "b200zkp_batch_shape": (C.c_int, [C.c_void_p, u32p]),
    "b200zkp_batch_cap": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200zkp_batch_coeffs": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200zkp_batch_leaves": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200zkp_batch_digests": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200zkp_batch_rows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]),
    "b200zkp_batch_lde_values": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p]),
    "b200zkp_batch_device_ptrs": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]),
    "b200zkp_batch_eval_ext2": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200zkp_dev_eval_ext2": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]),
    "b200zkp_dev_gather": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p,
                                     C.c_uint64, C.c_void_p, C.c_void_p]),
    "b200zkp_batch_openings": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_void_p]),
    "b200zkp_fri_begin": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p)]),
    "b200zkp_fri_begin_from_coeffs": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(C.c_void_p)]),
    "b200zkp_fri_free": (None, [C.c_void_p]),
    "b200zkp_fri_shape": (C.c_int, [C.c_void_p, u32p]),
    "b200zkp_fri_coeffs": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200zkp_fri_commit_layer": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]),
    "b200zkp_fri_fold": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200zkp_fri_final_poly": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200zkp_fri_query": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]),
    "b200zkp_pow_grind": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint64, u64p]),
    "b200zkp_merkle_new": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.POINTER(C.c_void_p)]),
    "b200zkp_tree_free": (None, [C.c_void_p]),
    "b200zkp_tree_cap": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200zkp_tree_digests": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200zkp_tree_prove": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "b200zkp_poseidon_permute": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "b200zkp_duplex_chain": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p]),
    "b200zkp_hash_no_pad": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p]),
    "b200zkp_hash_or_noop": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p]),
    "b200zkp_two_to_one": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "b200zkp_ntt": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32]),
    "b200zkp_intt": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32]),
    "b200zkp_coset_intt": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint64]),
    "b200zkp_dev_coset_intt": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint64]),
    "b200zkp_coset_lde": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]),
    "b200zkp_dev_intt": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.c_uint32]),
    "b200zkp_dev_lde": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]),
    "b200zkp_dev_salt": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]),
    "b200zkp_dev_random_field": (C.c_int, [C.c_void_p, C.c_char_p, C.c_char_p, C.c_uint64, C.c_uint64, C.c_void_p]),
    "b200zkp_dev_merkle": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p]),
    "b200zkp_dev_lde_merkle": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]),
    "b200zkp_dev_commit": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200zkp_dev_transpose_to_rows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint64, C.c_uint64, C.c_void_p]),
    "b200zkp_partial_products_and_zs": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p,
                                                C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]),
    "b200zkp_dev_partial_products_and_zs": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32,
                                                    C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint64]),
    "b200zkp_dev_quotient_values": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64,
                                            C.c_void_p, C.c_uint64]),
    "b200zkp_comm_unique_id": (C.c_int, [C.POINTER(C.c_uint8)]),
    "b200zkp_comm_init_rank": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint8), C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "b200zkp_comm_init_all": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.POINTER(C.c_void_p)]),
    "b200zkp_comm_destroy": (None, [C.c_void_p]),
    "b200zkp_comm_last_error": (C.c_char_p, [C.c_void_p]),
    "b200zkp_comm_shape": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32)]),
    "b200zkp_comm_set_exchange_group": (C.c_int, [C.c_void_p, C.c_uint32]),
    "b200zkp_comm_set_peer_exchange": (C.c_int, [C.c_void_p, C.c_int]),
    "b200zkp_comm_peer_exchange": (C.c_int, [C.c_void_p]),
    "b200zkp_sharded_create": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(C.c_void_p)]),
    "b200zkp_sharded_free": (None, [C.c_void_p]),
    "b200zkp_sharded_layout": (C.c_int, [C.c_void_p, C.c_int, u64p]),
    "b200zkp_sharded_columns": (C.c_int, [C.c_void_p, C.c_int, u32p, C.c_uint32, u32p]),
    "b200zkp_sharded_commit": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_void_p]),
    "b200zkp_sharded_commit_from_values": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p,
                                                   C.POINTER(C.c_void_p)]),
    "b200zkp_sharded_synchronize": (C.c_int, [C.c_void_p]),
    "b200zkp_sharded_device_ptrs": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                            C.POINTER(C.c_void_p)]),
    "b200zkp_sharded_rows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]),
    "b200zkp_field_op": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "b200zkp_int_pipe_bench": (C.c_int, [C.c_void_p, C.c_int, C.c_uint32, C.POINTER(C.c_double)]),
    "b200zkp_ctx_buffer_bytes": (C.c_int, [C.c_void_p, u64p, u64p]),
}

EXPORTED_SYMBOLS = tuple(_SIGS)


def lib() -> C.CDLL:
    """Load (building first if the sources are newer) the shared library; raises if that is impossible."""
    global _lib
    if _lib is None:
        if needs_build():
            build()
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(l, name)      # AttributeError here = the library does not export the declared ABI
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib
