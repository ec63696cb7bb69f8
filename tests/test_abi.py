"""The C-ABI library builds for sm_100a, loads, exports exactly what include/b200zkp.h declares, and refuses to
compute without a CUDA device (no CPU fallback).  No compute calls here."""
import ctypes as C
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    """every entry point declared by include/*.h (the drop-in surface b200zkp.h and the test probes b200zkp_test.h)"""
    text = ""
    for name in sorted(os.listdir(os.path.join(ROOT, "include"))):
        if name.endswith(".h"):
            with open(os.path.join(ROOT, "include", name)) as f:
                text += f.read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(b200zkp_[a-z0-9_]+)\s*\(", text)))


def test_library_builds_and_exports_declared_abi():
    import intmax_zkp_core_b200 as z
    from intmax_zkp_core_b200 import _lib
    lib = z.lib()
    decl = declared_symbols()
    assert len(decl) >= 35
    for name in decl:
        assert hasattr(lib, name), f"{name} declared in include/b200zkp.h but not exported"
    assert sorted(_lib.EXPORTED_SYMBOLS) == decl            # the ctypes table binds every declared entry point
    assert b"sm_100a" in lib.b200zkp_version()
    # probes and micro-benchmarks are not part of the drop-in surface
    with open(os.path.join(ROOT, "include", "b200zkp.h")) as f:
        assert "b200zkp_field_op" not in f.read()


def test_library_is_sm_100a_only():
    from intmax_zkp_core_b200 import _lib
    _lib.lib()
    out = subprocess.run(["cuobjdump", "-lelf", _lib.LIB_PATH], capture_output=True, text=True)
    if out.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    archs = set(re.findall(r"sm_\d+a?", out.stdout))
    assert archs == {"sm_100a"}, archs


def test_no_cpu_fallback_without_device():
    import intmax_zkp_core_b200 as z
    lib = z.lib()
    if lib.b200zkp_device_count() > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(z.B200ZkpError):
        z.Context(0)
    h = C.c_void_p()
    assert lib.b200zkp_ctx_create(0, None, C.byref(h)) < 0 and not h.value
    with pytest.raises(z.B200ZkpError):
        z.PoseidonHash.two_to_one([0, 0, 0, 0], [0, 0, 0, 0])


def test_product_never_imports_oracle():
    """oracle/ is test infrastructure: nothing under the package, include/ or host/ may reference it."""
    bad = []
    for base in ("intmax_zkp_core_b200", "include", "host"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, base)):
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".h", ".hpp", ".cpp")):
                    with open(os.path.join(dirpath, f), errors="ignore") as fh:
                        for i, line in enumerate(fh, 1):
                            if (re.search(r"^\s*(from|import)\s+oracle\b", line) or re.search(r'#include\s+"[^"]*oracle/', line)
                                    or re.search(r"liboracle|libcpubaseline|\borc_\w+\(|\bcpub_\w+\(", line)):
                                bad.append(f"{os.path.join(dirpath, f)}:{i}")
    assert not bad, bad


def test_host_mirror_argument_errors():
    """plonky2's asserts surface as ValueError before anything touches the device."""
    import numpy as np
    import intmax_zkp_core_b200 as z
    with pytest.raises(ValueError):
        z.log2_strict(6)
    with pytest.raises(ValueError):
        z.MerkleTree.new(np.zeros((6, 5), np.uint64), 1, ctx=object())
    with pytest.raises(ValueError):
        z.MerkleTree.new(np.zeros((8, 5), np.uint64), 4, ctx=object())
    with pytest.raises(ValueError):
        z.PolynomialBatch.from_values(np.zeros((3, 8), np.uint64), 1, False, 5, ctx=object())
    assert z.HashOut.from_hex(z.HashOut([1, 2, 3, 2**63]).to_hex()) == z.HashOut([1, 2, 3, 2**63])


def test_bench_profile_blocks_are_keyed_to_the_kernel_sources():
    """bench.py's roofline blocks read ncu figures from profiles/*.json; each carries the hash of the kernel sources it was
    captured from and is reported `stale` when they changed.  The committed profiles must load, and the staleness test must
    react to a different key."""
    import json
    import sys
    sys.path.insert(0, ROOT)
    import bench
    for fn, key in ((bench.leaf_mix, bench.kernel_source_key), (bench.ntt_mix, bench.ntt_source_key)):
        m = fn()
        assert m is not None and isinstance(m["stale"], bool) and len(key()) == 16
        assert m["stale"] == (m["source_key"] != key())
    blk = bench.ntt_roofline_block(18.8, 2.54, 135 << 20, 135 << 20, 20, 6550.1)
    assert blk["bound"].startswith("int") and 0.05 < blk["lde"]["hbm_frac"] < 0.2
    assert abs(blk["lde"]["butterflies_per_s"] - (135 << 20) * 8 * 10 / 18.8e-3) < 1e3
    json.dumps(blk)
    if "profile" in blk:
        assert 0.5 < blk["profile"]["alu_pipe_busy"] <= 1.0 and len(blk["profile"]["lde_passes"]) == 3


def test_bench_dump_outputs_are_exact_and_bounded(tmp_path):
    """bench.py --dump-outputs: the sample is the same on every call, the float64 limbs give back every uint64 word, and the
    files of the benchmarked shape stay under 64 MB."""
    import sys
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    n_log, k = 20, 135
    N = 1 << (n_log + bench.RATE_BITS)
    sizes = {"coeffs_index": 1 << n_log, "leaves_index": N, "digests_index": 2 * (N - (1 << bench.CAP_HEIGHT))}
    idx = bench.dump_indices(sizes, k)
    again = bench.dump_indices(sizes, k)
    for name, size in sizes.items():
        i = idx[name]
        assert (i == again[name]).all() and i[0] == 0 and i[-1] == size - 1 and (np.diff(i) > 0).all()
    rows = len(idx["coeffs_index"]) + len(idx["leaves_index"])
    total = 16 * (rows * k + 4 * len(idx["digests_index"]) + (4 << bench.CAP_HEIGHT)) + 8 * sum(len(i) for i in idx.values())
    assert total < 64 << 20
    w = np.array([[0, 1, bench.P - 1], [2**32 - 1, 2**32, 2**64 - 1]], dtype=np.uint64)
    bench.dump_outputs(str(tmp_path), {"w": w}, {"w_index": np.array([0, 7])})
    got = np.load(tmp_path / "w.npy")
    assert got.dtype == np.float64 and got.shape == (2, 3, 2)
    assert (got[..., 0].astype(np.uint64) + (got[..., 1].astype(np.uint64) << np.uint64(32)) == w).all()
    assert (np.load(tmp_path / "w_index.npy") == [0, 7]).all()
