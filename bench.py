#!/usr/bin/env python3
"""bench.py — polynomial-commitment throughput (BASELINE.json metric: LDE+Merkle commit cells/s; block-proof-shaped
commit latency in ms).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

A step = one PolynomialBatch::from_values over BASELINE.json configs[2]: 2^20 rows x 135 columns, rate_bits 3,
Poseidon Merkle cap_height 4 (cell = one input element).  Inputs are synthetic (SplitMix64 mod p, SURVEY.md 8d).
  value         whole-job cells/s with inputs resident in HBM, CUDA events on the launching stream, max over ranks
  e2e           same metric through the host-buffer C ABI (b200zkp_commit_from_values at N = 1, b200zkp_sharded_commit with
                host inputs at N > 1): pinned host values -> H2D -> commit -> cap D2H, every step
  roofline      dominant kernel (Poseidon leaf hash): integer-multiply-pipe slots per second against the measured IMAD
                rate (the kernel is integer bound: ~1 Poseidon permutation per cell), with the HBM figures beside it
  parity_check  N = 1: the multithreaded CPU port commits the SAME full-size input once; cap, digest XOR, coefficient XOR
                and LDE XOR must equal the GPU's.  N > 1: a 2^10 x 135 commitment is run through the same partitioned
                path and compared with the oracle on every rank (cap, leaves, digests, coefficients, openings).
  cpu_baseline  that full-size CPU run (or a bounded sample on a slow host), cores stated: a reported baseline
  latency_ms    median device-resident commit latency for the real-circuit shapes of SURVEY.md section 8 (N = 1)
N > 1: ONE commitment partitioned over N GPUs (strong scaling) entirely behind the C ABI (b200zkp_comm_init_rank +
b200zkp_sharded_commit: NCCL is called from the C library); torch.distributed (gloo) only carries the NCCL id, the
barriers and the max over ranks.
--impl reference: times the CPU restatement only (the reference's Rust prover cannot be built here: DESIGN.md), with every
host thread, on a bounded row sample of the same workload sized so that W + K steps end within a few minutes.
B200ZKP_BENCH_CONFIG=5: BASELINE.json configs[4] (2^24 x 256, needs 8 GPUs) with per-rank opening checks.
--dump-outputs DIR: after the timed steps, what the last one returned (cap, and a fixed sample of coefficients, leaves and
digests) as float64 .npy files (dump_outputs), so that two builds can be compared output for output on the same input.
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_LOG, K, RATE_BITS, CAP_HEIGHT = 20, 135, 3, 4
if os.environ.get("B200ZKP_BENCH_CONFIG") == "5":
    N_LOG, K = 24, 256
METRIC = "LDE+Merkle commit cells/s"
UNIT = "cells/s"
P = 0xFFFFFFFF00000001


def workload_name(n_log=N_LOG, k=K):
    return f"synthetic commitment 2^{n_log} rows x {k} columns, rate_bits={RATE_BITS}, Poseidon Merkle cap_height={CAP_HEIGHT}"


def bench_config(n_log, k, world):
    """`config` of the JSON line — the same dict for the b200 and the reference arm (the reference arm's bounded sample is
    described in its cpu_baseline.sample, not here)"""
    return {"workload": workload_name(n_log, k), "n_log": n_log, "k": k, "rate_bits": RATE_BITS, "cap_height": CAP_HEIGHT,
            "cells_per_step": k << n_log,
            "l2": "no flush needed: every step streams 8nk bytes of input and 64nk of LDE (>> 126 MB L2)",
            "partition": "single GPU" if world == 1 else
            f"one commitment over {world} GPUs: column-sharded iNTT (columns dealt in groups of max(8, N)), all-gather of the coefficient shards (fused into the first LDE pass over NVLink peer memory; NCCL point-to-point as fallback), leaf-range LDE+Merkle, all-gather cap"}


def algorithmic_bytes(n_log, k, r=RATE_BITS, h=CAP_HEIGHT):
    n, N = 1 << n_log, 1 << (n_log + r)
    return 8 * n * k + 8 * n * k + 8 * N * k + 64 * (N - (1 << h)) + 32 * (1 << h)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    return 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def kernel_source_key():
    """sha256 over the sources of the leaf-hash kernel: the key profiles/leaf_mix.json was captured under"""
    h = hashlib.sha256()
    for name in ("goldilocks.cuh", "poseidon.cuh", "poseidon_tables.cuh", "merkle_kernels.cuh"):
        with open(os.path.join(ROOT, "intmax_zkp_core_b200", "csrc", name), "rb") as f:
            h.update(f.read())
    return h.hexdigest()[:16]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.gpu)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for (t, r) in self.rows if t0 <= t <= t1 + 0.2 and len(r) >= 8] or [r for (_, r) in self.rows if len(r) >= 8]
        sm, mx, reasons = [], None, set()
        for r in rows:
            try:
                sm.append(float(r[1])); mx = float(r[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_threads_all():
    """every host core for the OpenMP port, whatever OMP_NUM_THREADS says (torchrun exports 1 to its workers)"""
    from oracle import oracle as O
    return O.baseline_set_threads(host_cores())


def cpu_commit_once(values):
    from oracle import oracle as O
    t0 = time.perf_counter()
    res, stages = O.baseline_commit(values, RATE_BITS, CAP_HEIGHT)
    return res, stages, time.perf_counter() - t0


def cpu_rate_estimate():
    """cells/s of the CPU port on this host from a 2^14-row probe (hash-dominated, so the rate carries to larger sizes)"""
    from oracle import oracle as O
    v = O.synthetic_values(K, 1 << 14)
    cpu_commit_once(v)
    _, _, dt = cpu_commit_once(v)
    return (K << 14) / dt


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as O
    O.build()
    cores = cpu_threads_all()
    # bounded sample: the largest row count whose W + K steps fit the budget (default 300 s), never more than the workload
    budget = float(os.environ.get("B200ZKP_REF_BUDGET_S", "300"))
    est = cpu_rate_estimate()
    n_log = N_LOG
    if os.environ.get("B200ZKP_REF_SAMPLE_LOG"):
        n_log = int(os.environ["B200ZKP_REF_SAMPLE_LOG"])
    else:
        while n_log > 14 and (args.steps + args.warmup) * (K << n_log) / est > budget:
            n_log -= 1
    v = O.synthetic_values(K, 1 << n_log)
    for _ in range(args.warmup):
        cpu_commit_once(v)
    ts, stages = [], None
    for _ in range(args.steps):
        _, stages, dt = cpu_commit_once(v)
        ts.append(dt)
    dt = sum(ts) / len(ts)
    rate = (K << n_log) / dt
    sample = (f"each step = one from_values on 2^{n_log} x {K} (" + ("the full workload" if n_log == N_LOG else
              f"1/{1 << (N_LOG - n_log)} of the rows of the workload; cells/s is size-independent to a few percent: hash dominated") +
              f"), all {cores} host threads (OpenMP); C restatement of plonky2 @ f99ed9c's CPU path (oracle/cpu_baseline.c) — the "
              f"Rust prover cannot be built here; stage s ifft/lde/transpose/merkle = " + "/".join(f"{s:.2f}" for s in stages[:4]))
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u64 (Goldilocks field)", "data": "synthetic",
        "config": bench_config(N_LOG, K, args.gpus),
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample, "sample_n_log": n_log},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ------------------------------------------------------------------------------------------------ GPU arm helpers
def bind_to_gpu_numa_node(gpu_index):
    """N > 1: run this rank (and allocate its pinned staging memory) on the CPUs next to its GPU, so that eight uploads do not
    all cross the same socket link (NVML's ideal CPU affinity of the device); harmless where NVML or the call is unavailable"""
    try:
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(gpu_index))
    except Exception:
        pass


def synth_host(torch, np, cols, n, rows_alloc=None):
    """pinned (rows_alloc, n) int64 tensor holding v[c][i] = splitmix64(c*n + i) mod p for the columns `cols`"""
    cols = np.asarray(list(cols), dtype=np.uint64)
    col_begin, col_end = 0, int(cols.size)
    idx = (cols[:, None] * np.uint64(n) + np.arange(n, dtype=np.uint64)[None, :]).reshape(-1)
    with np.errstate(over="ignore"):
        zed = (idx + np.uint64(1)) * np.uint64(0x9E3779B97F4A7C15)
        zed = (zed ^ (zed >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        zed = (zed ^ (zed >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        zed = zed ^ (zed >> np.uint64(31))
    zed = np.where(zed >= np.uint64(P), zed - np.uint64(P), zed).reshape(col_end - col_begin, n)
    host = torch.zeros((max(rows_alloc or 0, col_end - col_begin, 1), n), dtype=torch.int64).pin_memory()
    host[:col_end - col_begin].copy_(torch.from_numpy(zed.view(np.int64)))
    return host


def xor_all(t):
    """XOR of every word of a CUDA int64 tensor: halving on the device while the count is even, numpy for the rest"""
    import numpy as np
    x = t.reshape(-1)
    while x.numel() > 1 and x.numel() % 2 == 0 and x.numel() > 4096:
        h = x.numel() // 2
        x = x[:h] ^ x[h:]
    return int(np.bitwise_xor.reduce(x.cpu().numpy().view(np.uint64)))


def np_xor(a):
    import numpy as np
    return int(np.bitwise_xor.reduce(a.reshape(-1).view(np.uint64)))


def dump_indices(sizes, k, rows=4096):
    """the fixed sample of --dump-outputs: for each name -> length in `sizes`, sorted indices from one seeded generator, first
    and last included; at most `rows` of them, fewer for wide matrices so that a sampled (rows, k) matrix stays under 24 MB"""
    import numpy as np
    rows = max(3, min(rows, (24 << 20) // (16 * k)))
    rng = np.random.default_rng(20)
    return {name: np.unique(np.concatenate([[0, size - 1], rng.integers(0, size, rows - 2)])).astype(np.int64)
            for name, size in sizes.items()}


def dump_outputs(path, outputs, index):
    """--dump-outputs: each uint64 array of `outputs` (numpy or torch int64) as path/<name>.npy in float64, with a last axis of
    2 holding the low and the high 32 bits of every word (a field element does not fit the 53-bit mantissa, its halves do), and
    each array of `index` (the rows a sample holds) as float64.  At 2^20 x 135 the files come to 18 MB."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, a in outputs.items():
        w = np.ascontiguousarray(a.cpu().numpy() if hasattr(a, "cpu") else a).view(np.uint64)
        limbs = np.stack([w & np.uint64(0xFFFFFFFF), w >> np.uint64(32)], axis=-1).astype(np.float64)
        np.save(os.path.join(path, name + ".npy"), limbs)
    for name, a in index.items():
        np.save(os.path.join(path, name + ".npy"), np.asarray(a, dtype=np.float64))


def parity_full_single_gpu(torch, np, host_vals, out, n_log, k):
    """BASELINE.md section 4: the CPU port commits the same input once and every output is compared with the GPU's
    (device-resident result `out` of the timed path).  Falls back to a 2^18-row sample on hosts where the full size would take
    more than ~150 s.  Returns (parity_check dict, cpu_baseline dict)."""
    import intmax_zkp_core_b200 as z
    from intmax_zkp_core_b200 import device as D
    from oracle import oracle as O
    O.build()
    cores = cpu_threads_all()
    est = cpu_rate_estimate()
    full = (k << n_log) / est <= float(os.environ.get("B200ZKP_PARITY_BUDGET_S", "150"))
    cn_log = n_log if full else min(n_log, 18)
    n = 1 << cn_log
    if full:
        v = host_vals.numpy().view(np.uint64)[:k]
        gpu = out
    else:
        hv = synth_host(torch, np, 0, k, n)
        v = hv.numpy().view(np.uint64)[:k]
        ctx = D.torch_context(torch.cuda.current_device())
        gpu = D.commit_device(ctx, hv.cuda(), RATE_BITS, CAP_HEIGHT)
        torch.cuda.synchronize()
    ref, stages, dt = cpu_commit_once(np.ascontiguousarray(v))
    N = n << RATE_BITS
    checks = {
        "cap_equal": bool((gpu.cap.cpu().numpy().view(np.uint64) == ref["cap"]).all()),
        "digests_xor_equal": xor_all(gpu.digests[:2 * (N - (1 << CAP_HEIGHT))]) == np_xor(ref["digests"]),
        "coeffs_xor_equal": xor_all(gpu.coeffs) == np_xor(ref["coeffs"]),
        "lde_xor_equal": xor_all(gpu.lde) == np_xor(ref["leaves"]),
    }
    # a handful of full rows and digests at fixed positions (XORs cannot see a permutation; the cap can, these localise it)
    rows = [0, 1, N // 3, N // 2, N - 1]
    lde_rows = gpu.lde[:, rows].t().cpu().numpy().view(np.uint64)
    checks["sampled_rows_equal"] = bool((lde_rows == ref["leaves"][rows]).all())
    checks["first_digests_equal"] = bool((gpu.digests[:64].cpu().numpy().view(np.uint64) == ref["digests"][:64]).all())
    rate = (k << cn_log) / dt
    parity = {"config": workload_name(cn_log, k) + (" (the benchmarked input)" if full else " (row sample: host too slow for the full size)"),
              "checker": "oracle/cpu_baseline.c (multithreaded CPU port), bit-for-bit", **checks,
              "all_equal": all(checks.values()), "cpu_seconds": round(dt, 2)}
    baseline = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": (f"one from_values on 2^{cn_log} x {k} (" + ("the full workload, same input as the GPU arm" if full else
                           f"1/{1 << (n_log - cn_log)} of the rows") + f"), {dt * 1e3:.0f} ms; C restatement of plonky2's CPU path with "
                           f"OpenMP (oracle/cpu_baseline.c), stage s ifft/lde/transpose/merkle = " + "/".join(f"{s:.2f}" for s in stages[:4]))}
    return parity, baseline


def parity_sharded_small(torch, np, dist, comm, rank, world, dev):
    """N > 1: a 2^10 x 135 commitment through the SAME partitioned C-ABI path, compared with the single-threaded oracle on
    every rank: cap, this rank's leaves, digests, all coefficients, openings of global indices.  Returns True on all ranks
    only if every rank agrees."""
    from intmax_zkp_core_b200 import device as D
    from oracle import oracle as O
    O.build()
    n_log, k = 10, 135
    n = 1 << n_log
    v = O.synthetic_values(k, n, seed=11)
    ref = O.commit(v, RATE_BITS, CAP_HEIGHT)
    lay = D.shard_layout(n_log, k, RATE_BITS, CAP_HEIGHT, rank, world)
    sh = D.ShardedCommitment(comm, n_log, k, RATE_BITS, CAP_HEIGHT)
    mine = np.ascontiguousarray(v[lay["cols"]])
    ok = True
    for host_path in (False, True):
        t = torch.from_numpy(mine.view(np.int64)) if mine.size else None
        if host_path:
            cap_host = torch.zeros((1 << CAP_HEIGHT, 4), dtype=torch.int64).pin_memory()
            sh.run_from_host(t.pin_memory() if t is not None else None, cap_out=cap_host)
            ok &= bool((cap_host.numpy().view(np.uint64) == ref["cap"]).all())
        else:
            sh.run(t.to(dev) if t is not None else None)
        sh.synchronize()
        torch.cuda.synchronize()
        ok &= bool((sh.cap.cpu().numpy().view(np.uint64) == ref["cap"]).all())
        ok &= bool((sh.lde.cpu().numpy().view(np.uint64).T == ref["leaves"][lay["leaf_begin"]:lay["leaf_end"]]).all())
        ok &= bool((sh.coeffs_all.cpu().numpy().view(np.uint64)[:k] == ref["coeffs"]).all())
        sub = 2 * (((n << RATE_BITS) >> CAP_HEIGHT) - 1)
        ok &= bool((sh.digests.cpu().numpy().view(np.uint64)[:(lay["cap_end"] - lay["cap_begin"]) * sub]
                    == ref["digests"][lay["cap_begin"] * sub:lay["cap_end"] * sub]).all())
    N = n << RATE_BITS
    idx = [0, N // world - 1, N // world, N // 2, N - 1]
    rows, sib = sh.rows(idx)
    for j, x in enumerate(idx):
        ok &= bool((rows[j] == ref["leaves"][x]).all()) and bool(O.merkle_verify(rows[j], x, sib[j], ref["cap"]))
    sh.close()
    flag = torch.tensor([1 if ok else 0], dtype=torch.int32)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    return bool(flag.item())


def parity_openings_large(torch, np, sh, rank, world, n_log, k, n_rows=8, n_cols=4):
    """Sizes the oracle cannot commit (config #5): per rank, `n_rows` opened leaves of ITS OWN range are checked against the
    returned coefficients (Horner evaluation by the oracle at the leaf's LDE point, `n_cols` columns each) and their Merkle paths
    against the gathered cap with the oracle's hash."""
    from oracle import oracle as O
    O.build()
    N = 1 << (n_log + RATE_BITS)
    N_loc = N // world
    rng = np.random.default_rng(1234)               # same list on every rank: b200zkp_sharded_rows is collective
    idx = []
    for g in range(world):
        idx += [g * N_loc, (g + 1) * N_loc - 1] + [int(x) for x in g * N_loc + rng.integers(0, N_loc, n_rows - 2)]
    rows, sib = sh.rows(idx)
    cap = sh.cap.cpu().numpy().view(np.uint64)
    cols = sorted(set([0, k - 1] + [int(c) for c in rng.integers(0, k, n_cols)]))[:max(n_cols, 2)]
    coeffs = {c: sh.coeffs_all[c].cpu().numpy().view(np.uint64) for c in cols}
    ok, checked = True, 0
    for j, x in enumerate(idx):
        if x // N_loc != rank:
            continue
        ok &= bool(O.merkle_verify(rows[j], x, sib[j], cap))
        nat = int(format(x, f"0{n_log + RATE_BITS}b")[::-1], 2)          # leaf x = LDE row bitrev(x)
        for c in cols:
            ok &= int(rows[j][c]) == O.eval_at_lde_point(coeffs[c], RATE_BITS, nat)
        checked += 1
    return ok, checked


def latency_block(torch, np, ctx, reps=20):
    """BASELINE.json's second metric ("block proof latency (ms)"): the commit shapes of one plonky2 proof at the row counts
    SURVEY.md section 8 estimates for the reference's circuits, device resident, median of `reps` after 5 warm-ups, plus the
    opening proof on the four oracles of a 2^16-row proof."""
    from intmax_zkp_core_b200 import device as D
    out = {}
    shapes = [(12, 135, False), (14, 135, False), (16, 135, False), (16, 85, False), (16, 20, False), (16, 16, True)]
    for n_log, k, is_coeffs in shapes:
        v = torch.randint(0, 2**62, (k, 1 << n_log), dtype=torch.int64, device="cuda")
        buf = D.DeviceCommitment(n_log, k, RATE_BITS, CAP_HEIGHT, v.device)
        ts = []
        for it in range(reps + 5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            D.commit_device(ctx, v, RATE_BITS, CAP_HEIGHT, out=buf, is_coeffs=is_coeffs)
            e1.record()
            torch.cuda.synchronize()
            if it >= 5:
                ts.append(e0.elapsed_time(e1))
        out[f"2^{n_log}x{k}" + (" from_coeffs" if is_coeffs else "")] = round(statistics.median(ts), 4)
    try:
        import intmax_zkp_core_b200 as z
        import intmax_zkp_core_b200.fri as zf
        n_log = 16
        hctx = z.Context(torch.cuda.current_device())
        rng = np.random.default_rng(n_log)
        ks = (85, 135, 20, 16)
        oracles = [z.PolynomialBatch.from_coeffs(rng.integers(0, 2**63, size=(kk, 1 << n_log), dtype=np.uint64), RATE_BITS, False,
                                                 CAP_HEIGHT, ctx=hctx) for kk in ks]
        params = zf.standard_recursion_fri_config().fri_params(n_log)
        zeta = (int(rng.integers(1, 2**63)), int(rng.integers(1, 2**63)))
        g = pow(1753635133440165772, 1 << (32 - n_log), P)
        gz = (zeta[0] * g % P, zeta[1] * g % P)
        inst = zf.FriInstanceInfo([
            zf.FriBatchInfo(zeta, [zf.FriPolynomialInfo(o, i) for o, kk in enumerate(ks) for i in range(kk)]),
            zf.FriBatchInfo(gz, zf.FriPolynomialInfo.from_range(2, range(2)))])
        ts = []
        for it in range(6):
            ch = zf.Challenger(hctx)
            for o in oracles:
                ch.observe_cap(o._cap)
            hctx.synchronize()
            t0 = time.perf_counter()
            for o in oracles:
                o.eval_ext2(np.array(zeta, np.uint64))
            oracles[2].eval_ext2(np.array(gz, np.uint64))
            zf.prove_openings(inst, oracles, ch, params, True)
            if it >= 1:
                ts.append((time.perf_counter() - t0) * 1e3)
        out["opening_proof_2^16 (85+135+20+16 polys, standard_recursion_config, host wall clock)"] = round(statistics.median(ts), 4)
        del oracles
        hctx.close()
        out.update(prove_chain_latency(torch, np, ctx, n_log))
    except Exception as e:      # the latency block must never take the headline down with it
        out["opening_proof_2^16"] = f"failed: {e!r}"
    return out


def prove_chain_latency(torch, np, ctx, n_log=16, reps=5):
    """The device-resident middle of plonky2's prove() for a 2^n_log-row standard_recursion_config circuit whose gate set is
    Noop / Constant / PublicInput / Arithmetic / Poseidon: wires commitment -> Z + partial products (N1a) -> their commitment ->
    vanishing polynomial on the coset / Z_H (N1b) -> coset_ifft + quotient chunk commitment (N1c).  Only challenges and caps would
    cross PCIe.  Timing is data independent, so the matrices are random (the satisfied-circuit checks live in tests/)."""
    from intmax_zkp_core_b200 import device as D, prover as zp
    n = 1 << n_log
    gates = [(zp.GATE_NOOP, 0, (0, 4)), (zp.GATE_CONSTANT, 0, (0, 4)), (zp.GATE_PUBLIC_INPUT, 0, (0, 4)), (zp.GATE_ARITHMETIC, 0, (0, 4)),
             (zp.GATE_POSEIDON, 1, (4, 5))]
    common = zp.CommonCircuitData(n_log, gates, 2)
    rnd = lambda k: torch.randint(0, 2**62, (k, n), dtype=torch.int64, device="cuda")
    cs, wires = rnd(84), rnd(135)
    com_cs = D.commit_device(ctx, cs, RATE_BITS, CAP_HEIGHT)         # CircuitBuilder::build, not part of prove()
    com_w = D.DeviceCommitment(n_log, 135, RATE_BITS, CAP_HEIGHT, wires.device)
    com_z = D.DeviceCommitment(n_log, 20, RATE_BITS, CAP_HEIGHT, wires.device)
    betas, gammas, alphas = [3, 5], [7, 11], [13, 17]
    k_is = common.k_is
    stages = {"wires_commit": [], "zs_partial_products": [], "zs_commit": [], "quotient_values": [], "quotient_commit": [], "total": []}
    for it in range(reps + 2):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
        ev[0].record()
        D.commit_device(ctx, wires, RATE_BITS, CAP_HEIGHT, out=com_w)
        ev[1].record()
        zpp = zp.zs_partial_products_device(ctx, wires[:80], cs[4:84], k_is, betas, gammas, 8)
        ev[2].record()
        D.commit_device(ctx, zpp, RATE_BITS, CAP_HEIGHT, out=com_z)
        ev[3].record()
        q = zp.compute_quotient_values_device(ctx, common, com_cs.lde, com_w.lde, com_z.lde, betas, gammas, alphas, [1, 2, 3, 4])
        ev[4].record()
        zp.commit_quotient_device(ctx, q, n_log, RATE_BITS, CAP_HEIGHT)
        ev[5].record()
        torch.cuda.synchronize()
        if it >= 2:
            for name, a, b in zip(list(stages)[:5], ev[:5], ev[1:]):
                stages[name].append(a.elapsed_time(b))
            stages["total"].append(ev[0].elapsed_time(ev[5]))
    return {f"prove_middle_2^{n_log} (wires commit -> Z -> commit -> quotient -> commit; device resident)":
            {k: round(statistics.median(v), 4) for k, v in stages.items()}}


def leaf_mix():
    """dynamic instruction mix of one permutation of the shipped leaf-hash kernel (ncu source counters), keyed by the hash of
    the kernel sources it was captured from; `stale` when the sources have changed since"""
    p = os.path.join(ROOT, "profiles", "leaf_mix.json")
    try:
        with open(p) as f:
            m = json.load(f)
    except Exception:
        return None
    m["stale"] = m.get("source_key") != kernel_source_key()
    return m


def ntt_roofline_block(lde_ms, intt_ms, lde_cells, intt_cells, n_log, hbm_peak):
    """The transforms against both roofs.  They are bound by the ALU pipe, not by HBM (a butterfly of two 8-byte elements is ~28
    integer instructions, 20 of them on the ALU pipe; log2(n) / 2 butterflies per element and transform): `alu_pipe_busy` is
    ncu's pipe utilisation of the slowest LDE pass of the tracked capture (the integer roof of a pass is 100 %), the HBM figures
    are algorithmic bytes over the live stage times."""
    m = ntt_mix()
    blk = {"bound": "int (ALU pipe)",
           "lde": {"ms": lde_ms, "algorithmic_gbs": (72 * lde_cells) / (lde_ms * 1e-3) / 1e9 if lde_ms else None,
                   "butterflies_per_s": lde_cells * 8 * n_log / 2 / (lde_ms * 1e-3) if lde_ms else None},
           "intt": {"ms": intt_ms, "algorithmic_gbs": (16 * intt_cells) / (intt_ms * 1e-3) / 1e9 if intt_ms else None},
           "hbm_peak_gbs": hbm_peak}
    if blk["lde"]["algorithmic_gbs"]:
        blk["lde"]["hbm_frac"] = blk["lde"]["algorithmic_gbs"] / hbm_peak
    if m:
        lde = [l for l in m["launches"] if l["ms"] and l["ms"] > 2.0] or m["launches"]
        blk["profile"] = {"file": "profiles/ntt_mix.json", "stale": m["stale"], "source_key": m["source_key"],
                          "lde_passes": [{k: l[k] for k in ("kernel", "ms", "dram_gbs", "alu_pipe_pct", "fmaheavy_pipe_pct", "issue_pct", "registers")} for l in lde],
                          "alu_pipe_busy": max(l["alu_pipe_pct"] for l in lde) / 100.0,
                          "dram_frac_of_measured_peak": max(l["dram_gbs"] for l in lde) / hbm_peak}
    return blk


def ntt_source_key():
    h = hashlib.sha256()
    for name in ("goldilocks.cuh", "ntt_ct_kernels.cuh"):
        with open(os.path.join(ROOT, "intmax_zkp_core_b200", "csrc", name), "rb") as f:
            h.update(f.read())
    return h.hexdigest()[:16]


def ntt_mix():
    """per-pass ncu figures of the transform kernels (profiles/ntt_mix.json, tools/ncu_ntt.py), keyed by the hash of the kernel
    sources they were captured from; `stale` when the sources have changed since"""
    p = os.path.join(ROOT, "profiles", "ntt_mix.json")
    try:
        with open(p) as f:
            m = json.load(f)
    except Exception:
        return None
    m["stale"] = m.get("source_key") != ntt_source_key()
    return m


# ------------------------------------------------------------------------------------------------ GPU arm
def run_b200(args):
    import ctypes as C
    import numpy as np
    import torch
    import torch.distributed as dist
    import intmax_zkp_core_b200 as z
    from intmax_zkp_core_b200 import device as D

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit("launch N > 1 through torch.distributed.run (one rank per GPU)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        bind_to_gpu_numa_node(local_rank)
        dist.init_process_group("gloo")        # bootstrap, barriers and the max over ranks only; the data path is NCCL from C
    n_log = int(os.environ.get("B200ZKP_BENCH_N_LOG", str(N_LOG)))
    k = int(os.environ.get("B200ZKP_BENCH_K", str(K)))
    n, N = 1 << n_log, 1 << (n_log + RATE_BITS)
    cells = n * k

    ctx = D.torch_context(local_rank)          # enqueues on torch's current stream: torch.cuda.Event sees our kernels
    lay = D.shard_layout(n_log, k, RATE_BITS, CAP_HEIGHT, rank, world)
    parity = None
    comm = None
    if world > 1:
        comm = D.Comm.from_torch_distributed(ctx)
        if os.environ.get("B200ZKP_EXCHANGE_GROUP"):
            comm.set_exchange_group(int(os.environ["B200ZKP_EXCHANGE_GROUP"]))
        if not os.environ.get("B200ZKP_SKIP_PARITY"):
            parity = {"config": "2^10 x 135 through the same partitioned C-ABI path, every rank vs oracle/oracle.c "
                                "(cap, leaves, digests, coefficients, openings; device and host inputs)",
                      "parity_ok": parity_sharded_small(torch, np, dist, comm, rank, world, dev)}

    # synthetic input: v[c][i] = splitmix64(c*n + i) mod p; each rank generates only its column shard
    host_vals = synth_host(torch, np, lay["cols"], n, lay["kp"] if world > 1 else k)
    dev_vals = host_vals.to(dev)

    if world == 1:
        out = D.DeviceCommitment(n_log, k, RATE_BITS, CAP_HEIGHT, dev)

        def step():
            D.commit_device(ctx, dev_vals, RATE_BITS, CAP_HEIGHT, out=out)
    else:
        sh = D.ShardedCommitment(comm, n_log, k, RATE_BITS, CAP_HEIGHT)

        def step():
            sh.run(dev_vals)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    sync_all()

    # ---- timed region (device-resident)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    ctx.stage_ms()                      # clear spans
    ctx.set_timing(True)
    launches0 = ctx.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    t_wall0 = time.time()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    sync_all()
    t_wall1 = time.time()
    ms_total = e0.elapsed_time(e1)
    launches = ctx.launch_count - launches0
    stages = ctx.stage_ms()
    ctx.set_timing(False)
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    t = torch.tensor([ms_total], dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    value = cells / (ms_step * 1e-3)

    if args.dump_outputs:
        if world == 1:
            idx = dump_indices({"coeffs_index": n, "leaves_index": N, "digests_index": out.digests.shape[0]}, k)
            at = {name: torch.as_tensor(i, device=dev) for name, i in idx.items()}
            dump_outputs(args.dump_outputs, {"cap": out.cap, "coeffs": out.coeffs[:, at["coeffs_index"]].t(),
                                             "leaves": out.lde[:, at["leaves_index"]].t(),
                                             "digests": out.digests[at["digests_index"]]}, idx)
        else:
            # every rank holds its own leaf range and subtree: the sampled leaves are opened through the collective
            # b200zkp_sharded_rows, and the digests, split over the ranks, are not written
            idx = dump_indices({"coeffs_index": n, "leaves_index": N}, k)
            leaves, _ = sh.rows(idx["leaves_index"])
            if rank == 0:
                cols = sh.coeffs_all[:k][:, torch.as_tensor(idx["coeffs_index"], device=dev)].t()
                dump_outputs(args.dump_outputs, {"cap": sh.cap, "coeffs": cols, "leaves": leaves}, idx)

    # ---- end to end through the host-buffer API (pinned host input, H2D + commit + cap D2H per step)
    cap_host = torch.empty((1 << CAP_HEIGHT, 4), dtype=torch.int64).pin_memory()
    if world == 1:
        hctx = z.Context(local_rank)
        lib = hctx._lib

        def e2e_step():
            h = C.c_void_p()
            hctx.check(lib.b200zkp_commit_from_values(hctx._h, C.c_void_p(host_vals.data_ptr()), n_log, k, RATE_BITS,
                                                      CAP_HEIGHT, None, C.byref(h)))
            hctx.check(lib.b200zkp_batch_cap(h, C.c_void_p(cap_host.data_ptr())))
            lib.b200zkp_batch_free(h)
        h2d_bytes = 8 * n * k
    else:
        def e2e_step():
            sh.run_from_host(host_vals, cap_out=cap_host)
        h2d_bytes = 8 * n * lay["n_cols"]
    for _ in range(max(1, min(args.warmup, 2))):
        e2e_step()
    sync_all()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    sync_all()
    dt = torch.tensor([(time.perf_counter() - t0) / args.steps], dtype=torch.float64)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    e2e_value = cells / float(dt.item())
    cap_dev = (out.cap if world == 1 else sh.cap).cpu()
    assert bool((cap_dev == cap_host).all()), "device-resident and end-to-end paths disagree on the cap"
    # the same synthetic input must give the same cap for every N (compare across runs)
    cap_checksum = "%016x" % (int(np.bitwise_xor.reduce(cap_dev.numpy().view(np.uint64).reshape(-1))))

    # ---- strict drop-in: + D2H of coefficients, row-major leaves and digests, overlapped with the hashing (N = 1 only)
    e2e_strict = None
    if world == 1 and not os.environ.get("B200ZKP_SKIP_STRICT"):
        row = k
        outs = [torch.empty(sz, dtype=torch.int64).pin_memory() for sz in (k * n, N * row, 8 * (N - (1 << CAP_HEIGHT)))]

        def strict_step():
            hctx.check(lib.b200zkp_commit_copy_back(hctx._h, C.c_void_p(host_vals.data_ptr()), 0, n_log, k, RATE_BITS, CAP_HEIGHT, None,
                                                    C.c_void_p(outs[0].data_ptr()), C.c_void_p(outs[1].data_ptr()),
                                                    C.c_void_p(outs[2].data_ptr()), C.c_void_p(cap_host.data_ptr()), None))
        strict_step()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(max(1, min(args.steps, 3))):
            strict_step()
        torch.cuda.synchronize()
        dt_s = (time.perf_counter() - t0) / max(1, min(args.steps, 3))
        e2e_strict = {"value": cells / dt_s, "unit": UNIT, "ms_per_step": dt_s * 1e3, "h2d_bytes_per_step": 8 * n * k,
                      "d2h_bytes_per_step": sum(o.numel() for o in outs) * 8 + (32 << CAP_HEIGHT),
                      "api": "b200zkp_commit_copy_back: coefficients + row-major leaves + digests + cap to pinned host memory"}
        del outs
    if world == 1:
        hctx.trim()          # hand the cached 10.7 GB of the host-API batches back before the checks below allocate

    # ---- large-size parity properties for shapes the oracle cannot commit (config #5)
    if world > 1 and n_log > 20 and not os.environ.get("B200ZKP_SKIP_PARITY"):
        ok5, checked = parity_openings_large(torch, np, sh, rank, world, n_log, k)
        flag = torch.tensor([1 if ok5 else 0, checked], dtype=torch.int32)
        dist.all_reduce(flag[:1], op=dist.ReduceOp.MIN)
        dist.all_reduce(flag[1:], op=dist.ReduceOp.SUM)
        parity["openings_check"] = {"what": "per rank: opened leaves of its own range — Horner evaluation of the returned coefficients "
                                            "at the leaf's LDE point (oracle) and Merkle path to the gathered cap (oracle hash)",
                                    "rows_checked": int(flag[1].item()), "all_ok": bool(flag[0].item())}

    if rank == 0:
        peak, peak_src = measured_peaks()
        N_local = lay["N_local"]
        leaf_ms, leaf_cnt = stages["leaf_hash"]
        leaf_ms_avg = leaf_ms / max(leaf_cnt, 1)
        leaf_bytes = 8 * N_local * k + 32 * N_local          # SURVEY.md 8d: 64 B/cell read + 32*2^r/k written
        achieved = leaf_bytes / (leaf_ms_avg * 1e-3) / 1e9 if leaf_ms_avg else 0.0
        perms = N * ((k + 7) // 8) + (N - (1 << CAP_HEIGHT))
        lde_ms = stages["lde"][0] / args.steps
        intt_ms = stages["intt"][0] / args.steps
        lde_cells = (cells // world) if world > 1 else cells
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u64 (Goldilocks field, 32-bit IMAD/IADD3 limbs)", "data": "synthetic",
            "config": bench_config(n_log, k, world),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 32 << CAP_HEIGHT,
                    "api": "b200zkp_commit_from_values + b200zkp_batch_cap (pinned host buffers)" if world == 1 else
                           "b200zkp_sharded_commit (host inputs): pinned column shard H2D in column-group chunks, pipelined with the inverse transforms, the gather, the coset transforms and the leaf sponges (resumable) + tree + cap D2H per rank"},
            "gpu_launches": int(launches),
            "roofline": {"kernel": "merkle::leaf_hash_kernel", "bound": "int", "hbm": {
                             "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": leaf_bytes},
                         "avg_launch_ms": leaf_ms_avg, "traffic": None,
                         "note": "integer-pipe bound by construction (~1 Poseidon permutation per cell, no tensor-core shape): "
                                 "achieved/peak/frac are integer-multiply-pipe slots; the HBM reading of the same launch is under 'hbm'"},
            "commit_hbm": {"bytes_per_step": algorithmic_bytes(n_log, k),
                           "achieved_gbs": algorithmic_bytes(n_log, k) / (ms_step * 1e-3) / 1e9,
                           "frac_of_peak": algorithmic_bytes(n_log, k) / (ms_step * 1e-3) / 1e9 / (peak * world)},
            "ntt_hbm": {"lde_algorithmic_gbs": (72 * lde_cells) / (lde_ms * 1e-3) / 1e9 if lde_ms else None,
                        "intt_algorithmic_gbs": (16 * (n * lay["n_cols"])) / (intt_ms * 1e-3) / 1e9 if intt_ms else None,
                        "peak": peak, "note": "SURVEY.md 8d stage bytes: LDE 72 B/cell, iNTT 16 B/cell (rank 0's share at N > 1)"},
            "ntt_roofline": ntt_roofline_block(lde_ms, intt_ms, lde_cells, n * lay["n_cols"], n_log, peak),
            "stages_ms_per_step": {s: v[0] / args.steps for s, v in stages.items()},
            "poseidon_perms_per_s": perms / (ms_step * 1e-3),
            "lde_cells_per_s": value * (1 << RATE_BITS),          # SURVEY.md 8d: the same throughput counted in LDE cells
            "cap_checksum": cap_checksum,
        }
        if world > 1:
            line["exchange"] = ("peer memory (coefficient tiles pulled over NVLink inside ntc::ct_pull_kernel, flags in peer memory)"
                                if comm.peer_exchange else "NCCL point-to-point groups")
        if e2e_strict:
            line["e2e_strict"] = e2e_strict
        if parity is not None:
            line["parity_check"] = parity
        mix = leaf_mix()
        if world == 1:
            gips = {}
            for kind, name in ((0, "imad_wide"), (1, "iadd3"), (2, "imad"), (3, "imad_wide+lop3"), (4, "lop3"), (5, "imad_hi"), (6, "imad+lop3"), (7, "iadd3_carry_pair"), (8, "imad_wide_noacc")):
                g = C.c_double()
                ctx.check(ctx._lib.b200zkp_int_pipe_bench(ctx._h, kind, 2000, C.byref(g)))
                gips[name] = g.value
            line["int_pipe"] = {"unit": "giga thread-instructions/s (dependent chains, all SMs)", **gips}
            if os.environ.get("B200ZKP_WRITE_PEAKS"):
                with open(os.path.join(ROOT, "MEASURED_INT_PEAK.json"), "w") as f:
                    json.dump({"imad_gips": gips["imad"], "imad_wide_gips": gips["imad_wide"], "iadd3_gips": gips["iadd3"], "lop3_gips": gips["lop3"],
                               "how": "b200zkp_int_pipe_bench: dependent chains of one instruction kind on every SM, 2000 rounds; "
                                      "giga thread-instructions/s", "sm_mhz": clocks.get("sm_mhz") if clocks else None,
                               "when": time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime())}, f, indent=1)
        # second roof of SURVEY.md 8d: the leaf hash against the issue rate of the integer-multiply (fmaheavy) pipe, the
        # busier of the two integer pipes.  Instruction mix per permutation: profiles/leaf_mix.json (ncu source counters),
        # keyed by the hash of the kernel sources; IMAD.WIDE = 2 slots (issues at half the IMAD rate)
        int_peak = None
        if world == 1:
            int_peak, int_src = gips["imad"] * 1e9, "measured in this run (b200zkp_int_pipe_bench kind 2)"
        else:
            try:
                with open(os.path.join(ROOT, "MEASURED_INT_PEAK.json")) as f:
                    int_peak, int_src = json.load(f)["imad_gips"] * 1e9, "MEASURED_INT_PEAK.json (of measured)"
            except Exception:
                int_peak = None
        if mix and int_peak and leaf_ms_avg:
            leaf_perms = N_local * ((k + 7) // 8)
            slots = 2 * mix["imad_wide"] + mix["fma_single_slot"]
            rate = leaf_perms * slots / (leaf_ms_avg * 1e-3)
            line["roofline"].update({
                "achieved": rate, "peak": int_peak, "unit": "IMAD-slot thread-instr/s (IMAD.WIDE = 2 slots)", "frac": rate / int_peak,
                "peak_source": int_src, "slots_per_permutation": slots, "permutations_per_launch": leaf_perms,
                "alu_frac": leaf_perms * mix["alu"] / (leaf_ms_avg * 1e-3) / (gips["lop3"] * 1e9) if world == 1 else None,
                "issue_frac": leaf_perms * mix["instructions"] / (leaf_ms_avg * 1e-3) / (2 * int_peak),
                "instruction_mix": mix})
            if not mix["stale"] and mix.get("traffic_bytes") and n_log == 20 and k == 135 and world == 1:
                line["roofline"]["traffic"] = mix["traffic_bytes"]
        if world == 1 and not os.environ.get("B200ZKP_SKIP_CPU"):
            par, base = parity_full_single_gpu(torch, np, host_vals, out, n_log, k)
            line["parity_check"] = par
            line["cpu_baseline"] = base
        if world == 1 and not os.environ.get("B200ZKP_SKIP_LATENCY"):
            line["latency_ms"] = latency_block(torch, np, ctx)
        print(json.dumps(line))
    if world > 1:
        sh.close()
        comm.close()
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step (cap, sampled coefficients, leaves, digests) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl b200)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
