#!/usr/bin/env python3
"""Timing of the whole plonky2 prove() on the device (prover.prove) for the gate set of a standard_recursion_config verifier
circuit: the 14 kinds of tests/interpolation_ref.recursion_circuit, with LowDegreeInterpolation(4), 2 challenges,
quotient_degree_factor 8, standard_recursion_config's FRI (rate 3, cap 4, arity 16, 16 PoW bits, 28 queries).

The work does not depend on the values, so the witness and the constants / sigmas are random (with quotient_degree_factor =
2^quotient_degree_bits = 8 there is no divisibility check, so a random witness still gives a complete proof).  Constants and
sigmas are committed once (circuit_data), outside the timed window.  Per size: --warmup proofs, then the median and min / max
of --reps proofs timed with the host clock around prove() (which ends in device-to-host copies); then, in separate proofs, the
per-stage split from CUDA events on the ctx stream (prover.PROVE_STAGES) and the kernel launches per proof.  The card's name
and power limit are read in the same run; one JSON line per size is printed and appended to --out.
--zk: the same circuit proved with zero_knowledge = true and = false in the same run, alternating proof by proof (a fresh salt
key from the OS for every zk proof, as prove() draws it), timed and split the same way; before the sizes, one line with the time
of b200zkp_dev_random_field alone for the 4 x 2^19 salt elements of one 2^16-row commitment (CUDA events, median of --reps
launches of 20 calls each).
GPU only.   python tools/prove_timing.py [--sizes 12 14 16] [--zk] [--out profiles/r4_prove_timing.jsonl]"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch

from intmax_zkp_core_b200 import device as D, fri as zf, prover as zp
from quotient_timing import card, gate_sets


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[12, 14, 16])
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--zk", action="store_true", help="also prove with zero_knowledge, alternating with the plain proofs")
    ap.add_argument("--out", default=None, help="default: profiles/r4_prove_timing.jsonl, with --zk profiles/r5_prove_zk_timing.jsonl")
    a = ap.parse_args()
    if a.reps < 10:
        ap.error("--reps must be at least 10")
    if a.out is None:
        a.out = os.path.join(ROOT, "profiles", "r5_prove_zk_timing.jsonl" if a.zk else "r4_prove_timing.jsonl")
    name, power = card()
    ctx = D.torch_context(0)
    if a.zk:
        emit(a.out, dict(card=name, power_limit=power, **salt_timing(ctx, a.reps)))
    gates, num_selectors = gate_sets()["recursion"]
    fri_config = zf.standard_recursion_fri_config()
    public_inputs = list(range(8))
    for n_log in a.sizes:
        n = 1 << n_log
        rnd = lambda k: torch.randint(0, 2**62, (k, n), dtype=torch.int64, device="cuda")
        common = zp.CommonCircuitData(n_log, gates, num_selectors)
        cs_values = rnd(num_selectors + 2 + 80)
        modes = [False, True] if a.zk else [False]
        datas = {zk: zp.circuit_data(ctx, common, cs_values, fri_config, zero_knowledge=zk) for zk in modes}
        wires = rnd(135)
        run = lambda zk, on_stage=None: zp.prove(ctx, datas[zk], wires, public_inputs, True, on_stage=on_stage)
        for _ in range(a.warmup):
            for zk in modes:
                run(zk)
        ts = {zk: [] for zk in modes}
        for _ in range(a.reps):
            for zk in modes:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                run(zk)
                ts[zk].append((time.perf_counter() - t0) * 1e3)
        splits = {zk: {s: [] for s in zp.PROVE_STAGES} for zk in modes}
        launches = {zk: [] for zk in modes}
        for _ in range(a.reps):
            for zk in modes:
                events = []
                rec = lambda stage: (events.append((stage, torch.cuda.Event(enable_timing=True))), events[-1][1].record())
                l0 = ctx.launch_count
                run(zk, rec)
                launches[zk].append(ctx.launch_count - l0)
                events[-1][1].synchronize()
                for (s, e0), (_, e1) in zip(events, events[1:]):
                    splits[zk][s].append(e0.elapsed_time(e1))
        out = {"card": name, "power_limit": power, "n_log": n_log, "gates": len(gates), "num_challenges": 2,
               "fri": {"rate_bits": fri_config.rate_bits, "cap_height": fri_config.cap_height,
                       "arities": datas[False].fri_params.reduction_arity_bits, "pow_bits": fri_config.proof_of_work_bits,
                       "queries": fri_config.num_query_rounds}, "reps": a.reps}
        for zk in modes:
            v = ts[zk]
            res = {"prove_ms_median": round(statistics.median(v), 3), "min_ms": round(min(v), 3), "max_ms": round(max(v), 3),
                   "stage_ms_median": {s: round(statistics.median(x), 3) for s, x in splits[zk].items()},
                   "launches_per_proof": int(statistics.median(launches[zk]))}
            if a.zk:
                out["zk" if zk else "plain"] = res
            else:
                out.update(res)
        if a.zk:
            out["zk_overhead_ms_median"] = round(out["zk"]["prove_ms_median"] - out["plain"]["prove_ms_median"], 3)
        emit(a.out, out)
        del datas, wires
    ctx.close()


def emit(path, out):
    print(json.dumps(out), flush=True)
    if path:
        with open(path, "a") as f:
            f.write(json.dumps(out) + "\n")


def salt_timing(ctx, reps: int, n_log: int = 16, rate_bits: int = 3, calls: int = 20) -> dict:
    """b200zkp_dev_random_field alone: the SALT_SIZE * 2^(n_log + rate_bits) salt elements of one commitment"""
    count = zp.SALT_SIZE << (n_log + rate_bits)
    out = torch.empty(count, dtype=torch.int64, device="cuda")
    key = os.urandom(32)
    for _ in range(3):
        zp.random_field_device(ctx, key, zp.oracle_nonce(1), count, out=out)
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(calls):
            zp.random_field_device(ctx, key, zp.oracle_nonce(1), count, out=out)
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1) / calls)
    med = statistics.median(ms)
    return {"what": "b200zkp_dev_random_field", "elements": count, "ms_median": round(med, 4), "min_ms": round(min(ms), 4),
            "max_ms": round(max(ms), 4), "reps": reps, "calls_per_rep": calls, "bytes_written_per_s": round(8 * count / med * 1e3)}


if __name__ == "__main__":
    main()
