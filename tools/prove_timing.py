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
GPU only.   python tools/prove_timing.py [--sizes 12 14 16] [--out profiles/r4_prove_timing.jsonl]"""
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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_prove_timing.jsonl"))
    a = ap.parse_args()
    if a.reps < 10:
        ap.error("--reps must be at least 10")
    name, power = card()
    ctx = D.torch_context(0)
    gates, num_selectors = gate_sets()["recursion"]
    fri_config = zf.standard_recursion_fri_config()
    public_inputs = list(range(8))
    for n_log in a.sizes:
        n = 1 << n_log
        rnd = lambda k: torch.randint(0, 2**62, (k, n), dtype=torch.int64, device="cuda")
        common = zp.CommonCircuitData(n_log, gates, num_selectors)
        data = zp.circuit_data(ctx, common, rnd(num_selectors + 2 + 80), fri_config)
        wires = rnd(135)
        run = lambda on_stage=None: zp.prove(ctx, data, wires, public_inputs, True, on_stage=on_stage)
        for _ in range(a.warmup):
            run()
        ts = []
        for _ in range(a.reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            run()
            ts.append((time.perf_counter() - t0) * 1e3)
        splits = {s: [] for s in zp.PROVE_STAGES}
        launches = []
        for _ in range(a.reps):
            events = []
            rec = lambda stage: (events.append((stage, torch.cuda.Event(enable_timing=True))), events[-1][1].record())
            l0 = ctx.launch_count
            run(rec)
            launches.append(ctx.launch_count - l0)
            events[-1][1].synchronize()
            for (s, e0), (_, e1) in zip(events, events[1:]):
                splits[s].append(e0.elapsed_time(e1))
        out = {"card": name, "power_limit": power, "n_log": n_log, "gates": len(gates), "num_challenges": 2,
               "fri": {"rate_bits": fri_config.rate_bits, "cap_height": fri_config.cap_height,
                       "arities": data.fri_params.reduction_arity_bits, "pow_bits": fri_config.proof_of_work_bits,
                       "queries": fri_config.num_query_rounds},
               "prove_ms_median": round(statistics.median(ts), 3), "min_ms": round(min(ts), 3), "max_ms": round(max(ts), 3),
               "reps": a.reps, "stage_ms_median": {s: round(statistics.median(v), 3) for s, v in splits.items()},
               "launches_per_proof": int(statistics.median(launches))}
        print(json.dumps(out), flush=True)
        if a.out:
            with open(a.out, "a") as f:
                f.write(json.dumps(out) + "\n")
        del data, wires
    ctx.close()


if __name__ == "__main__":
    main()
