#!/usr/bin/env python3
"""Row N1b timing: compute_quotient_values_device (vanish::quotient_values_kernel plus its small table upload) on random
device-resident LDEs, 2 challenges, quotient_degree_factor 8, for two gate sets:
  five       Noop / Constant / PublicInput / Arithmetic / Poseidon, the set bench.py's prove_chain_latency uses;
  recursion  the 14 gates of a standard_recursion_config verifier circuit (the 13 other kinds + LowDegreeInterpolation(4));
  ecdsa      those 14 plus the plonky2_u32 gates of a circuit built with the ecdsa feature (U32AddMany at two arities): 20.
The kernel's work does not depend on the values, so the matrices are random.  CUDA events, median of --reps calls after
--warmup calls; one JSON line per (set, size), with the card's name and power limit.  B200ZKP_LIB selects another build of the
library of the same `b200zkp_vanishing_desc` layout, so two builds can be timed alternately in one session (a build that
refuses a gate set reports it as unsupported).
GPU only.   python tools/quotient_timing.py [--sizes 12 14 16] [--sets five recursion ecdsa] [--label NAME]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch

from intmax_zkp_core_b200 import _lib, device as D, prover as zp


def gate_sets():
    five = [(zp.GATE_NOOP, 0, (0, 4)), (zp.GATE_CONSTANT, 0, (0, 4)), (zp.GATE_PUBLIC_INPUT, 0, (0, 4)),
            (zp.GATE_ARITHMETIC, 0, (0, 4)), (zp.GATE_POSEIDON, 1, (4, 5))]
    # sorted by degree, with the selector groups gates/selectors.rs forms for max_degree 8 (tests/interpolation_ref.py builds the
    # same list): degrees 0 1 1 1 2 2 2 2 | 3 3 3 | 4 5 | 7
    kinds = [(zp.GATE_NOOP, ()), (zp.GATE_CONSTANT, ()), (zp.GATE_PUBLIC_INPUT, ()), (zp.GATE_POSEIDON_MDS, ()),
             (zp.GATE_BASE_SUM, (2, 63)), (zp.GATE_REDUCING, (43,)), (zp.GATE_REDUCING_EXTENSION, (32,)),
             (zp.GATE_INTERPOLATION_LOW_DEGREE, (4,)), (zp.GATE_ARITHMETIC, ()), (zp.GATE_ARITHMETIC_EXTENSION, ()),
             (zp.GATE_MUL_EXTENSION, ()), (zp.GATE_EXPONENTIATION, (66,)), (zp.GATE_RANDOM_ACCESS, (4, 4, 2)), (zp.GATE_POSEIDON, ())]
    groups = [(0, 6), (6, 11), (11, 13), (13, 14)]
    selector = [0] * 6 + [1] * 5 + [2] * 2 + [3]
    rec = [(k, s, groups[s], pr) for (k, pr), s in zip(kinds, selector)]
    # tests/u32_ref.py's ecdsa_circuit: the degree-4 u32 gates after ExponentiationGate; degrees 0 1 1 1 2 2 | 2 2 3 3 3 |
    # 4 4 4 4 | 4 4 4 | 5 | 7
    u32 = [(zp.GATE_U32_ARITHMETIC, (3,)), (zp.GATE_U32_ADD_MANY, (3, 5)), (zp.GATE_U32_ADD_MANY, (16, 3)),
           (zp.GATE_U32_SUBTRACTION, (6,)), (zp.GATE_U32_RANGE_CHECK, (4,)), (zp.GATE_COMPARISON, (32, 16))]
    kinds = kinds[:12] + u32 + kinds[12:]
    groups = [(0, 6), (6, 11), (11, 15), (15, 18), (18, 19), (19, 20)]
    selector = [0] * 6 + [1] * 5 + [2] * 4 + [3] * 3 + [4, 5]
    ecdsa = [(k, s, groups[s], pr) for (k, pr), s in zip(kinds, selector)]
    return {"five": (five, 2), "recursion": (rec, 4), "ecdsa": (ecdsa, len(groups))}


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=30)
        power = q.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[12, 14, 16])
    ap.add_argument("--sets", nargs="+", default=["five", "recursion"])
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--label", default="")
    a = ap.parse_args()
    if a.reps < 10:
        ap.error("--reps must be at least 10")
    name, power = card()
    ctx = D.torch_context(0)
    sets = gate_sets()
    betas, gammas, alphas = [3, 5], [7, 11], [13, 17]
    for n_log in a.sizes:
        Q = 8 << n_log                                        # n << quotient_degree_bits points
        rnd = lambda k: torch.randint(0, 2**62, (k, Q), dtype=torch.int64, device="cuda")
        wires, zpp = rnd(135), rnd(20)
        out = torch.empty((2, Q), dtype=torch.int64, device="cuda")
        for s in a.sets:
            gates, num_selectors = sets[s]
            common = zp.CommonCircuitData(n_log, gates, num_selectors)
            cs = rnd(num_selectors + 2 + 80)
            rec = {"label": a.label, "lib": os.path.relpath(_lib.LIB_PATH, ROOT), "card": name, "power_limit": power,
                   "gate_set": s, "n_gates": len(gates), "n_log": n_log, "points": Q}
            run = lambda: zp.compute_quotient_values_device(ctx, common, cs, wires, zpp, betas, gammas, alphas, [1, 2, 3, 4], out=out)
            try:
                for _ in range(a.warmup):
                    run()
            except _lib.B200ZkpError as e:
                rec["unsupported"] = str(e)
                print(json.dumps(rec), flush=True)
                continue
            ts = []
            for _ in range(a.reps):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                run()
                e1.record()
                e1.synchronize()
                ts.append(e0.elapsed_time(e1))
            rec.update(quotient_values_ms_median=round(statistics.median(ts), 4), min_ms=round(min(ts), 4),
                       max_ms=round(max(ts), 4), reps=a.reps)
            print(json.dumps(rec), flush=True)
            del cs
    ctx.close()


if __name__ == "__main__":
    main()
