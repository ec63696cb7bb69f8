"""The interpolation cases of vanish::quotient_point (csrc/vanishing_kernels.cuh), stepped on the CPU by tests/emu, against
tests/interpolation_ref.py (oracle/vanishing_ref.py with the two gates) word for word: the recursion gate set (LowDegreeInterpolation(4)) and HighDegreeInterpolation(3)."""
import ctypes as C
import random

import numpy as np
import pytest

from helpers import P, bitrev_perm
from test_emu_kernels import emu, ptr  # noqa: F401  (the fixture that builds tests/emu)


@pytest.mark.parametrize("interpolation", [(15, 4), (14, 3), (15, 1), (14, 1)])
def test_quotient_point_body_with_interpolation(emu, oracle, interpolation):
    from oracle import perm_ref as PR
    import interpolation_ref as I
    n_log, r = 5, 3
    c = I.recursion_circuit(n_log, seed=2, interpolation=interpolation)
    rnd = random.Random(9)
    betas, gammas, alphas = ([rnd.randrange(P) for _ in range(2)] for _ in range(3))
    zs_pp = PR.partial_products_and_zs([c.wires[j] for j in range(80)], c.sigmas, c.k_is, betas, gammas, 8)
    lde = lambda cols: [oracle.coset_lde(oracle.ifft(np.array(col, np.uint64)), r) for col in cols]
    l_cs, l_w, l_z = lde(c.constants + c.sigmas), lde(c.wires), lde(zs_pp)
    want = np.array(I.quotient_values(c, l_cs, l_w, l_z, betas, gammas, alphas, 8, r, 3), np.uint64)
    perm = bitrev_perm(n_log + r)
    leaf = lambda cols: np.ascontiguousarray(np.stack([col[perm] for col in cols]))
    gates = np.array([[g, c.selector_indices[i], *c.groups[c.selector_indices[i]], *(list(c.gate_params[i]) + [0, 0, 0])[:3]]
                      for i, g in enumerate(c.gates)], np.uint32)
    out = np.zeros((2, 1 << (n_log + r)), np.uint64)
    a = lambda v: np.array(v, np.uint64)
    cs_l, w_l, z_l = leaf(l_cs), leaf(l_w), leaf(l_z)
    emu.emu_quotient_values(ptr(cs_l), ptr(w_l), ptr(z_l), n_log, 3, c.num_selectors, 2, 8, gates.ctypes.data_as(C.POINTER(C.c_uint32)),
                            len(c.gates), ptr(a(c.k_is)), ptr(a(betas)), ptr(a(gammas)), ptr(a(alphas)), ptr(a(c.pi_hash)), ptr(out))
    assert (out == want).all()
