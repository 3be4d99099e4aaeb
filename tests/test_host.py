"""Host logic and the C-ABI library without a GPU: expression compile, symmetry groups, model inputs,
the group compiler of libdmv_b200 (host-side self-check entry), exported symbols, loud failure."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import yaml

from distributed_matvec_b200 import _native as nat
from distributed_matvec_b200.config import basis_from_dict, load_config_from_yaml
from distributed_matvec_b200.expr import compile_terms, parse_expression
from oracle import pyoracle as po

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DATA = os.path.join(ROOT, "data")


def test_expression_parser():
    p = parse_expression("0.8 × σˣ₀ σˣ₁")
    assert len(p) == 1 and p[0].coeff == 0.8 and [f.comp for f in p[0].factors] == ["x", "x"]
    p = parse_expression("σ⁺₀ σ⁻₁ + σ⁻₀ σ⁺₁")
    assert len(p) == 2 and [f.site for f in p[1].factors] == [0, 1]
    p = parse_expression("-0.3j × Sᶻ₁₂")
    assert p[0].coeff == -0.3j and p[0].factors[0].site == 12 and p[0].factors[0].kind == "S"
    with pytest.raises(ValueError):
        parse_expression("σˣ")


def test_heisenberg_bond_compiles_to_two_terms_per_bond():
    off, diag = compile_terms([{"expression": "σˣ₀ σˣ₁", "sites": [[0, 1]]}, {"expression": "σʸ₀ σʸ₁", "sites": [[0, 1]]},
                               {"expression": "σᶻ₀ σᶻ₁", "sites": [[0, 1]]}], 2)
    # sigma^x sigma^x + sigma^y sigma^y = 2 (s+ s- + s- s+): parallel spins cancel exactly
    assert len(off) == 2 and set(off.r.tolist()) == {1, 2} and np.all(off.v == 2) and np.all(off.x == 3)
    assert len(diag) == 1 and diag.s[0] == 3 and diag.v[0] == 1
    off, diag = compile_terms([{"expression": "Sˣ₀ Sˣ₁", "sites": [[0, 1]]}, {"expression": "Sʸ₀ Sʸ₁", "sites": [[0, 1]]},
                               {"expression": "Sᶻ₀ Sᶻ₁", "sites": [[0, 1]]}], 2)
    assert np.allclose(off.v, 0.5) and np.allclose(diag.v, 0.25)


@pytest.mark.parametrize("name,order", [("heisenberg_chain_24_symm", 96), ("heisenberg_chain_32_symm", 128),
                                        ("heisenberg_square_4x4", 256), ("heisenberg_square_6x6", 576),
                                        ("heisenberg_chain_36_symm", 144), ("heisenberg_kagome_12_symm", 2),
                                        ("heisenberg_chain_10", 2)])
def test_group_orders(name, order):
    basis, _ = load_config_from_yaml(os.path.join(DATA, name + ".yaml"))
    assert len(basis.group) == order


def test_inconsistent_sectors_are_rejected():
    b = basis_from_dict({"number_spins": 4, "symmetries": [{"permutation": [1, 2, 3, 0], "sector": 1},
                                                            {"permutation": [2, 3, 0, 1], "sector": 0}]})
    with pytest.raises(ValueError):
        b.group


def test_model_inputs_equal_the_reference_inputs():
    """data/*.yaml are normalised copies of the reference's model inputs (tools/gen_models.py), which are kept verbatim
    under tests/golden/reference_models/."""
    ref_dir = os.path.join(ROOT, "tests", "golden", "reference_models")
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from gen_models import normalise
    names = sorted(f for f in os.listdir(ref_dir) if f.endswith(".yaml"))
    assert len(names) == 22
    for f in names:
        with open(os.path.join(ref_dir, f), encoding="utf-8") as fh:
            ref = normalise(yaml.safe_load(fh))
        with open(os.path.join(DATA, f), encoding="utf-8") as fh:
            ours = yaml.safe_load(fh)
        assert yaml.safe_load(yaml.safe_dump(ref, allow_unicode=True)) == ours, f


def test_library_exports_every_declared_symbol():
    """The C-ABI library loads without a GPU and exports every function include/dmv_b200.h declares."""
    with open(os.path.join(ROOT, "include", "dmv_b200.h"), encoding="utf-8") as f:
        header = f.read()
    declared = set(re.findall(r"\b((?:dmv|ls_chpl)_[a-z0-9_]+)\s*\(", header))
    declared -= {"dmv_context", "dmv_basis_desc", "dmv_operator_desc"}
    lib = nat.lib()
    for name in sorted(declared):
        assert hasattr(lib, name), name
    assert declared == set(nat.EXPORTED_SYMBOLS), declared ^ set(nat.EXPORTED_SYMBOLS)
    assert lib.dmv_version() >= 100
    lib.ls_chpl_init()
    lib.ls_chpl_finalize()


def test_no_silent_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from distributed_matvec_b200 import Operator
    _, matrix = load_config_from_yaml(os.path.join(DATA, "heisenberg_chain_10.yaml"))
    with pytest.raises(nat.DmvError, match="no CPU fallback"):
        Operator(matrix)


@pytest.mark.parametrize("name", ["heisenberg_kagome_12_symm", "issue_01", "heisenberg_chain_24_symm",
                                  "heisenberg_square_4x4", "heisenberg_chain_32_symm", "heisenberg_chain_36_symm",
                                  "heisenberg_square_6x6", "heisenberg_chain_40_symm"])
def test_group_compiler_matches_oracle(name):
    """The orbit program (coset networks x shift chain) that the GPU kernels execute, evaluated on the host
    by the library's self-check entry, gives the oracle's orbit representatives and stabiliser sizes."""
    basis, _ = load_config_from_yaml(os.path.join(DATA, name + ".yaml"))
    g = basis.group
    bd = nat.BasisDesc()
    bd.number_sites, bd.hamming_weight, bd.spin_inversion, bd.has_permutations = (
        basis.number_sites, -1 if basis.hamming_weight is None else basis.hamming_weight, basis.spin_inversion, 1)
    perms, flips, chars = (np.ascontiguousarray(g.perms), np.ascontiguousarray(g.flips),
                           np.ascontiguousarray(g.characters))
    bd.group_order, bd.perms, bd.flips, bd.characters = len(g), perms.ctypes.data, flips.ctypes.data, chars.ctypes.data
    rng = np.random.default_rng(0)
    states = rng.integers(0, 2**basis.number_sites, size=3000, dtype=np.uint64)
    info = np.zeros(6, dtype=np.int64)
    reps = np.zeros_like(states)
    stab = np.zeros(states.shape[0], dtype=np.int32)
    nat.check(nat.lib().dmv_debug_compile_group(C.byref(bd), info.ctypes.data, states.shape[0], states.ctypes.data,
                                                reps.ctypes.data, stab.ctypes.data))
    o_reps, _, o_norms = po.state_info(basis, states)
    assert np.array_equal(reps, o_reps)
    assert info[0] * info[2] * (2 if info[5] else 1) == len(g)      # n_q * n_t * flip = |G|
    if g.all_characters_trivial:
        assert np.allclose(np.sqrt(stab / len(g)), o_norms, atol=1e-15)
    # which chain subgroups are recognised as block rotations (canonical form without walking the chain; the call
    # above has already checked it against the walk for every probe state): mode 2 = one block (chains), 1 = R x k
    ext = np.zeros(12, dtype=np.int64)
    nat.check(nat.lib().dmv_debug_compile_group(C.byref(bd), ext.ctypes.data, -1, None, None, None))
    expect = {"heisenberg_chain_24_symm": (2, 24, 1), "heisenberg_chain_32_symm": (2, 32, 1),
              "heisenberg_chain_36_symm": (2, 36, 1), "heisenberg_chain_40_symm": (2, 40, 1),
              "heisenberg_square_4x4": (1, 4, 4), "heisenberg_square_6x6": (1, 6, 6)}
    if name in expect:
        assert tuple(ext[6:9]) == expect[name], (name, ext)
    print(name, "canon (mode, k, R, pair LUT, chain cosets, chain stages) =", [int(v) for v in ext[6:12]],
          "orbit (n_q, n_stages, n_t) =", [int(v) for v in ext[:3]])
    if name == "heisenberg_square_6x6":      # D4 walked with three reflections (3 + 3 + 5 delta-swaps), no full network
        assert ext[9] == 1 and ext[10] == 8 and ext[11] <= 7 * 5


@pytest.mark.parametrize("name", ["heisenberg_square_4x4", "heisenberg_chain_24_symm", "heisenberg_kagome_12_symm"])
def test_canonical_form_sweep_over_a_whole_product(name):
    """tools/canonical_form_sweep.py on the models small enough for the CPU suite: every state one product canonicalises
    (alpha ^ x_t for every emitting term, and alpha itself) through the device functions compiled for the host and through
    the oracle; representatives and norms agree bit for bit.  The same sweep at full size (6 x 6 square: 601 067 490
    states; chain_36_symm: 1 230 759 430): profiles/r02_canonical_form_sweep_*.log."""
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "canonical_form_sweep.py"), name, "2"],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "representative mismatches 0, norm mismatches 0" in out.stdout, out.stdout


def test_tridiagonal_lowest_eigenpair():
    """Host half of dmv_lanczos (Sturm bisection + pivoted inverse iteration) against numpy, including nearly
    decoupled blocks, tiny off-diagonals and clustered eigenvalues."""
    rng = np.random.default_rng(4)
    cases = []
    for k in (1, 2, 3, 10, 57, 300):
        cases.append((rng.normal(size=k), rng.normal(size=max(k - 1, 0))))
    a, b = rng.normal(size=40), rng.normal(size=39)
    b[17] = 1e-13                                   # nearly decoupled blocks
    cases.append((a, b))
    cases.append((np.full(30, 2.0), np.full(29, -1.0)))          # discrete Laplacian
    cases.append((np.concatenate([np.full(10, -3.0), rng.normal(size=10)]), np.full(19, 1e-9)))   # clustered
    for a, b in cases:
        k = a.shape[0]
        a = np.ascontiguousarray(a); b = np.ascontiguousarray(b if k > 1 else np.zeros(1))
        theta, vec = C.c_double(), np.zeros(k)
        nat.check(nat.lib().dmv_debug_tridiagonal_lowest(k, a.ctypes.data, b.ctypes.data, C.byref(theta), vec.ctypes.data))
        T = np.diag(a) + (np.diag(b[:k - 1], 1) + np.diag(b[:k - 1], -1) if k > 1 else 0)
        w = np.linalg.eigvalsh(T)
        assert abs(theta.value - w[0]) <= 1e-12 * max(1.0, np.abs(w).max())
        assert abs(np.linalg.norm(vec) - 1.0) < 1e-12
        assert np.linalg.norm(T @ vec - theta.value * vec) <= 1e-8 * max(1.0, np.abs(w).max())


def _torus_generators(k, R, reflections=True):
    """Translations (and reflections) of an R x k torus numbered row by row, site = k y + x."""
    n = k * R
    gens = [[k * (i // k) + ((i % k + 1) % k) for i in range(n)]]
    if R > 1:
        gens.append([(i + k) % n for i in range(n)])
    if reflections:
        gens.append([k * (i // k) + (k - 1 - i % k) for i in range(n)])          # x -> -x
        if R > 1:
            gens.append([k * (R - 1 - i // k) + i % k for i in range(n)])        # y -> -y
        if R == k and k > 1:
            gens.append([k * (i % k) + i // k for i in range(n)])                # transpose
    return [{"permutation": g, "sector": 0} for g in gens]


@pytest.mark.parametrize("k,R,inversion,expect_mode", [
    (5, 1, None, 2), (7, 1, 1, 2), (12, 1, 1, 2), (33, 1, 1, 2), (40, 1, None, 2), (64, 1, 1, 2),   # chains: zero runs
    (2, 2, 1, 1), (3, 2, None, 1), (4, 3, 1, 1), (5, 5, 1, 1), (6, 4, None, 1), (4, 8, 1, 1),      # tori: pair LUT
    (6, 6, 1, 1), (6, 6, None, 1), (3, 3, 1, 1), (4, 4, None, 1), (6, 8, 1, 1), (3, 8, None, 1), (5, 4, 1, 1),
    (7, 3, 1, 1), (8, 8, 1, 1), (8, 2, None, 1),                                                  # tori: single-block LUT
    (16, 2, 1, 0)])                                                                               # blocks too wide: walk
def test_block_rotation_canonical_form_on_random_lattices(k, R, inversion, expect_mode):
    """The canonical form of the translation subgroup (zero-run search, block LUT, pair LUT, coset chain through cheap
    involutions) against the oracle's bit-by-bit group action, for chains and tori of many shapes -- evaluated on the
    host by the library (the same functions the kernels run).  dmv_debug_compile_group additionally checks every probe
    state against the chain walk and runs the 266-state self-check of the compiler."""
    from distributed_matvec_b200.symmetry import build_group
    from distributed_matvec_b200.config import basis_from_dict
    n = k * R
    basis = basis_from_dict({"number_spins": n, "hamming_weight": None, "spin_inversion": inversion,
                             "symmetries": _torus_generators(k, R)})
    g = basis.group
    bd = nat.BasisDesc()
    bd.number_sites, bd.hamming_weight, bd.spin_inversion, bd.has_permutations = n, -1, inversion or 0, 1
    perms, flips, chars = (np.ascontiguousarray(g.perms), np.ascontiguousarray(g.flips), np.ascontiguousarray(g.characters))
    bd.group_order, bd.perms, bd.flips, bd.characters = len(g), perms.ctypes.data, flips.ctypes.data, chars.ctypes.data
    rng = np.random.default_rng(k * 100 + R)
    hi = 2**n if n < 64 else 2**63
    states = rng.integers(0, hi, size=1500, dtype=np.uint64)
    if n == 64:
        states |= rng.integers(0, 2, size=1500, dtype=np.uint64) << np.uint64(63)
    states[:6] = [0, (2**n - 1) if n < 64 else 2**64 - 1, 1, 0x5555555555555555 & (2**n - 1 if n < 64 else 2**64 - 1),
                  (1 << (n - 1)), 3]
    states[6:300] &= rng.integers(0, hi, size=294, dtype=np.uint64)       # sparse words: long zero runs, many ties
    if R > 1:   # lattices with repeated rows / columns and transpose-symmetric patterns: tied top pairs
        bm = (1 << k) - 1
        for j in range(300, 600):
            rows = rng.integers(0, bm + 1, size=2)
            pattern = [int(rows[(y * int(rng.integers(1, 3))) % 2]) for y in range(R)]
            states[j] = sum(r << (k * y) for y, r in enumerate(pattern)) & (hi - 1 if n < 64 else 2**64 - 1)
        if R == k:
            for j in range(600, 800):
                m = rng.integers(0, 2, size=(k, k))
                m = np.triu(m) | np.triu(m, 1).T        # symmetric bit matrix
                states[j] = sum(int(m[y, a]) << (k * y + a) for y in range(R) for a in range(k))
    reps = np.zeros_like(states)
    stab = np.zeros(states.shape[0], dtype=np.int32)
    info = np.zeros(6, dtype=np.int64)
    nat.check(nat.lib().dmv_debug_compile_group(C.byref(bd), info.ctypes.data, states.shape[0], states.ctypes.data,
                                                reps.ctypes.data, stab.ctypes.data))
    o_reps, _, o_norms = po.state_info(basis, states)
    assert np.array_equal(reps, o_reps)
    ext = np.zeros(12, dtype=np.int64)
    nat.check(nat.lib().dmv_debug_compile_group(C.byref(bd), ext.ctypes.data, -1, None, None, None))
    assert ext[6] == expect_mode, (k, R, [int(v) for v in ext])
    # full-space-group canonical form (orbit_min_torus): needs both reflections, 3 <= k <= 6, 3 <= R <= 8
    ext = np.zeros(16, dtype=np.int64)
    nat.check(nat.lib().dmv_debug_compile_group(C.byref(bd), ext.ctypes.data, -2, None, None, None))
    want = 0
    if expect_mode == 1 and 3 <= k <= 6 and 3 <= R <= 8:
        want = 2 if R == k else 1
    assert ext[12] == want, (k, R, [int(v) for v in ext])
    assert ext[15] == (2 if expect_mode == 2 else 0)      # chains with the mirror: one pass over the runs
    if expect_mode == 1:
        assert (ext[7], ext[8]) == (k, R) and ext[9] == (1 if 2 * k <= 12 else 0)
