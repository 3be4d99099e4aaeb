"""Edge-case parity of the row kernels: every selectable k_rows / k_rows_batch / k_gather variant, the open-addressing
table at its collisions and wrap-around, states missing from the basis, 1- to 64-site bases and empty ranks -- each
product compared element by element with the exactly rounded sum of its row.

Exact reference (section 1).  H is assembled from the oracle: the off-diagonal entries h_ij of computeOffDiag with unit
x (source j = the column, po.state_index of the emitted state = the row) and the diagonal d_i of po.apply_diag (the
diagonal terms commute with the group, so this is also the projected diagonal).  The assembly is checked against
po.matvec_global before it is trusted.  For a vector x, y_i = sum_j h_ij x_j is summed exactly: every product is split
into two doubles without error (Dekker's two-product) and math.fsum rounds the sum of the pieces correctly; y_i is kept
as hi + lo with lo the correctly rounded residual, so |y_i - (hi + lo)| <= u |lo|.  A CPU test checks this against
fractions.Fraction arithmetic on the same doubles.

Bound.  A kernel result is accepted element by element when

    |y_i - y_i^exact| <= (T_i + 6) u sum_j |h_ij| |x_j|,     u = 2^-53,

with T_i the number of terms of row i: the diagonal terms active on state i plus the larger of the entries the oracle
puts into row i and the entries it emits from source i (the push kernels receive the first, the row kernels walk the
second).  The kernels add the diagonal terms of a state in their own order, and d_i may cancel to nearly 0, so the
diagonal enters the sum of absolute values as |x_i| sum_t |v_t| over its active terms rather than as |d_i| |x_i|.  Derivation for
k_rows (the longest operation sequence; k_gather has norms 1 and omits the first two roundings):

    v_j = fl(x_j n_j)                        (k_table_fill)           1 rounding
    r_i = fl(1 / n_i)                                                  1 rounding
    a_i = fma(c_t, v_j, a_i) over the terms  (T_i - 1 fused steps)     T_i - 1 roundings on the longest path
    y_i = fma(r_i, a_i, fl(d_i x_i))                                   1 rounding (+1 on the diagonal product, and
                                                                       one per diagonal term summed into d_i)

so each product c_t x_j n_j / n_i reaches y_i through at most T_i + 2 roundings.  The oracle's h_ij = c_t chi (n_i / n_j)
is itself rounded twice (the norm ratio and the product; chi = +-1 here), so the kernel's exact coefficient and h_ij
differ by at most 2 u relative.  First order: T_i + 4 units of u per unit of sum |h_ij x_j|; the remaining 2 cover the
second-order terms of gamma_m = m u / (1 - m u) and the atomics of the scatter kernels, whose order is arbitrary but whose
chain is no longer.  Complex vectors are checked per component (the operators here are real).
"""
import dataclasses
import math
import os
from fractions import Fraction
from types import SimpleNamespace

import numpy as np
import pytest

from distributed_matvec_b200.config import basis_from_dict, load_config_from_yaml, operator_from_dict
from oracle import pyoracle as po

DATA = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "data")
U = 2.0 ** -53


def _load(name):
    return load_config_from_yaml(os.path.join(DATA, name + ".yaml"))


def _custom(n, hw, terms, **basis_kw):
    basis = basis_from_dict({"number_spins": n, "hamming_weight": hw, **basis_kw})
    return basis, operator_from_dict({"terms": terms}, basis)


def _ring(n, hw, symmetries=(), zz=1.0):
    """Heisenberg ring on n sites at Hamming weight hw; symmetries: 'T' translations, 'M' mirror (sector 0)."""
    bonds = [[i, (i + 1) % n] for i in range(n)]
    gens = []
    if "T" in symmetries:
        gens.append({"permutation": [(i + 1) % n for i in range(n)], "sector": 0})
    if "M" in symmetries:
        gens.append({"permutation": [n - 1 - i for i in range(n)], "sector": 0})
    terms = [{"expression": "σˣ₀ σˣ₁", "sites": bonds}, {"expression": "σʸ₀ σʸ₁", "sites": bonds},
             {"expression": f"{zz} × σᶻ₀ σᶻ₁", "sites": bonds}]
    return _custom(n, hw, terms, **({"symmetries": gens} if gens else {}))


GENERAL = {
    # two-body, bond-dependent couplings: k_gather with a coefficient LUT, 32-bit rows
    "anisotropic_bonds": lambda: _custom(12, 6, [
        {"expression": "σ⁺₀ σ⁻₁", "sites": [[i, (i + 1) % 12] for i in range(12)]},
        {"expression": "σ⁻₀ σ⁺₁", "sites": [[i, (i + 1) % 12] for i in range(12)]},
        {"expression": "0.37 × σ⁺₀ σ⁻₁", "sites": [[i, (i + 3) % 12] for i in range(0, 12, 2)]},
        {"expression": "0.37 × σ⁻₀ σ⁺₁", "sites": [[i, (i + 3) % 12] for i in range(0, 12, 2)]},
        {"expression": "1.3 × σᶻ₀ σᶻ₁", "sites": [[i, (i + 1) % 12] for i in range(12)]}]),
    # more than 32 sites: the 64-bit rows of k_gather, uniform coefficient
    "wide_two_magnon": lambda: _custom(34, 2, [
        {"expression": "σˣ₀ σˣ₁", "sites": [[i, (i + 1) % 34] for i in range(34)]},
        {"expression": "σʸ₀ σʸ₁", "sites": [[i, (i + 1) % 34] for i in range(34)]},
        {"expression": "σᶻ₀ σᶻ₁", "sites": [[i, (i + 1) % 34] for i in range(34)]}]),
    # spin inversion (odd sector): k_gather with the inversion projection, directory index
    "inversion_two_body": lambda: _custom(12, 6, [
        {"expression": "σˣ₀ σˣ₁", "sites": [[i, (i + 1) % 12] for i in range(12)]},
        {"expression": "σʸ₀ σʸ₁", "sites": [[i, (i + 1) % 12] for i in range(12)]},
        {"expression": "0.5 × σᶻ₀ σᶻ₁", "sites": [[i, (i + 2) % 12] for i in range(12)]}], spin_inversion=-1),
    "heisenberg_chain_16": lambda: _load("heisenberg_chain_16"),
}


def _model(name):
    return GENERAL[name]() if name in GENERAL else _load(name)


def _x(n, cplx, seed):
    rng = np.random.default_rng(seed)
    x = rng.random(n) - 0.5
    if cplx:
        x = x + 1j * (rng.random(n) - 0.5)
    return x


# ------------------------------------------------------------------------------------------------------------------
# 1. exact per-row reference
# ------------------------------------------------------------------------------------------------------------------
def _two_prod(a, b):
    """a * b = p + e exactly (Dekker / Veltkamp; no overflow or underflow at these magnitudes)."""
    f = 134217729.0   # 2^27 + 1
    ca, cb = f * a, f * b
    ah = ca - (ca - a)
    al = a - ah
    bh = cb - (cb - b)
    bl = b - bh
    p = a * b
    e = ((ah * bh - p) + ah * bl + al * bh) + al * bl
    return p, e


class ExactRef:
    """The nonzeros of H from the oracle, and y = H x summed exactly per row."""

    def __init__(self, matrix, reps):
        self.matrix = matrix
        self.reps = np.ascontiguousarray(reps, dtype=np.uint64)
        n = self.n = self.reps.shape[0]
        betas, coeffs, _, offsets = po.compute_off_diag(matrix, 1, self.reps, np.ones(n))
        assert np.all(coeffs.imag == 0), "the reference handles real operators"
        cols = np.repeat(np.arange(n), np.diff(offsets))
        rows = po.state_index(self.reps, betas)
        assert np.all(rows >= 0)
        d = po.apply_diag(matrix, self.reps, np.ones(n))
        # the kernels sum the diagonal terms of a state themselves: count them as terms of the row, and bound their
        # rounding by the sum of their absolute values (d_i may cancel to nearly 0)
        dg = matrix.diag
        ones = SimpleNamespace(diag=dataclasses.replace(dg, v=np.ones_like(dg.v), s=np.zeros_like(dg.s)))
        absd = SimpleNamespace(diag=dataclasses.replace(dg, v=np.abs(dg.v).astype(dg.v.dtype), s=np.zeros_like(dg.s)))
        n_diag = np.real(po.apply_diag(ones, self.reps, np.ones(n))).round().astype(np.int64)
        self.diag_abs = np.real(po.apply_diag(absd, self.reps, np.ones(n)))
        # one list of terms: the diagonal first, then the off-diagonal entries, grouped by row
        rows = np.concatenate([np.arange(n), rows])
        cols = np.concatenate([np.arange(n), cols])
        h = np.concatenate([np.real(d), coeffs.real])
        order = np.argsort(rows, kind="stable")
        self.rows, self.cols, self.h = rows[order], cols[order], h[order]
        self.bounds = np.searchsorted(self.rows, np.arange(n + 1))
        emitted = np.diff(offsets)
        received = np.diff(self.bounds) - 1
        self.terms = np.maximum(emitted, received) + np.maximum(n_diag, 1)
        self.emitted_betas, self.offsets = betas, offsets

    def _exact_real(self, x):
        p, e = _two_prod(self.h, x[self.cols])
        s = np.abs(self.h) * np.abs(x[self.cols])
        pl, el = p.tolist(), e.tolist()
        hi = np.empty(self.n)
        lo = np.empty(self.n)
        b = self.bounds.tolist()
        for i in range(self.n):
            parts = pl[b[i]:b[i + 1]] + el[b[i]:b[i + 1]]
            hi[i] = math.fsum(parts)
            parts.append(-hi[i])
            lo[i] = math.fsum(parts)
        absum = np.add.reduceat(s, self.bounds[:-1]) if self.n else np.zeros(0)
        diag = self.bounds[:-1]                          # the diagonal is the first entry of every row
        absum += np.maximum(self.diag_abs - np.abs(self.h[diag]), 0.0) * np.abs(x)
        return hi, lo, absum

    def exact(self, x):
        """-> list of (hi, lo, sum |h| |x|) per real component of x."""
        x = np.asarray(x)
        if np.iscomplexobj(x):
            return [self._exact_real(np.ascontiguousarray(x.real)), self._exact_real(np.ascontiguousarray(x.imag))]
        return [self._exact_real(np.ascontiguousarray(x, dtype=np.float64))]

    def excess(self, y, x, ex=None):
        """max_i |y_i - y_i^exact| / bound_i  (<= 1: accepted)."""
        ex = ex if ex is not None else self.exact(x)
        y = np.asarray(y)
        comps = [y.real, y.imag] if np.iscomplexobj(y) else [y]
        assert len(comps) == len(ex)
        worst = 0.0
        for yc, (hi, lo, s) in zip(comps, ex):
            err = np.abs((yc - hi) - lo)
            bound = (self.terms + 6) * U * s
            with np.errstate(divide="ignore", invalid="ignore"):
                r = np.where(bound > 0, err / np.where(bound > 0, bound, 1.0), np.where(err > 0, np.inf, 0.0))
            worst = max(worst, float(r.max(initial=0.0)))
        return worst

    def assert_close(self, y, x, ex=None, what=""):
        e = self.excess(y, x, ex)
        assert e <= 1.0, (what, e)


_REFS = {}


def _ref(key, matrix, reps):
    if key not in _REFS:
        _REFS[key] = ExactRef(matrix, reps)
    return _REFS[key]


@pytest.mark.parametrize("name", ["heisenberg_kagome_12_symm", "heisenberg_square_4x4", "heisenberg_chain_10",
                                  "anisotropic_bonds", "inversion_two_body"])
def test_reference_assembly_matches_oracle(name):
    basis, matrix = _model(name)
    reps, _ = po.enumerate_states(basis)
    ref = ExactRef(matrix, reps)
    for cplx in (False, True):
        x = _x(reps.shape[0], cplx, 3)
        want = po.matvec_global(matrix, reps, x, 1)
        ex = ref.exact(x)
        got = ex[0][0] + 1j * ex[1][0] if cplx else ex[0][0]
        assert np.abs(got - want).max() <= 1e-13 * max(1.0, np.abs(want).max())


def test_reference_is_exact_against_fractions():
    """hi + lo equals the exact rational sum of the double products to within u |lo|."""
    basis, matrix = _load("heisenberg_chain_24_symm")
    reps, _ = po.enumerate_states(basis)
    ref = ExactRef(matrix, reps)
    x = _x(reps.shape[0], False, 5)
    (hi, lo, _), = ref.exact(x)
    for i in np.random.default_rng(0).choice(reps.shape[0], 200, replace=False):
        a, b = ref.bounds[i], ref.bounds[i + 1]
        exact = sum((Fraction(float(h)) * Fraction(float(x[c])) for h, c in zip(ref.h[a:b], ref.cols[a:b])), Fraction(0))
        assert abs(exact - Fraction(hi[i]) - Fraction(lo[i])) <= Fraction(U) * abs(Fraction(lo[i])), i


def test_reference_bound_accepts_the_oracle():
    for name in ("heisenberg_chain_24_symm", "heisenberg_square_4x4", "heisenberg_chain_16"):
        basis, matrix = _load(name)
        reps, _ = po.enumerate_states(basis)
        ref = ExactRef(matrix, reps)
        for cplx in (False, True):
            x = _x(reps.shape[0], cplx, 7)
            ref.assert_close(po.matvec_global(matrix, reps, x, 1), x, what=(name, cplx))


def test_reference_bound_rejects_a_moved_element():
    basis, matrix = _load("heisenberg_chain_24_symm")
    reps, _ = po.enumerate_states(basis)
    ref = ExactRef(matrix, reps)
    x = _x(reps.shape[0], False, 7)
    ex = ref.exact(x)
    hi, lo, s = ex[0]
    y = hi.copy()
    assert ref.excess(y, x, ex) <= 1.0
    i = int(np.argmax(s))
    y[i] += 8 * (ref.terms[i] + 6) * U * s[i]
    assert ref.excess(y, x, ex) > 1.0


def test_reference_cost_on_the_largest_edge_basis():
    """The exact reference stays cheap on the largest basis of the edge set (C(64, 3) = 41 664 states)."""
    import time
    basis, matrix = _ring(64, 3)
    reps, _ = po.enumerate_states(basis)
    assert reps.shape[0] == 41664
    t = time.perf_counter()
    ref = ExactRef(matrix, reps)
    ref.exact(_x(reps.shape[0], True, 1))
    assert time.perf_counter() - t < 30.0


# ------------------------------------------------------------------------------------------------------------------
# 3 (host half). the open-addressing tables restated: table_slot (dmv_device.cuh) and the bucket counts (dmv_api.cu)
# ------------------------------------------------------------------------------------------------------------------
def _table_slot(keys, n_buckets):
    with np.errstate(over="ignore"):
        h = np.asarray(keys, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15)
    return (((h >> np.uint64(32)) * np.uint64(n_buckets)) >> np.uint64(32)).astype(np.int64)


# name: (buckets per state, slots per bucket) of the table a product uses (auto sizing on a small basis)
TABLES = {"f64": (2, 2), "c128": (8, 1), "batch": (8, 1), "c128_4": (4, 1), "c128_2": (2, 1),
          "batch_4": (4, 1), "batch_2": (2, 1)}


def _probe_lengths(reps, per_state, cap):
    """Linear probing with `cap` slots per bucket, keys inserted in index order.  -> (home, final bucket, buckets
    probed) per key.  Only what does not depend on the order is used: which buckets are full, and how many keys cross
    each bucket boundary (k_table_insert places the keys through concurrent atomicCAS in no fixed order, so WHICH key
    ends up displaced is not known on the host)."""
    n_buckets = max(16, per_state * reps.shape[0])
    home = _table_slot(reps, n_buckets)
    fill = np.zeros(n_buckets, dtype=np.int64)
    final = np.empty_like(home)
    for k, b in enumerate(home.tolist()):
        while fill[b] == cap:
            b = b + 1 if b + 1 < n_buckets else 0
        fill[b] += 1
        final[k] = b
    probes = (final - home) % n_buckets + 1
    return home, final, probes, n_buckets


def _forced_chain(reps, per_state, cap, longest=256):
    """True when EVERY insertion order leaves some key >= 2 buckets past its home (a look-up probes >= 3 buckets): some
    circular window of buckets [s .. b] holds the homes of more keys than the cap (b - s + 2) slots of [s .. b + 1], so
    at least one of those keys is stored beyond b + 1."""
    n_buckets = max(16, per_state * reps.shape[0])
    counts = np.bincount(_table_slot(reps, n_buckets), minlength=n_buckets)
    ext = np.concatenate([counts, counts])
    csum = np.concatenate([[0], np.cumsum(ext)])
    for length in range(1, min(n_buckets - 1, longest) + 1):
        in_window = csum[length:length + n_buckets] - csum[:n_buckets]     # homes in [s .. s + length - 1]
        if np.any(in_window > cap * (length + 1)):
            return True
    return False


def _table_properties(reps, table):
    """-> (some key crosses from the last bucket to bucket 0, every insertion order has a probe chain of >= 3)."""
    per_state, cap = TABLES[table]
    home, final, _, _ = _probe_lengths(reps, per_state, cap)
    return bool(np.any(final < home)), _forced_chain(reps, per_state, cap)


# Small symmetric rings (n, hw, T = translations / M = mirror) whose tables wrap from the last bucket to bucket 0 and
# have probe chains of >= 3 buckets in every insertion order (_forced_chain), found by a search over rings of 4 .. 24
# sites.  At 8 one-slot buckets per state
# (the complex128 and batch tables) no small ring's cluster reaches the last bucket, so the wrap of those tables is
# covered at 4 and 2 buckets per state ("rows_table_per_state"), the density large bases get automatically.
TABLE_MODELS = {
    "f64": [(21, 5, "TM"), (22, 6, "TM")],
    "c128": [(24, 4, "T")], "batch": [(24, 4, "T")],
    "c128_4": [(18, 5, "TM"), (14, 5, "TM")], "batch_4": [(18, 5, "TM"), (14, 5, "TM")],
    "c128_2": [(14, 3, "TM"), (12, 3, "TM")], "batch_2": [(14, 3, "TM"), (12, 3, "TM")],
}
NO_WRAP_AT_AUTO = ("c128", "batch")


@pytest.mark.parametrize("table", sorted(TABLES))
def test_table_models_reach_wrap_and_long_chains(table):
    wrap = chain = False
    for spec in TABLE_MODELS[table]:
        basis, matrix = _ring(*spec)
        reps, _ = po.enumerate_states(basis)
        w, c = _table_properties(reps, table)
        wrap |= w
        chain |= c
    assert chain, table
    assert wrap or table in NO_WRAP_AT_AUTO, table


# ------------------------------------------------------------------------------------------------------------------
# GPU tests
# ------------------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.fail("these tests need a CUDA device (no CPU fallback exists)")
    return torch


def _op(matrix, **options):
    from distributed_matvec_b200 import Operator
    op = Operator(matrix)
    for k, v in options.items():
        op.set_option(k, v)
    return op


def _dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


ROWS_SMALL = {"heisenberg_kagome_12_symm": 0, "heisenberg_chain_24_symm": 0, "heisenberg_square_4x4": 4}


# ---- 2. variant matrix -----------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", sorted(ROWS_SMALL))
def test_rows_instantiations_full_vectors(torch_cuda, name):
    """k_rows<CE, TK, MPH, CTAS> for every rows_ctas x rows_index x element type, full vectors against the exact sums."""
    torch = torch_cuda
    basis, matrix = _load(name)
    op = _op(matrix, mode=1)
    op.basis.build()
    reps = op.basis.representatives()
    ref = _ref(name, matrix, reps)
    tk = ROWS_SMALL[name]
    for cplx in (False, True):
        x = _x(reps.shape[0], cplx, 41)
        ex = ref.exact(x)
        for rows_index in (0, 1):
            op.set_option("rows_index", rows_index)
            for ctas in (2, 3, 4):
                op.set_option("rows_ctas", ctas)
                y = op.matvec(_dev(torch, x)).cpu().numpy()
                assert op.info("rows") == 1
                if rows_index == 1:        # the dense index has one instantiation per TK, two CTAs per SM
                    want = 200 + 10 * tk + 1
                else:                      # four CTAs per SM has no TK = 4 instantiation: the generic orbit minimum
                    want = 100 * ctas + 10 * (0 if (ctas == 4 and tk == 4) else tk)
                assert op.info("rows_kernel") == want, (rows_index, ctas, op.info("rows_kernel"))
                ref.assert_close(y, x, ex, (name, cplx, rows_index, ctas))
    op.close()


@gpu
def test_rows_instantiations_square_6x6_sampled(torch_cuda):
    """TK = 6 (the 6x6 torus, 15.8 M states) with two and four CTAs per SM: 2048 sampled rows against the oracle."""
    torch = torch_cuda
    basis, matrix = _load("heisenberg_square_6x6")
    po.set_num_threads(max(1, len(os.sched_getaffinity(0))))
    op = _op(matrix, mode=1)
    op.basis.build()
    reps = op.basis.representatives()
    rows = np.sort(np.random.default_rng(17).choice(reps.shape[0], size=2048, replace=False))
    rows_d = _dev(torch, rows)
    model = po.Model(matrix)
    for cplx in (False, True):
        x = _x(reps.shape[0], cplx, 43)
        expect = po.expected_rows(matrix, reps, x, rows, model)
        xd = _dev(torch, x)
        for ctas in (2, 4):
            op.set_option("rows_ctas", ctas)
            got = op.matvec(xd)[rows_d].cpu().numpy()
            assert op.info("rows_kernel") == 100 * ctas + 60
            assert np.abs(got - expect).max() <= 1e-12 * np.abs(expect).max(), (cplx, ctas)
        del xd
    op.close()


@gpu
@pytest.mark.parametrize("name", ["heisenberg_chain_24_symm", "heisenberg_square_4x4"])
def test_rows_batch_widths(torch_cuda, name):
    """k_rows_batch at every width: real k = 1 .. 7 (7 = a batch of six and a batch of one), complex k = 1 .. 4, every
    column against the exact sums, and bit for bit against the single-vector k_rows with the dense index.  Both add a
    row's terms in the order they are popped (k_rows_batch keeps one request in flight; the dense-index k_rows retries a
    taken bucket of its overflow table in place), with the same fma per term, the same table values x n and the same
    final fma(1 / n_b, acc, d x).  The open-table k_rows is not bit-equal: it keeps two requests in flight and issues the
    retry of a term whose home bucket is taken after the request of the next term, so that term is added one place
    later; which keys are displaced depends on the order of the concurrent inserts of k_table_insert."""
    torch = torch_cuda
    tk = ROWS_SMALL[name]
    basis, matrix = _load(name)
    single = _op(matrix, mode=1, rows_index=1)
    single.basis.build()
    reps = single.basis.representatives()
    n = reps.shape[0]
    ref = _ref(name, matrix, reps)
    for cplx, ks in ((False, range(1, 8)), (True, range(1, 5))):
        for k in ks:
            X = np.stack([_x(n, cplx, 100 + j) for j in range(k)])
            op = _op(matrix, mode=1, rows_batch_min=1)
            op.basis.build()
            assert op.info("rows_batch_kernel") == 0
            Y = op.matvec_batch(_dev(torch, X)).cpu().numpy()
            assert op.info("rows_batch_kernel") == 200 + 10 * tk    # the batch kernel ran ...
            assert op.info("rows_kernel") == 0                      # ... and no single-vector k_rows
            op.close()
            for j in range(k):
                ref.assert_close(Y[j], X[j], what=(name, cplx, k, j))
                y1 = single.matvec(_dev(torch, X[j])).cpu().numpy()
                assert single.info("rows_kernel") == 200 + 10 * tk + 1
                assert np.array_equal(Y[j], y1), (name, cplx, k, j)
    single.close()


GATHER_MODELS = {"anisotropic_bonds": (1, 0), "wide_two_magnon": (0, 1), "inversion_two_body": (1, 1),
                 "heisenberg_chain_16": (1, 1)}   # name: (narrow rows, uniform coefficient)


@gpu
@pytest.mark.parametrize("name", sorted(GATHER_MODELS))
def test_gather_walks(torch_cuda, name):
    """k_gather with each walk over the emitting groups, f64 and c128, one vector and batches of 4 and 5: full vectors
    against the exact sums (the walks add a row's terms in different orders), each walk bit-reproducible."""
    torch = torch_cuda
    basis, matrix = _model(name)
    op = _op(matrix)
    op.basis.build()
    reps = op.basis.representatives()
    n = reps.shape[0]
    narrow, uniform = GATHER_MODELS[name]
    assert op.info("gather") == 1 and op.info("gather_narrow") == narrow and op.info("gather_uniform") == uniform
    ref = _ref(name, matrix, reps)
    for cplx in (False, True):
        X = np.stack([_x(n, cplx, 200 + j) for j in range(5)])
        exs = [ref.exact(X[j]) for j in range(5)]
        for walk, index in ((0, -1), (1, -1), (2, -1), (0, 0), (1, 0), (2, 0)):   # Lin tables, then the directory
            op.set_option("gather_walk", walk)
            op.set_option("index", index)
            assert op.info("index_mode") == (3 if index == -1 else 0)
            for k in (1, 4, 5):
                Xd = _dev(torch, X[:k])
                Y = (op.matvec(Xd[0])[None] if k == 1 else op.matvec_batch(Xd)).cpu().numpy()
                Y2 = (op.matvec(Xd[0])[None] if k == 1 else op.matvec_batch(Xd)).cpu().numpy()
                assert np.array_equal(Y, Y2), (name, cplx, walk, index, k)
                for j in range(k):
                    ref.assert_close(Y[j], X[j], exs[j], (name, cplx, walk, index, k, j))
    op.close()


CANON_DEFAULT = {"heisenberg_kagome_12_symm": 0, "heisenberg_chain_24_symm": 2, "heisenberg_square_4x4": 1}


@gpu
def test_canonical_forms_forced(torch_cuda):
    """Every canonical form of the orbit minimum forced on the products (k_rows, scatter, queued rows) of the small
    symmetric models, full vectors against the exact sums; modes 1 and 2 on sampled rows of the 6x6 torus.  "canon" = 0
    walks the chain (canon_mode 0); 1 and 2 keep the block-rotation form of the chain subgroup but drop the torus and
    dihedral forms (torus_mode 0, so k_rows takes its TK = 0 instantiation); 2 also drops the pair LUT and the coset
    networks, which no info key reports -- those products are held to the exact sums like the others."""
    torch = torch_cuda
    for name, default in CANON_DEFAULT.items():
        basis, matrix = _load(name)
        op = _op(matrix)
        op.basis.build()
        reps = op.basis.representatives()
        ref = _ref(name, matrix, reps)
        x = _x(reps.shape[0], True, 47)
        ex = ref.exact(x)
        tk = ROWS_SMALL[name]
        for canon in (-1, 0, 1, 2):
            op.set_option("canon", canon)
            assert op.info("canon_mode") == (0 if canon == 0 else default), (name, canon)
            if canon == -1:
                assert op.info("torus_mode") == (2 if tk else op.info("torus_mode"))
            else:
                assert op.info("torus_mode") == 0, (name, canon)
            for m, rows in ((1, -1), (0, -1), (1, 0)):
                op.set_option("mode", m)
                op.set_option("rows", rows)
                ref.assert_close(op.matvec(_dev(torch, x)).cpu().numpy(), x, ex, (name, canon, m, rows))
                if (m, rows) == (1, -1):
                    assert op.info("rows_kernel") == 300 + 10 * (tk if canon == -1 else 0), (name, canon)
            op.set_option("mode", -1)
            op.set_option("rows", -1)
        op.close()
    basis, matrix = _load("heisenberg_square_6x6")
    po.set_num_threads(max(1, len(os.sched_getaffinity(0))))
    op = _op(matrix)
    op.basis.build()
    reps = op.basis.representatives()
    rows = np.sort(np.random.default_rng(19).choice(reps.shape[0], size=2048, replace=False))
    x = _x(reps.shape[0], True, 53)
    expect = po.expected_rows(matrix, reps, x, rows)
    xd = _dev(torch, x)
    assert (op.info("canon_mode"), op.info("torus_mode")) == (1, 2)
    for canon in (1, 2):
        op.set_option("canon", canon)
        assert (op.info("canon_mode"), op.info("torus_mode")) == (1, 0), canon
        got = op.matvec(xd)[_dev(torch, rows)].cpu().numpy()
        assert op.info("rows_kernel") == 300, canon
        assert np.abs(got - expect).max() <= 1e-12 * np.abs(expect).max(), canon
    op.close()


# ---- 3. hash-table edges -----------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("table", sorted(TABLES))
def test_table_wrap_and_chains(torch_cuda, table):
    """The models of TABLE_MODELS on the table they were chosen for, at the bucket count the host restates: full
    vectors against the exact sums."""
    torch = torch_cuda
    kind, _, forced = table.partition("_")
    for spec in TABLE_MODELS[table]:
        basis, matrix = _ring(*spec)
        op = _op(matrix, mode=1, rows_index=0, rows_table_per_state=int(forced or 0), rows_batch_min=1)
        op.basis.build()
        reps = op.basis.representatives()
        n = reps.shape[0]
        ref = _ref(("ring",) + spec, matrix, reps)
        buckets = max(16, TABLES[table][0] * n)
        if kind == "batch":
            for cplx, k in ((False, 1), (False, 5), (True, 3)):
                X = np.stack([_x(n, cplx, 300 + j) for j in range(k)])
                Y = op.matvec_batch(_dev(torch, X)).cpu().numpy()
                assert op.info("rows_batch_kernel") == 200 and op.info("rows_kernel") == 0
                assert op.info("rows_batch_buckets") == buckets, (table, spec)
                for j in range(k):
                    ref.assert_close(Y[j], X[j], what=(table, spec, cplx, k, j))
        else:
            x = _x(n, kind == "c128", 61)
            for y in (op.matvec(_dev(torch, x)).cpu().numpy(), op.matvec(x)):
                assert op.info("rows_kernel") == 300
                assert op.info("rows_table_buckets") == buckets, (table, spec)
                ref.assert_close(y, x, what=(table, spec))
        op.close()


@gpu
def test_table_per_state_option(torch_cuda):
    """rows_table_per_state accepts 0 / 2 / 4 / 8 and nothing else; the products agree at every density."""
    torch = torch_cuda
    basis, matrix = _load("heisenberg_chain_24_symm")
    op = _op(matrix, mode=1)
    op.basis.build()
    reps = op.basis.representatives()
    ref = _ref("heisenberg_chain_24_symm", matrix, reps)
    x = _x(reps.shape[0], True, 67)
    ex = ref.exact(x)
    for v in (3, 1, 16, -1):
        with pytest.raises(Exception, match="rows_table_per_state"):
            op.set_option("rows_table_per_state", v)
    for v in (2, 4, 8, 0):
        op.set_option("rows_table_per_state", v)
        ref.assert_close(op.matvec(_dev(torch, x)).cpu().numpy(), x, ex, v)
        X = np.stack([x, 2 * x, -x])
        Y = op.matvec_batch(_dev(torch, X)).cpu().numpy()
        for j in range(3):
            ref.assert_close(Y[j], X[j], what=(v, j))
    op.close()


# ---- 4. missing states -----------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", ["heisenberg_chain_24_symm", "heisenberg_square_4x4"])
def test_missing_state_in_symmetric_kernels(torch_cuda, name):
    """A representative the product reaches with a nonzero coefficient, removed from the basis, is an error in each
    symmetric kernel; the same context then gives the right product on the whole basis (the status does not stick)."""
    torch = torch_cuda
    basis, matrix = _load(name)
    reps, norms = po.enumerate_states(basis)
    ref = _ref(name, matrix, reps)
    nz = ref.h[ref.bounds[0]:] != 0
    reached = np.unique(ref.rows[ref.bounds[0]:][nz & (ref.rows[ref.bounds[0]:] != ref.cols[ref.bounds[0]:])])
    drop = reached[np.linspace(0, reached.shape[0] - 1, 4).astype(int)]
    keep = np.ones(reps.shape[0], dtype=bool)
    keep[drop] = False
    x_full = _x(reps.shape[0], False, 71)
    ex = ref.exact(x_full)
    cases = [("k_rows", dict(mode=1, rows_index=0), 1), ("k_rows dense", dict(mode=1, rows_index=1), 1),
             ("k_rows_batch", dict(mode=1), 2), ("k_pull", dict(mode=1, rows=0), 1), ("k_generate", dict(mode=0), 1)]
    tk = ROWS_SMALL[name]
    expect_ran = {"k_rows": (1, 1, 300 + 10 * tk, 0), "k_rows dense": (1, 1, 200 + 10 * tk + 1, 0),
                  "k_rows_batch": (1, 1, 0, 200 + 10 * tk), "k_pull": (1, 0, 0, 0), "k_generate": (0, 0, 0, 0)}
    for what, options, k in cases:
        op = _op(matrix, **options)
        op.basis.uncheckedSetRepresentatives(reps[keep], norms[keep])
        x = x_full[keep]
        with pytest.raises(Exception, match="invalid index"):
            if k == 1:
                op.matvec(_dev(torch, x))
                op.synchronize()
            else:
                op.matvec_batch(_dev(torch, np.stack([x, -x])))
                op.synchronize()
        # the kernel that found the missing state is the one the case means
        ran = (op.info("pull"), op.info("rows"), op.info("rows_kernel"), op.info("rows_batch_kernel"))
        assert ran == expect_ran[what], (what, ran)
        op.basis.uncheckedSetRepresentatives(reps, norms)
        if k == 1:
            y = op.matvec(_dev(torch, x_full)).cpu().numpy()
            ref.assert_close(y, x_full, ex, what)
        else:
            Y = op.matvec_batch(_dev(torch, np.stack([x_full, x_full]))).cpu().numpy()
            ref.assert_close(Y[0], x_full, ex, what)
            ref.assert_close(Y[1], x_full, ex, what)
        op.close()


# ---- 5. shapes and layouts -------------------------------------------------------------------------------------------
def _edge_specs():
    out = []
    for n in (31, 32, 33, 63, 64):
        for hw in sorted({0, 1, 2, 3, n - 1, n}):
            for sym in ("", "T", "TM"):
                out.append((n, hw, sym))
    return out


@gpu
@pytest.mark.parametrize("spec", _edge_specs(), ids=lambda s: f"n{s[0]}_w{s[1]}_{s[2] or 'none'}")
def test_edge_bases(torch_cuda, spec):
    """Chains of 31 .. 64 sites at Hamming weights 0 .. 3 and n - 1, n, with and without translations (+ mirror):
    every product mode and index mode, f64 and c128, against the exact sums.  Includes the one state ~0 of 64 sites
    (equal to the empty key of the k_rows table) and bases of one state."""
    torch = torch_cuda
    n, hw, sym = spec
    basis, matrix = _ring(n, hw, sym, zz=0.75)
    reps, _ = po.enumerate_states(basis)
    ref = _ref(("ring",) + spec, matrix, reps)
    modes = {"auto": (-1, None), "push": (0, None), "pull": (1, None), "pull_queued": (1, 0)}
    for mode, (m, off) in modes.items():
        op = _op(matrix, mode=m)
        if off is not None:
            op.set_option("gather", 0)
            op.set_option("rows", 0)
        op.basis.build()
        assert np.array_equal(op.basis.representatives(), reps)
        for cplx in (False, True):
            x = _x(reps.shape[0], cplx, 73)
            ex = ref.exact(x)
            for index in (-1, 2, 0):
                op.set_option("index", index)
                ref.assert_close(op.matvec(x), x, ex, (mode, cplx, index, "host"))
                ref.assert_close(op.matvec(_dev(torch, x)).cpu().numpy(), x, ex, (mode, cplx, index, "device"))
        op.close()


@gpu
@pytest.mark.parametrize("spec", [(4, 2, ""), (6, 3, "TM"), (5, 1, "T"), (6, 2, ""), (8, 4, "TM"), (10, 3, "TM")],
                         ids=lambda s: f"n{s[0]}_w{s[1]}_{s[2] or 'none'}")
def test_empty_ranks(torch_cuda, spec):
    """Eight logical ranks on bases with fewer than eight states or with ranks that own none: the record exchange and
    the replicated form against the exact sums."""
    torch = torch_cuda
    from distributed_matvec_b200 import EmulatedCluster
    P = 8
    basis, matrix = _ring(*spec)
    reps, _ = po.enumerate_states(basis)
    masks = po.locale_idx_of(reps, P)
    assert np.bincount(masks, minlength=P).min() == 0
    ref = _ref(("ring",) + spec, matrix, reps)
    for cplx in (False, True):
        x = _x(reps.shape[0], cplx, 79)
        ex = ref.exact(x)
        cl = EmulatedCluster(matrix, P).build()
        xb = [_dev(torch, x[masks == r]) for r in range(P)]
        for form in ("records", "replicated"):
            yb = cl.matvec(xb) if form == "records" else cl.matvec_replicated(xb)
            y = np.zeros_like(x)
            for r in range(P):
                y[masks == r] = yb[r].cpu().numpy()
            ref.assert_close(y, x, ex, (form, cplx))
        cl.close()


@gpu
def test_row_chunked_rows_with_host_vectors(torch_cuda):
    """heisenberg_chain_32_symm (4.7 M states): the host-vector product cuts k_rows into row chunks and fills the table
    with the first one; it equals the device-vector product bit for bit.  The same for the host-staged batch."""
    torch = torch_cuda
    basis, matrix = _load("heisenberg_chain_32_symm")
    op = _op(matrix)
    op.basis.build()
    n = op.basis.numberStates()
    assert n >= 1 << 16 and op.info("rows") == 1
    for cplx in (False, True):
        x = _x(n, cplx, 83)
        yd = op.matvec(_dev(torch, x)).cpu().numpy()
        yh = op.matvec(x)
        assert np.array_equal(yh, yd), cplx
        X = np.stack([_x(n, cplx, 90 + j) for j in range(3)])
        Yd = op.matvec_batch(_dev(torch, X)).cpu().numpy()
        Yh = op.matvec_batch(X)
        assert np.array_equal(Yh, Yd), cplx
    op.close()


@gpu
@pytest.mark.parametrize("spec", [(4, 0, ""), (2, 1, ""), (3, 1, ""), (4, 1, "TM"), (6, 2, "TM")],
                         ids=lambda s: f"n{s[0]}_w{s[1]}_{s[2] or 'none'}")
def test_lanczos_tiny_bases(torch_cuda, spec):
    """Lanczos on bases of 1, 2 and 3 states: the exact lowest eigenvalue (k = 1 tridiagonal, stop at n_global)."""
    basis, matrix = _ring(*spec, zz=0.6)
    reps, _ = po.enumerate_states(basis)
    assert 1 <= reps.shape[0] <= 3
    n = reps.shape[0]
    H = np.zeros((n, n))
    for j in range(n):
        e = np.zeros(n)
        e[j] = 1.0
        H[:, j] = po.matvec_global(matrix, reps, e, 1)
    want = np.linalg.eigvalsh((H + H.T) / 2)[0]
    op = _op(matrix)
    op.basis.build()
    for cplx in (False, True):
        e0, vec, iters, res = op.lanczos(max_iters=50, tol=1e-12, complex_vectors=cplx)
        assert abs(e0 - want) <= 1e-12 * max(1.0, abs(want)), (spec, cplx, e0, want)
        assert 1 <= iters <= n
        assert abs(np.linalg.norm(vec) - 1.0) < 1e-12
    op.close()
