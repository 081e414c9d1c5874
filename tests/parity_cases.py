"""Parity checks shared by the emulator tests (CPU, small sizes) and the GPU tests (C ABI on a B200)."""
import numpy as np

import bn254 as o


def omega_words(oc, k, inverse=False):
    w = o.omega_for(k)
    if inverse:
        w = pow(w, -1, o.R_MOD)
    return oc.ints_to_words([o.to_mont(w, o.R_MOD)])[0]


def affine_of(oc, jac):
    return oc.g1_to_affine(np.ascontiguousarray(jac, dtype=np.uint64))


def check_field(L, oc, n=2048):
    a, b = oc.random_fr(1, n), oc.random_fr(2, n)
    a[0] = 0
    b[1] = 0
    a[2] = b[2]
    for f in ("fr", "fq"):
        for op in ("add", "sub", "mul"):
            assert (L.field_op(f, op, a, b) == oc.field_op(f, op, a, b)).all(), (f, op)
        assert (L.field_op(f, "sqr", a) == oc.field_op(f, "mul", a, a)).all(), (f, "sqr")
    assert (L.field_op("fr", "from_mont", a) == oc.fr_from_mont(a)).all()
    assert (L.field_op("fr", "to_mont", a) == oc.fr_to_mont(a)).all()
    m = min(n, 64)
    inv = L.field_op("fq", "inv", a[3:m])
    one = L.field_op("fq", "mul", inv, a[3:m])
    R1 = oc.ints_to_words([(1 << 256) % o.P_MOD])[0]
    assert (one == R1).all()


def check_group(L, oc, n=64):
    def aff(w):
        v = oc.words_to_ints(np.ascontiguousarray(w).reshape(-1, 4))
        return [None if (v[2 * i] == 0 and v[2 * i + 1] == 0) else (o.from_mont(v[2 * i], o.P_MOD), o.from_mont(v[2 * i + 1], o.P_MOD))
                for i in range(len(v) // 2)]
    P, Q = oc.gen_points(7, n), oc.gen_points(9, n)
    Q[5] = P[5]          # doubling branch
    Q[6] = 0             # identity operands
    P[7] = 0
    Q[8, :4] = P[8, :4]  # q = -p
    Q[8, 4:] = oc.field_op("fq", "sub", np.zeros((1, 4), dtype=np.uint64), P[8:9, 4:])[0]
    pa, qa = aff(P), aff(Q)
    r = [aff(L.ec_op(op, P, Q)) for op in range(4)]
    for i in range(n):
        s = o.g1_add(pa[i], qa[i])
        assert r[0][i] == s, (i, "add")
        assert r[3][i] == s, (i, "jacobian")
        assert r[1][i] == o.g1_add(pa[i], o.g1_neg(qa[i])), (i, "sub")
        assert r[2][i] == (o.g1_mul(s, 4) if s else None), (i, "x4")


def check_ntt(L, oc, k, seed=0):
    a = oc.random_fr(0xA000 + 97 * k + seed, 1 << k)
    for inverse in (False, True):
        w = omega_words(oc, k, inverse)
        got = L.ntt(a.copy(), w, k)
        want = oc.best_fft(a, w, k)
        assert (got == want).all(), "NTT mismatch at k=%d inverse=%s" % (k, inverse)


def check_fr_transpose(L, oc, shapes=((32, 32), (64, 96), (256, 32), (1, 5), (33, 70), (96, 1), (1024, 512))):
    """h2b_fr_transpose_dev against numpy: whole 32 x 32 tiles (the TMA bulk-copy kernel on the GPU) and ragged shapes"""
    for rows, cols in shapes:
        a = oc.random_fr(0x7A00 + rows * 131 + cols, rows * cols).reshape(rows, cols, 4)
        got = L.fr_transpose(a)
        assert got.shape == (cols, rows, 4) and (got == a.transpose(1, 0, 2)).all(), "transpose mismatch %dx%d" % (rows, cols)


def edge_msm_inputs(L, oc, n, kind, seed):
    s = L.gen_scalars(seed, n, kind)
    P = oc.gen_points(seed + 1, n) if n <= (1 << 16) else L.gen_points(seed + 1, n)
    if n > 40:
        s[1] = 0
        P[3] = 0
        P[5] = P[4]
        s[5] = s[4]
        P[9] = P[8]
    return s, P


def check_msm(L, oc, n, kind=0, windows=(0,), seed=1):
    s, P = edge_msm_inputs(L, oc, n, kind, seed + n)
    want = affine_of(oc, oc.best_multiexp(s, P))
    for cw in windows:
        L.set_msm_window(cw)
        try:
            got = affine_of(oc, L.msm(s, P))
        finally:
            L.set_msm_window(0)
        assert (got == want).all(), "MSM mismatch n=%d kind=%d window=%d" % (n, kind, cw)


def check_msm_tables(L, oc, n, spacing, kind=0, seed=5, windows=(0,), ranges=None):
    """Registered base set with precomputed window tables: full range and sub-ranges, forced table spacing."""
    s, P = edge_msm_inputs(L, oc, n, kind, seed + n)
    L.set_msm_precomp(spacing)
    try:
        h = L.register_bases(P)
    finally:
        L.set_msm_precomp(0)
    try:
        info = L.base_set_info(h)
        assert info["n_tables"] > 1 and info["spacing"] == (spacing or info["spacing"]), info
        for (off, m) in (ranges or [(0, n)]):
            want = affine_of(oc, oc.best_multiexp(s[off:off + m], P[off:off + m]))
            for cw in windows:
                L.set_msm_window(cw)
                try:
                    got = affine_of(oc, L.msm_registered(s[off:off + m], h, off))
                finally:
                    L.set_msm_window(0)
                assert (got == want).all(), "table MSM mismatch n=%d range=(%d,%d) spacing=%d window=%d" % (n, off, m, spacing, cw)
    finally:
        L.unregister_bases(h)


def check_msm_single_bucket(L, oc, n, scalar=1, tables=True):
    """Every scalar equal: the whole sorted list is one bucket, cut into many slices (multi-chunk tree combine)."""
    P = oc.gen_points(901, n) if n <= (1 << 16) else L.gen_points(901, n)
    one = oc.fr_to_mont(np.array([[scalar, 0, 0, 0]], dtype=np.uint64))
    s = np.repeat(one, n, axis=0)
    want = affine_of(oc, oc.best_multiexp(s, P))
    if tables:
        h = L.register_bases(P)
        try:
            got = affine_of(oc, L.msm_registered(s, h))
        finally:
            L.unregister_bases(h)
    else:
        got = affine_of(oc, L.msm(s, P))
    assert (got == want).all()


def check_msm_random(L, oc, examples, max_n, spacings, windows):
    """Property test over the MSM's shape space: random length, scalar mix (incl. 0, 1, r-1, duplicates, identity bases),
    table spacing / plain mode (-1), forced window, sub-range of a registered set -- always the oracle's affine result."""
    from hypothesis import given, settings, strategies as st, HealthCheck

    one = oc.fr_to_mont(np.array([[1, 0, 0, 0]], dtype=np.uint64))[0]
    minus_one = oc.field_op("fr", "sub", np.zeros((1, 4), dtype=np.uint64), one.reshape(1, 4))[0]

    @settings(max_examples=examples, deadline=None, suppress_health_check=list(HealthCheck), derandomize=True)
    @given(n=st.integers(1, max_n), seed=st.integers(0, 10 ** 6), spacing=st.sampled_from(list(spacings)),
           window=st.sampled_from(list(windows)), kind=st.integers(0, 1), off_frac=st.floats(0, 0.9))
    def run(n, seed, spacing, window, kind, off_frac):
        s = L.gen_scalars(seed, n, kind)
        P = oc.gen_points(seed + 1, n)
        rng = np.random.default_rng(seed)
        for i in rng.integers(0, n, size=min(n, 6)):
            choice = rng.integers(0, 5)
            if choice == 0:
                s[i] = 0
            elif choice == 1:
                s[i] = one
            elif choice == 2:
                s[i] = minus_one
            elif choice == 3:
                P[i] = 0
            else:
                P[i] = P[rng.integers(0, n)]
        if spacing < 0:
            L.set_msm_window(window)
            try:
                got = affine_of(oc, L.msm(s, P))
            finally:
                L.set_msm_window(0)
            want = affine_of(oc, oc.best_multiexp(s, P))
        else:
            off = int(off_frac * n)
            m = n - off
            L.set_msm_precomp(spacing)
            try:
                h = L.register_bases(P)
            finally:
                L.set_msm_precomp(0)
            try:
                L.set_msm_window(window)
                got = affine_of(oc, L.msm_registered(s[:m], h, off))
            finally:
                L.set_msm_window(0)
                L.unregister_bases(h)
            want = affine_of(oc, oc.best_multiexp(s[:m], P[off:off + m]))
        assert (got == want).all(), (n, seed, spacing, window, kind, off_frac)

    run()


def check_grand_product_blocks(L, oc, sizes):
    """batch inversion (zeros stay zero) and exclusive prefix product against the oracle, ragged sizes"""
    for n in sizes:
        a = oc.random_fr(0xD000 + n, n)
        if n > 3:
            a[1] = 0
            a[n - 1] = 0
            a[n // 2] = a[n // 2 - 1]
        assert (L.fr_batch_invert(a) == oc.fr_batch_invert(a)).all(), ("batch_invert", n)
        assert (L.fr_prefix_product(a) == oc.fr_prefix_product(a)).all(), ("prefix_product", n)
        if n > 8:
            b = a.copy()
            b[b.sum(axis=1) == 0] = a[0]                                   # no zeros: the product never collapses
            assert (L.fr_prefix_product(b) == oc.fr_prefix_product(b)).all(), ("prefix_product nz", n)


def check_poly_eval_and_division(L, oc, sizes):
    """eval_polynomial and kate_division against the oracle, plus the identity a(X) = q(X) (X - b) + a(b) at a random point"""
    for n in sizes:
        a = oc.random_fr(0xE000 + n, n)
        x, b = oc.random_fr(0xE100 + n, 1)[0], oc.random_fr(0xE200 + n, 1)[0]
        assert (L.fr_eval_polynomial(a, x) == oc.fr_eval_polynomial(a, x)).all(), ("eval", n)
        q = L.fr_kate_division(a, b)
        assert (q == oc.fr_kate_division(a, b)).all(), ("kate", n)
        if n > 1:
            # a(x) == q(x) * (x - b) + a(b), all through the device evaluation
            ax, qx, ab = L.fr_eval_polynomial(a, x), L.fr_eval_polynomial(q, x), L.fr_eval_polynomial(a, b)
            xmb = oc.field_op("fr", "sub", x.reshape(1, 4), b.reshape(1, 4))
            rhs = oc.field_op("fr", "add", oc.field_op("fr", "mul", qx.reshape(1, 4), xmb), ab.reshape(1, 4))
            assert (rhs[0] == ax).all(), ("identity", n)


def check_golden_ntt(L, g):
    for k in (1, 2, 3, 5, 8):
        for tag, wkey in (("fwd", "omega"), ("inv", "omega_inv")):
            a = np.array(g["k%d_in" % k], dtype=np.uint64, order="C")
            got = L.ntt(a, g["k%d_%s" % (k, wkey)], k)
            assert (got == g["k%d_%s" % (k, tag)]).all(), (k, tag)


def check_msm_opposite_points(L, oc, n, kind):
    """A duplicate point, an identity base, and P and -P with equal scalars (one bucket, the pair cancels), through a registered
    base set and the plain call."""
    s, P = L.gen_scalars(n, n, kind), oc.gen_points(n + 1, n)
    P[5] = P[4]
    P[7] = 0
    P[9, :4] = P[8, :4]
    P[9, 4:] = oc.field_op("fq", "sub", np.zeros((1, 4), dtype=np.uint64), P[8:9, 4:])[0]
    s[9] = s[8]
    want = affine_of(oc, oc.best_multiexp(s, P))
    h = L.register_bases(P)
    try:
        assert (affine_of(oc, L.msm_registered(s, h, 0)) == want).all(), (n, kind)
    finally:
        L.unregister_bases(h)
    assert (affine_of(oc, L.msm(s, P)) == want).all(), (n, kind, "plain")


def check_golden_msm(L, oc, g):
    for tag in ("n1", "n2", "n8", "n64", "n200", "cancel", "anchor"):
        got = affine_of(oc, L.msm(g[tag + "_scalars"], g[tag + "_bases"]))
        assert (got == g[tag + "_result"]).all(), tag


# ---- quotient evaluation (evaluate_h) ---------------------------------------------------------------------------------
def random_graph(rng, n_fixed, n_advice, n_instance, n_challenges, n_calcs, n_rot=4, reuse_targets=False):
    """A random GraphEvaluator in upstream's vocabulary: every Calculation / ValueSource variant, Horner with 0..6 parts,
    dead calculations, Stores of columns / constants / intermediates.  -> (constants, rotations, calcs, parts, n_intermediates)"""
    n_const = 3 + int(rng.integers(0, 4))
    rotations = [0] + [int(v) for v in rng.integers(-3, 4, size=n_rot - 1)]
    calcs, parts, defined = [], [], []
    n_inter = n_calcs if not reuse_targets else max(2, n_calcs // 3)

    def source():
        kinds = [0, 5, 6, 7, 8, 9, 10] if n_challenges else [0, 6, 7, 8, 9, 10]
        kinds += [2] * (2 if n_fixed else 0) + [3] * (4 if n_advice else 0) + [4] * (1 if n_instance else 0)
        kinds += [1] * (14 if defined else 0)
        k = int(rng.choice(kinds))
        if k == 0:
            return (0, int(rng.integers(0, n_const)), 0)
        if k == 1:
            # mostly recent values (chains), sometimes an old one (long live ranges)
            return (1, defined[-1 - int(rng.integers(0, min(3, len(defined))))] if rng.random() < 0.7 else int(rng.choice(defined)), 0)
        if k in (2, 3, 4):
            return (k, int(rng.integers(0, {2: n_fixed, 3: n_advice, 4: n_instance}[k])), int(rng.integers(0, len(rotations))))
        if k == 5:
            return (5, int(rng.integers(0, n_challenges)), 0)
        return (k, 0, 0)

    for c in range(n_calcs):
        op = int(rng.choice([0, 1, 2, 2, 2, 3, 4, 5, 6, 6, 7]))
        a, b = source(), source()
        po, pl = 0, 0
        if op == 6:
            pl = int(rng.integers(0, 7))
            po = len(parts)
            parts.extend(source() for _ in range(pl))
        target = c if not reuse_targets else int(rng.integers(0, n_inter))
        calcs.append([op, target, *a, *b, po, pl])
        if target not in defined:
            defined.append(target)
    # the result: a Horner in y over a sample of what was defined, so that most of the program is reachable
    pl = min(len(defined), 24)
    po = len(parts)
    parts.extend((1, int(t), 0) for t in rng.choice(defined, size=pl, replace=False))
    calcs.append([6, defined[-1] if reuse_targets else n_calcs, 10, 0, 0, 9, 0, 0, po, pl])
    if not reuse_targets:
        n_inter += 1
    return (None, np.array(rotations, dtype=np.int32), np.array(calcs, dtype=np.uint32).reshape(-1, 10),
            np.array(parts, dtype=np.uint32).reshape(-1, 3), n_inter), n_const


def wide_graph(n_live):
    """n_live products that all stay live: each is consumed once by a running sum and once more by a running product"""
    calcs = [[2, i, 3, 0, 0, 0, 3 + (i % 3), 0, 0, 0] for i in range(n_live)]                  # v_i = advice0 * constant
    t = n_live
    calcs.append([0, t, 1, 0, 0, 1, 1, 0, 0, 0])                                              # s = v_0 + v_1
    for i in range(2, n_live):
        calcs.append([0, t + 1, 1, t, 0, 1, i, 0, 0, 0])
        t += 1
    for i in range(n_live):
        calcs.append([2 if i % 2 else 1, t + 1, 1, t, 0, 1, i, 0, 0, 0])                      # s = s (* or -) v_i
        t += 1
    return (None, np.array([0], dtype=np.int32), np.array(calcs, dtype=np.uint32), np.zeros((0, 3), dtype=np.uint32), t + 1), 6


def _graph_pair(oc, graph, n_const, seed):
    """(oracle tuple, product GraphArrays) of one random graph with random constants"""
    from halo2_scaffold_b200._lib import GraphArrays
    constants = oc.random_fr(seed, n_const)
    constants[0] = 0
    g = (constants,) + graph[1:]
    return g, GraphArrays(*g)


def check_evaluate_graph(L, oc, cases):
    """h2b_evaluate_graph_dev against the sequential walk of the oracle on random graphs.  cases: (size, rot_scale, n_calcs, seed)"""
    from halo2_scaffold_b200 import evaluation as ev
    for size, rot_scale, n_calcs, seed in cases:
        rng = np.random.default_rng(seed)
        nf, na, ni, nch = int(rng.integers(0, 3)), int(rng.integers(1, 5)), int(rng.integers(0, 2)), int(rng.integers(0, 3))
        graph, n_const = random_graph(rng, nf, na, ni, nch, n_calcs, reuse_targets=bool(seed % 3 == 2))
        g, ga = _graph_pair(oc, graph, n_const, seed)
        cols = [oc.random_fr(seed * 131 + j, size) for j in range(nf + na + ni)]
        fixed, advice, instance = cols[:nf], cols[nf:nf + na], cols[nf + na:]
        sc = oc.random_fr(seed * 7 + 1, nch + 4)
        challenges, (beta, gamma, theta, y) = sc[:nch], sc[nch:]
        values = oc.random_fr(seed * 7 + 2, size)
        want = oc.evaluate_graph(g, fixed, advice, instance, challenges, beta, gamma, theta, y, values, rot_scale)
        got = ev.evaluate_graph(L, ga, fixed, advice, instance, challenges, beta, gamma, theta, y, values, rot_scale)
        assert (got == want).all(), ("evaluate_graph", size, rot_scale, n_calcs, seed, L.evaluate_graph_info())


def standard_plonk_like(n_advice_groups=1):
    """gate polynomials in the shape of examples/standard_plonk.rs (q_a a + q_b b + q_c c + q_ab a b + constant + instance = 0),
    one per advice triple, plus a rotated term and a lookup argument over the first advice column"""
    from halo2_scaffold_b200 import evaluation as ev
    polys, f = [], 0
    for gidx in range(n_advice_groups):
        a, b, c = ev.Advice(3 * gidx), ev.Advice(3 * gidx + 1), ev.Advice(3 * gidx + 2)
        q_a, q_b, q_c, q_ab, const = (ev.Fixed(f + j) for j in range(5))
        f += 5
        poly = ev.Sum(ev.Sum(ev.Sum(ev.Sum(ev.Sum(ev.Product(q_a, a), ev.Product(q_b, b)), ev.Product(q_c, c)),
                                    ev.Product(q_ab, ev.Product(a, b))), const), ev.Instance(0))
        polys.append(poly)
        # a * (a[next] - b) - 3 * c[prev] : rotations, Negated, Scaled
        polys.append(ev.Sum(ev.Product(a, ev.Sum(ev.Advice(3 * gidx, 1), ev.Negated(b))), ev.Negated(ev.Scaled(ev.Advice(3 * gidx + 2, -1), 3))))
    lookups = [([ev.Product(ev.Fixed(0), ev.Advice(0)), ev.Advice(1, 1)], [ev.Fixed(1), ev.Fixed(2)])]
    return polys, lookups, f, 3 * n_advice_groups


def check_evaluate_h(L, oc, cases):
    """Evaluator::evaluate_h (custom gates, permutations, lookups) through the host mirror against the oracle's three loops.
    cases: (extended_k, k, groups, seed)"""
    from halo2_scaffold_b200 import evaluation as ev
    from halo2_scaffold_b200.domain import fr_to_words
    for ek, k, groups, seed in cases:
        size, rot_scale = 1 << ek, 1 << (ek - k)
        polys, lookup_exprs, nf, na = standard_plonk_like(groups)
        E = ev.Evaluator(polys, lookup_exprs)
        fixed = [oc.random_fr(seed * 1000 + j, size) for j in range(nf)]
        advice = [oc.random_fr(seed * 1000 + 100 + j, size) for j in range(na)]
        instance = [oc.random_fr(seed * 1000 + 200, size)]
        sc = oc.random_fr(seed * 1000 + 300, 8)
        beta, gamma, theta, y, delta, zeta, extended_omega = sc[:7]
        extended_omega = fr_to_words(o.omega_for(ek))
        l0, l_last, l_active = (oc.random_fr(seed * 1000 + 400 + j, size) for j in range(3))
        # permutation over all advice columns + one fixed column, chunk_len 2 (degree 4): ceil(n_cols / 2) sets
        perm_cols = [("advice", j) for j in range(na)] + [("fixed", 0)]
        chunk_len = 2
        n_sets = (len(perm_cols) + chunk_len - 1) // chunk_len
        perm = dict(product_cosets=[oc.random_fr(seed * 1000 + 500 + j, size) for j in range(n_sets)], columns=perm_cols,
                    cosets=[oc.random_fr(seed * 1000 + 600 + j, size) for j in range(len(perm_cols))], chunk_len=chunk_len, last_rotation=-6,
                    delta=delta, zeta=zeta, extended_omega=extended_omega)
        lks = [dict(product_coset=oc.random_fr(seed * 1000 + 700, size), permuted_input_coset=oc.random_fr(seed * 1000 + 701, size),
                    permuted_table_coset=oc.random_fr(seed * 1000 + 702, size))]
        got = E.evaluate_h(size=size, rot_scale=rot_scale, fixed=fixed, advice=advice, instance=instance, challenges=np.zeros((0, 4), dtype=np.uint64),
                           y=y, beta=beta, gamma=gamma, theta=theta, l0=l0, l_last=l_last, l_active_row=l_active, permutation=perm, lookups=lks, lib=L)

        def tup(g):
            a = g.arrays()
            return (a.constants, a.rotations, a.calculations, a.parts, a.n_intermediates)
        ch = np.zeros((0, 4), dtype=np.uint64)
        want = oc.evaluate_graph(tup(E.custom_gates), fixed, advice, instance, ch, beta, gamma, theta, y, np.zeros((size, 4), dtype=np.uint64), rot_scale)
        by_type = {"advice": advice, "fixed": fixed, "instance": instance}
        want = oc.evaluate_h_permutation(want, rot_scale, perm["product_cosets"], [by_type[t][i] for t, i in perm_cols], perm["cosets"], chunk_len, -6,
                                         l0, l_last, l_active, beta, gamma, y, delta, zeta, extended_omega)
        want = oc.evaluate_h_lookup(tup(E.lookups[0]), fixed, advice, instance, ch, beta, gamma, theta, y, want, rot_scale, lks[0]["product_coset"],
                                    lks[0]["permuted_input_coset"], lks[0]["permuted_table_coset"], l0, l_last, l_active)
        assert (got == want).all(), ("evaluate_h", ek, k, groups, seed)


# ---- SRS on-disk format ----------------------------------------------------------------------------------------------------
def check_g1_codec(L, oc, n, seed=5):
    """G1Affine::{to_bytes, from_bytes} and the raw formats against the oracle, identity and invalid encodings included"""
    from halo2_scaffold_b200._lib import H2BError
    P = oc.gen_points(seed, n)
    if n > 3:
        P[2] = 0                                                   # the identity
    want_bytes = oc.g1_to_bytes(P)
    assert (L.g1_encode(P) == want_bytes).all()
    assert (L.g1_decode(want_bytes, 0) == P).all()
    dec, first = oc.g1_from_bytes(want_bytes)
    assert first == n and (dec == P).all()
    raw = P.view(np.uint8).reshape(n, 64)
    assert (L.g1_decode(raw, 1) == P).all() and (L.g1_decode(raw, 2) == P).all()
    if n > 8:
        # x with no square root of x^3 + 3, a non-canonical x, and a raw point off the curve -> refused at the right index
        bad = want_bytes.copy()
        x = 4
        while pow(x ** 3 + 3, (o.P_MOD - 1) // 2, o.P_MOD) == 1:
            x += 1
        bad[5] = np.frombuffer(x.to_bytes(32, "little"), dtype=np.uint8)
        bad[7] = np.frombuffer((o.P_MOD + 1).to_bytes(32, "little"), dtype=np.uint8)
        assert oc.g1_from_bytes(bad)[1] == 5
        try:
            L.g1_decode(bad, 0)
            raise AssertionError("invalid encoding accepted")
        except H2BError as e:
            assert "point 5" in str(e)
        off = raw.copy()
        off[6, 0] ^= 1
        try:
            L.g1_decode(off, 1)
            raise AssertionError("off-curve point accepted")
        except H2BError as e:
            assert "point 6" in str(e)
        assert (L.g1_decode(off, 2).view(np.uint8).reshape(n, 64) == off).all()         # unchecked: taken as is


def check_srs_file_round_trip(L, oc, tmp_path, k, seed=3):
    """ParamsKZG::write_custom -> read_custom in all three formats: same points, resident base sets that commit correctly;
    and the file bytes equal the big-int writer's (oracle/bn254.py) for small k"""
    import halo2_scaffold_b200 as h2
    from halo2_scaffold_b200.kzg import SerdeFormat
    n = 1 << k
    g, gl = oc.gen_points(seed, n), oc.gen_points(seed + 1, n)
    g2 = bytes(range(256))
    params = h2.ParamsKZG(k, g, gl, lib=L, g2_bytes=g2)
    scalars = oc.random_fr(seed + 2, n)
    want_c, want_l = affine_of(oc, oc.best_multiexp(scalars, g)), affine_of(oc, oc.best_multiexp(scalars, gl))
    for fmt in (SerdeFormat.Processed, SerdeFormat.RawBytes, SerdeFormat.RawBytesUnchecked):
        path = str(tmp_path / ("kzg_bn254_%d_%d.srs" % (k, fmt)))
        g2f = g2[:128] if fmt == SerdeFormat.Processed else g2
        params.g2_bytes = g2f
        params.write_custom(path, fmt)
        if k <= 6:
            def pts(w):
                v = oc.words_to_ints(np.ascontiguousarray(w).reshape(-1, 4))
                return [None if (v[2 * i] == 0 and v[2 * i + 1] == 0) else (o.from_mont(v[2 * i], o.P_MOD), o.from_mont(v[2 * i + 1], o.P_MOD))
                        for i in range(len(v) // 2)]
            ref = str(tmp_path / "ref.srs")
            o.srs_write(ref, k, pts(g), pts(gl), g2f, fmt)
            assert open(ref, "rb").read() == open(path, "rb").read(), fmt
            kk, rg, rgl, rg2 = o.srs_read(path, fmt)
            assert kk == k and rg == pts(g) and rgl == pts(gl) and rg2 == g2f
        back = h2.ParamsKZG.read_custom(path, fmt, lib=L)
        try:
            assert back.k == k and (back.g == g).all() and (back.g_lagrange == gl).all() and back.g2_bytes == g2f
            assert (affine_of(oc, back.commit(scalars)) == want_c).all(), fmt
            assert (affine_of(oc, back.commit_lagrange(scalars)) == want_l).all(), fmt
        finally:
            back.close()
    params.close()


def check_vanishing_division(L, oc, cases):
    """EvaluationDomain::divide_by_vanishing_poly through the mirror: against the big-int domain, and the identity
    h = q * (X^n - 1)  =>  extended_to_coeff(divide_by_vanishing_poly(coset evaluations of h)) = q.   cases: (j, k)"""
    import halo2_scaffold_b200 as h2
    for j, k in cases:
        dom, ref = h2.EvaluationDomain(j, k, lib=L), o.EvaluationDomain(j, k)
        n, en = 1 << k, 1 << ref.extended_k
        assert len(dom.t_evaluations) == 1 << (ref.extended_k - k) and dom.t_evaluations == ref.t_evaluations
        a = oc.random_fr(0xF000 + 16 * j + k, en)
        ai = [o.from_mont(v, o.R_MOD) for v in oc.words_to_ints(a)]
        want = oc.ints_to_words([o.to_mont(v, o.R_MOD) for v in ref.divide_by_vanishing_poly(ai)])
        assert (dom.divide_by_vanishing_poly(a) == want).all(), (j, k)
        # q of degree < n (j - 2); h = q X^n - q has n (j - 1) coefficients
        qn = n * (j - 2)
        q = [o.from_mont(v, o.R_MOD) for v in oc.words_to_ints(oc.random_fr(0xF100 + 16 * j + k, qn))]
        h = [0] * (n * (j - 1))
        for i, c in enumerate(q):
            h[i] = (h[i] - c) % o.R_MOD
            h[i + n] = (h[i + n] + c) % o.R_MOD
        z = [1, ref.g_coset, ref.g_coset_inv]
        hz = [c * z[i % 3] % o.R_MOD for i, c in enumerate(h)] + [0] * (en - len(h))
        h_ext = oc.ints_to_words([o.to_mont(v, o.R_MOD) for v in o.best_fft(hz, ref.extended_omega, ref.extended_k)])
        back = dom.extended_to_coeff(dom.divide_by_vanishing_poly(h_ext))
        want_q = oc.ints_to_words([o.to_mont(v, o.R_MOD) for v in q + [0] * (n * (j - 1) - qn)])
        assert (back == want_q).all(), ("quotient identity", j, k)


def check_grand_products(L, oc, sizes):
    """permutation::Argument::commit (per set, chained through last_z and delta^j) and lookup commit_product against the oracle;
    plus the argument's own telescoping property: with sigma = identity permutation (s_j = delta^j omega^i) every factor is 1"""
    from halo2_scaffold_b200.domain import fr_to_words
    DELTA = pow(7, 1 << 28, o.R_MOD)                  # Fr::DELTA = GENERATOR^(2^S)
    for n in sizes:
        k = max(1, (n - 1).bit_length())
        omega = fr_to_words(o.omega_for(k))
        sc = oc.random_fr(0x9000 + n, 3)
        beta, gamma, last_z = sc
        one = fr_to_words(1)
        for m, first_col in ((1, 0), (3, 0), (2, 3), (16, 5), (17, 0), (37, 2)):      # more than 16 columns: several launches per set
            vals = [oc.random_fr(0x9100 + 17 * n + j, n) for j in range(m)]
            sig = [oc.random_fr(0x9200 + 17 * n + j, n) for j in range(m)]
            dw = fr_to_words(pow(DELTA, first_col, o.R_MOD))
            lz = one if first_col == 0 else last_z
            want = oc.permutation_product(vals, sig, beta, gamma, fr_to_words(DELTA), dw, omega, lz)
            got = L.permutation_product(vals, sig, beta, gamma, fr_to_words(DELTA), dw, omega, lz)
            assert (got == want).all(), ("permutation_product", n, m, first_col)
        # identity permutation: sigma_j[i] = delta^j omega^i  =>  z stays at last_z on every row
        m = 3
        vals = [oc.random_fr(0x9300 + n + j, n) for j in range(m)]
        w = o.omega_for(k)
        sig = [oc.ints_to_words([o.to_mont(pow(DELTA, j, o.R_MOD) * pow(w, i, o.R_MOD) % o.R_MOD, o.R_MOD) for i in range(n)]) for j in range(m)]
        got = L.permutation_product(vals, sig, beta, gamma, fr_to_words(DELTA), one, omega, last_z)
        assert (got == last_z).all(), ("identity permutation", n)
        cols = [oc.random_fr(0x9400 + 5 * n + j, n) for j in range(4)]
        assert (L.lookup_product(*cols, beta, gamma) == oc.lookup_product(*cols, beta, gamma)).all(), ("lookup_product", n)
        # a' = a and s' = s: the product telescopes to one
        assert (L.lookup_product(cols[0], cols[1], cols[0], cols[1], beta, gamma) == one).all(), ("lookup identity", n)


def check_lincomb(L, oc, cases):
    """sum_j c_j * col_j against field operations of the oracle.  cases: (n, m)"""
    for n, m in cases:
        cols = [oc.random_fr(0xA100 + 3 * n + j, n) for j in range(m)]
        coeffs = oc.random_fr(0xA200 + n + m, m)
        if m > 2:
            coeffs[1] = 0
        want = np.zeros((n, 4), dtype=np.uint64)
        for j in range(m):
            want = oc.field_op("fr", "add", want, oc.field_op("fr", "mul", cols[j], np.repeat(coeffs[j:j + 1], n, axis=0)))
        assert (L.fr_lincomb(cols, coeffs) == want).all(), (n, m)


def check_lookup_permute(L, oc, cases):
    """permute_expression_pair against the oracle's restatement (sort + BTreeMap walk), and the argument's invariants: A' is a
    sorted permutation of A, S' a permutation of S, and every row has A'[r] == S'[r] or A'[r] == A'[r-1].
    cases: (n, usable_rows, table_size, kind)"""
    from halo2_scaffold_b200._lib import H2BError
    for n, usable, table_size, kind, seed in cases:
        rng = np.random.default_rng(seed)
        pool = oc.random_fr(0xC000 + seed, table_size)             # distinct table values (random 254-bit: full-width keys)
        if kind == "small":                                        # a range table 0 .. table_size - 1, as halo2-lib's lookup table
            pool = oc.fr_to_mont(np.array([[v, 0, 0, 0] for v in range(table_size)], dtype=np.uint64))
        # the table column: every pool value at least once (while rows last), the rest repeats; the input draws from the pool
        t_idx = np.concatenate([np.arange(min(table_size, n)), rng.integers(0, table_size, size=max(0, n - table_size))])
        rng.shuffle(t_idx)
        table = pool[t_idx]
        present = np.unique(t_idx[:usable])
        a_idx = present[rng.integers(0, len(present), size=n)] if usable else np.zeros(n, dtype=np.int64)
        if kind == "skewed" and usable:
            a_idx[: (3 * n) // 4] = present[0]                      # one value on most rows
        inp = pool[a_idx]
        want_a, want_t = oc.lookup_permute(inp, table, usable)
        got_a, got_t = L.lookup_permute(inp, table, usable)
        assert (got_a == want_a).all(), ("permuted input", n, usable, kind)
        assert (got_t == want_t).all(), ("permuted table", n, usable, kind)
        if usable:
            key = lambda w: sorted(map(tuple, w.tolist()))
            assert key(got_a) == key(inp[:usable]) and key(got_t) == key(table[:usable])
            same_as_table = (got_a == got_t).all(axis=1)
            same_as_prev = np.concatenate([[False], (got_a[1:] == got_a[:-1]).all(axis=1)])
            assert (same_as_table | same_as_prev).all()
        # an input value outside the table is refused
        if usable > 2 and kind != "small":
            bad = inp.copy()
            bad[1] = oc.random_fr(0xDEAD + seed, 1)[0]
            try:
                L.lookup_permute(bad, table, usable)
                raise AssertionError("missing table value accepted")
            except H2BError as e:
                assert "ConstraintSystemFailure" in str(e)


def check_golden_prover_oracle(oc, g):
    """the C++ restatements reproduce the big-int fixture of the widened rows (tests/golden/prover_golden.npz)"""
    c, sc = g["graph_cols"], g["graph_scalars"]
    graph = (g["graph_constants"], g["graph_rotations"], g["graph_calcs"], g["graph_parts"], 10)
    assert (oc.evaluate_graph(graph, c[:1], c[1:4], c[4:], sc[:1], sc[1], sc[2], sc[3], sc[4], g["graph_prev"], 2) == g["graph_out"]).all()
    ps = g["perm_scalars"]
    assert (oc.permutation_product(list(g["perm_values"]), list(g["perm_sigma"]), ps[0], ps[1], ps[2], ps[3], ps[4], ps[5]) == g["perm_z"]).all()
    lk = g["lookup_cols"]
    assert (oc.lookup_product(lk[0], lk[1], lk[2], lk[3], ps[0], ps[1]) == g["lookup_z"]).all()
    pa, pt = oc.lookup_permute(g["permute_input"], g["permute_table"], 13)
    assert (pa == g["permute_out_input"]).all() and (pt == g["permute_out_table"]).all()
    dec, first = oc.g1_from_bytes(g["codec_bytes"])
    assert first == len(g["codec_bytes"]) and (dec == g["codec_points"]).all()
    assert (oc.g1_to_bytes(g["codec_points"]) == g["codec_bytes"]).all()


def check_golden_prover(L, g):
    """the kernels (emulated or on the GPU) reproduce the same fixture through the C ABI"""
    import halo2_scaffold_b200 as h2
    from halo2_scaffold_b200 import evaluation as ev
    from halo2_scaffold_b200._lib import GraphArrays
    c, sc = g["graph_cols"], g["graph_scalars"]
    ga = GraphArrays(g["graph_constants"], g["graph_rotations"], g["graph_calcs"], g["graph_parts"], 10)
    assert (ev.evaluate_graph(L, ga, c[:1], c[1:4], c[4:], sc[:1], sc[1], sc[2], sc[3], sc[4], g["graph_prev"], 2) == g["graph_out"]).all()
    ps = g["perm_scalars"]
    assert (L.permutation_product(list(g["perm_values"]), list(g["perm_sigma"]), ps[0], ps[1], ps[2], ps[3], ps[4], ps[5]) == g["perm_z"]).all()
    lk = g["lookup_cols"]
    assert (L.lookup_product(lk[0], lk[1], lk[2], lk[3], ps[0], ps[1]) == g["lookup_z"]).all()
    pa, pt = L.lookup_permute(g["permute_input"], g["permute_table"], 13)
    assert (pa == g["permute_out_input"]).all() and (pt == g["permute_out_table"]).all()
    assert (h2.EvaluationDomain(4, 3, lib=L).divide_by_vanishing_poly(g["vanishing_in"]) == g["vanishing_out"]).all()
    assert (L.g1_decode(g["codec_bytes"], 0) == g["codec_points"]).all()
    assert (L.g1_encode(g["codec_points"]) == g["codec_bytes"]).all()


def check_evaluate_graph_property(L, oc, examples, max_rows, max_calcs):
    """Property test over the GraphEvaluator compiler: random program length, column counts, rotation scale, row count and target re-use --
    the re-scheduled, slot-allocated, register-forwarded program always gives the bits of upstream's sequential walk."""
    from hypothesis import given, settings, strategies as st, HealthCheck
    from halo2_scaffold_b200 import evaluation as ev

    @settings(max_examples=examples, deadline=None, suppress_health_check=list(HealthCheck), derandomize=True)
    @given(size=st.integers(1, max_rows), rot_scale=st.sampled_from([1, 2, 4, 8, 3]), n_calcs=st.integers(1, max_calcs), seed=st.integers(0, 10 ** 6),
           reuse=st.booleans(), nf=st.integers(0, 3), na=st.integers(1, 5), ni=st.integers(0, 2), nch=st.integers(0, 2))
    def run(size, rot_scale, n_calcs, seed, reuse, nf, na, ni, nch):
        rng = np.random.default_rng(seed)
        graph, n_const = random_graph(rng, nf, na, ni, nch, n_calcs, reuse_targets=reuse)
        g, ga = _graph_pair(oc, graph, n_const, seed)
        cols = [oc.random_fr(seed * 131 + j, size) for j in range(nf + na + ni)]
        fixed, advice, instance = cols[:nf], cols[nf:nf + na], cols[nf + na:]
        sc = oc.random_fr(seed * 7 + 1, nch + 4)
        challenges, (beta, gamma, theta, y) = sc[:nch], sc[nch:]
        values = oc.random_fr(seed * 7 + 2, size)
        want = oc.evaluate_graph(g, fixed, advice, instance, challenges, beta, gamma, theta, y, values, rot_scale)
        got = ev.evaluate_graph(L, ga, fixed, advice, instance, challenges, beta, gamma, theta, y, values, rot_scale)
        assert (got == want).all(), (size, rot_scale, n_calcs, seed, reuse, nf, na, ni, nch)

    run()


def check_quotient_is_a_polynomial(L, oc, k=4, seed=1, break_it=None):
    """The algebra the verifier relies on, end to end through the device entry points: for a SATISFIED toy circuit -- one
    multiplication gate, copy constraints between three advice columns (two permutation sets), one lookup -- the combination that
    evaluate_h computes vanishes on the whole domain, so (evaluate_h / (X^n - 1)) interpolates to a polynomial of degree < 3n: the top
    quarter of its 4n coefficients is zero.  A wrong rotation, sign, delta / omega bookkeeping or fill order anywhere in evaluate_h,
    the grand products or the lookup permutation breaks exactly this.  `break_it` perturbs one ingredient and must make it fail.
    Uses nothing recalled from upstream beyond the PLONK / halo2 argument itself."""
    import halo2_scaffold_b200 as h2
    from halo2_scaffold_b200 import evaluation as ev
    from halo2_scaffold_b200.domain import fr_to_words, FR_MODULUS as R
    rng = np.random.default_rng(seed)
    n, bf = 1 << k, 5
    u = n - (bf + 1)                                   # usable rows; row u carries l_last, rows u+1.. are blinding rows
    dom = h2.EvaluationDomain(4, k, lib=L)
    en, rot_scale = 1 << dom.extended_k, 1 << (dom.extended_k - k)
    W = lambda vals: np.stack([fr_to_words(int(v)) for v in vals])
    rnd = lambda: int(rng.integers(1, 1 << 62)) * int(rng.integers(1, 1 << 62)) % R
    DELTA = pow(7, 1 << 28, R)
    # ---- witness: c = a * b on the gated rows; copies a[i+1] = c[i] on even usable rows; a stays inside the lookup table
    table = [int(v) for v in rng.integers(0, 50, size=n)]
    q = [1 if (i < u and i % 2 == 0) else 0 for i in range(n)]
    a, b, c = [0] * n, [0] * n, [0] * n
    for i in range(n):
        a[i], b[i], c[i] = rnd(), rnd(), rnd()
    lk = [table[int(rng.integers(0, u))] for _ in range(n)]                  # lookup-advice column: values of the table's usable rows
    copies = []
    for i in range(0, u - 1, 2):
        c[i] = a[i] * b[i] % R
        a[i + 1] = c[i]                                                        # copy constraint (column 0, row i+1) == (column 2, row i)
        copies.append(((0, i + 1), (2, i)))
    cols_perm = [a, b, c]
    omega = dom.omega
    # sigma: identity delta^j omega^i with the two cells of every copy swapped
    sigma = [[pow(DELTA, j, R) * pow(omega, i, R) % R for i in range(n)] for j in range(3)]
    for (j0, i0), (j1, i1) in copies:
        sigma[j0][i0], sigma[j1][i1] = sigma[j1][i1], sigma[j0][i0]
    sc = [rnd() for _ in range(4)]
    beta, gamma, theta, y = sc
    if break_it == "witness":
        c[2] = (c[2] + 1) % R
    # ---- grand products and the lookup permutation on the device, through the host mirrors of the two argument provers (blinding rows included)
    from halo2_scaffold_b200 import prover
    chunk_len = 2
    blind = lambda count: W([rnd() for _ in range(count)])
    ints = lambda w: [o.from_mont(v, R) for v in oc.words_to_ints(np.ascontiguousarray(w))]
    zs, _ = prover.permutation_commit([W(cc) for cc in cols_perm], [W(sg) for sg in sigma], chunk_len=chunk_len, blinding_factors=bf, beta=fr_to_words(beta),
                                      gamma=fr_to_words(gamma), omega=fr_to_words(omega), blind=blind, lib=L)
    z_cols = [ints(z) for z in zs]
    assert len(z_cols) == 2 and z_cols[1][0] == z_cols[0][u], "the second set does not start at the first set's last_z"
    assert z_cols[-1][u] == 1 or break_it, "the permutation product does not close"
    pa, pt, _ = prover.lookup_commit_permuted(W(lk), W(table), blinding_factors=bf, blind=blind, lib=L)
    a_perm, s_perm = ints(pa), ints(pt)
    if break_it == "fill":
        a_perm[0], a_perm[u - 1] = a_perm[u - 1], a_perm[0]
    zl, _ = prover.lookup_commit_product(W(lk), W(table), W(a_perm), W(s_perm), blinding_factors=bf, beta=fr_to_words(beta), gamma=fr_to_words(gamma),
                                         blind=blind, lib=L)
    zl_int = ints(zl)
    assert zl_int[u] == 1 or break_it, "the lookup product does not close"
    # ---- everything to the extended coset
    ext = lambda vals: dom.coeff_to_extended(dom.lagrange_to_coeff(W(vals)))
    l0 = [1] + [0] * (n - 1)
    l_last = [1 if i == u else 0 for i in range(n)]
    l_active = [1 if i < u else 0 for i in range(n)]
    polys = [ev.Product(ev.Fixed(0), ev.Sum(ev.Product(ev.Advice(0), ev.Advice(1)), ev.Negated(ev.Advice(2))))]
    E = ev.Evaluator(polys, [([ev.Advice(3)], [ev.Fixed(1)])])
    sig_for_eval = sigma if break_it != "sigma" else [sigma[1], sigma[0], sigma[2]]
    h_ext = E.evaluate_h(size=en, rot_scale=rot_scale, fixed=[ext(q), ext(table)], advice=[ext(a), ext(b), ext(c), ext(lk)], instance=[],
                         challenges=np.zeros((0, 4), dtype=np.uint64), y=fr_to_words(y), beta=fr_to_words(beta), gamma=fr_to_words(gamma),
                         theta=fr_to_words(theta), l0=ext(l0), l_last=ext(l_last), l_active_row=ext(l_active),
                         permutation=dict(product_cosets=[ext(z) for z in z_cols], columns=[("advice", 0), ("advice", 1), ("advice", 2)],
                                          cosets=[ext(s) for s in sig_for_eval], chunk_len=chunk_len, last_rotation=-(bf + 1), delta=fr_to_words(DELTA),
                                          zeta=fr_to_words(dom.g_coset), extended_omega=fr_to_words(dom.extended_omega)),
                         lookups=[dict(product_coset=ext(zl_int), permuted_input_coset=ext(a_perm), permuted_table_coset=ext(s_perm))], lib=L)
    quotient = dom.divide_by_vanishing_poly(h_ext)
    coeffs = L.ntt(np.ascontiguousarray(quotient), fr_to_words(dom.extended_omega_inv), dom.extended_k)      # scaling / coset factors keep zeros zero
    top = coeffs[3 * n:]
    return not top.any(), h_ext


def check_lookup_permute_async(L, oc):
    """the asynchronous variant leaves the verdict in a device word: 0 for a satisfiable pair, 1 + a sorted row otherwise"""
    n, usable = 200, 194
    pool = oc.random_fr(0xC900, 30)
    rng = np.random.default_rng(9)
    table = pool[np.concatenate([np.arange(30), rng.integers(0, 30, size=n - 30)])]
    inp = table[:usable][rng.integers(0, usable, size=n)]
    for bad in (False, True):
        a = inp.copy()
        if bad:
            a[3] = oc.random_fr(0xC901, 1)[0]
        d = [L.dev_alloc(0, n * 32) for _ in range(4)] + [L.dev_alloc(0, 4)]
        try:
            L.h2d(0, d[0], a)
            L.h2d(0, d[1], table)
            L.lookup_permute_async_dev(0, d[0], d[1], usable, d[2], d[3], d[4])
            L.dev_sync(0)
            status = np.zeros(1, dtype=np.uint32)
            L.d2h(0, status, d[4])
            assert (status[0] != 0) == bad
            if not bad:
                pa, pt = np.empty((usable, 4), dtype=np.uint64), np.empty((usable, 4), dtype=np.uint64)
                L.d2h(0, pa, d[2]); L.d2h(0, pt, d[3])
                wa, wt = oc.lookup_permute(a, table, usable)
                assert (pa == wa).all() and (pt == wt).all()
        finally:
            for p in d:
                L.dev_free(0, p)


def check_evaluate_h_sharded(L, oc, ek=7, k=5, groups=2, seed=6, shards=((0, 40, 24), (40, 50, 24), (90, 38, 30))):
    """row-sharded evaluate_h: every shard sees only its slice (+ halo, wrap-around included) of every column, and the concatenation of the
    shards equals the unsharded evaluation; a halo that is too small is refused"""
    from halo2_scaffold_b200 import evaluation as ev
    from halo2_scaffold_b200._lib import H2BError
    from halo2_scaffold_b200.domain import fr_to_words
    size, rot_scale = 1 << ek, 1 << (ek - k)
    polys, lookup_exprs, nf, na = standard_plonk_like(groups)
    E = ev.Evaluator(polys, lookup_exprs)
    fixed = [oc.random_fr(seed * 1000 + j, size) for j in range(nf)]
    advice = [oc.random_fr(seed * 1000 + 100 + j, size) for j in range(na)]
    instance = [oc.random_fr(seed * 1000 + 200, size)]
    beta, gamma, theta, y, delta, zeta = oc.random_fr(seed * 1000 + 300, 6)
    l0, l_last, l_active = (oc.random_fr(seed * 1000 + 400 + j, size) for j in range(3))
    perm_cols = [("advice", j) for j in range(na)] + [("fixed", 0)]
    n_sets = (len(perm_cols) + 1) // 2
    kw = dict(size=size, rot_scale=rot_scale, fixed=fixed, advice=advice, instance=instance, challenges=np.zeros((0, 4), dtype=np.uint64), y=y, beta=beta,
              gamma=gamma, theta=theta, l0=l0, l_last=l_last, l_active_row=l_active,
              permutation=dict(product_cosets=[oc.random_fr(seed * 1000 + 500 + j, size) for j in range(n_sets)], columns=perm_cols,
                               cosets=[oc.random_fr(seed * 1000 + 600 + j, size) for j in range(len(perm_cols))], chunk_len=2, last_rotation=-6, delta=delta,
                               zeta=zeta, extended_omega=fr_to_words(o.omega_for(ek))),
              lookups=[dict(product_coset=oc.random_fr(seed * 1000 + 700, size), permuted_input_coset=oc.random_fr(seed * 1000 + 701, size),
                            permuted_table_coset=oc.random_fr(seed * 1000 + 702, size))], lib=L)
    # the reference result comes from the ORACLE's three sequential loops, not from an unsharded run of the same library
    def tup(g):
        a = g.arrays()
        return (a.constants, a.rotations, a.calculations, a.parts, a.n_intermediates)
    ch = np.zeros((0, 4), dtype=np.uint64)
    perm = kw["permutation"]
    lk0 = kw["lookups"][0]
    by_type = {"advice": advice, "fixed": fixed, "instance": instance}
    want = oc.evaluate_graph(tup(E.custom_gates), fixed, advice, instance, ch, beta, gamma, theta, y, np.zeros((size, 4), dtype=np.uint64), rot_scale)
    want = oc.evaluate_h_permutation(want, rot_scale, perm["product_cosets"], [by_type[t][i] for t, i in perm_cols], perm["cosets"], 2, -6, l0, l_last,
                                     l_active, beta, gamma, y, delta, zeta, perm["extended_omega"])
    want = oc.evaluate_h_lookup(tup(E.lookups[0]), fixed, advice, instance, ch, beta, gamma, theta, y, want, rot_scale, lk0["product_coset"],
                                lk0["permuted_input_coset"], lk0["permuted_table_coset"], l0, l_last, l_active)
    assert sum(r for _, r, _ in shards) == size
    parts = [E.evaluate_h(shard=sh, **kw) for sh in shards]
    assert (np.concatenate(parts) == want).all(), "row-sharded evaluate_h differs from the oracle"
    assert (E.evaluate_h(**kw) == want).all()
    try:
        E.evaluate_h(shard=(shards[0][0], shards[0][1], 6 * rot_scale - 1), **kw)          # last_rotation = -6 needs 6 * rot_scale rows of halo
        raise AssertionError("a halo that is too small was accepted")
    except H2BError as e:
        assert "halo" in str(e)


# ---- implicit SRS cache of h2b_msm_bn254_g1 (best_multiexp is a pure function) ---------------------------------------------------
def check_implicit_cache_is_content_addressed(L, oc, n, block, seed=41):
    """n: a multiple of the digest block, >= the cache threshold of this process.  Models create_proof followed by verify_proof
    (/root/reference/src/scaffold.rs:191-230): the same SRS vector over and over, re-loaded at new addresses, edited in place,
    prefixes of it, and small fresh arrays in between."""
    s, P = oc.random_fr(seed, n), oc.gen_points(seed + 1, n)
    want = affine_of(oc, oc.best_multiexp(s, P))
    st0 = L.implicit_cache_stats()
    for _ in range(3):      # 1st call: upload, 2nd: window tables are built, 3rd: tables reused
        assert (affine_of(oc, L.msm(s, P)) == want).all()
    st = L.implicit_cache_stats()
    assert st["uploads"] == st0["uploads"] + 1 and st["hits"] == st0["hits"] + 2, (st0, st)
    P2 = P.copy()           # the same vector at another address (scaffold.rs:174 re-reads the params file per proof): no new upload
    assert (affine_of(oc, L.msm(s, P2)) == want).all()
    assert L.implicit_cache_stats()["uploads"] == st["uploads"]
    # in-place edits of single rows that no sparse sample would look at: the old device copy must not be used
    for row in (1, 15, n // 2 + 3, n - 2):
        P2[row] = oc.gen_points(1000 + row, 1)[0]
        want2 = affine_of(oc, oc.best_multiexp(s, P2))
        assert (affine_of(oc, L.msm(s, P2)) == want2).all(), row
    st2 = L.implicit_cache_stats()
    assert st2["stale"] + st2["uploads"] > st["stale"] + st["uploads"]
    # only one limb of one coordinate changes (an invalid point, but the MSM of the OLD array must not come back)
    want_p = affine_of(oc, oc.best_multiexp(s, P))
    assert (affine_of(oc, L.msm(s, P)) == want_p).all()
    # prefixes that are whole blocks reuse the resident copy; ragged ones are uploaded per call
    up = L.implicit_cache_stats()["uploads"]
    for m in (n // 2 - (n // 2) % block, n - block):
        if m >= block and m * 1 >= 1:
            assert (affine_of(oc, L.msm(s[:m], P[:m])) == affine_of(oc, oc.best_multiexp(s[:m], P[:m]))).all(), m
    m = n - 3
    d0 = L.implicit_cache_stats()["direct"]
    assert (affine_of(oc, L.msm(s[:m], P[:m])) == affine_of(oc, oc.best_multiexp(s[:m], P[:m]))).all()
    assert L.implicit_cache_stats()["direct"] == d0 + 1
    # 17 points, only row 15 differs between two calls at the same address
    s17, P17 = oc.random_fr(seed + 5, 17), oc.gen_points(seed + 6, 17)
    a = affine_of(oc, L.msm(s17, P17))
    P17[15] = oc.gen_points(seed + 7, 1)[0]
    b = affine_of(oc, L.msm(s17, P17))
    assert (a != b).any() and (b == affine_of(oc, oc.best_multiexp(s17, P17))).all()
    return up


def check_implicit_cache_under_threads(L, oc, n, threads=8, rounds=3, seed=51):
    """8 host threads: distinct small base arrays (verifier-sized MSMs) interleaved with commits over one large vector.  The large
    vector is uploaded once and never evicted; every result is the oracle's."""
    import threading
    s, P = oc.random_fr(seed, n), oc.gen_points(seed + 1, n)
    want = affine_of(oc, oc.best_multiexp(s, P))
    assert (affine_of(oc, L.msm(s, P)) == want).all()
    up0 = L.implicit_cache_stats()["uploads"]
    small = []
    for t in range(threads):
        m = 20 + 7 * t
        ss, pp = oc.random_fr(seed + 10 + t, m), oc.gen_points(seed + 40 + t, m)
        small.append((ss, pp, affine_of(oc, oc.best_multiexp(ss, pp))))
    errors = []

    def worker(t):
        try:
            ss, pp, w = small[t]
            for r in range(rounds):
                if not (affine_of(oc, L.msm(ss, pp)) == w).all():
                    errors.append(("small", t, r))
                if not (affine_of(oc, L.msm(s, P)) == want).all():
                    errors.append(("large", t, r))
        except Exception as e:      # noqa: BLE001
            errors.append(("exception", t, repr(e)))

    th = [threading.Thread(target=worker, args=(t,)) for t in range(threads)]
    [x.start() for x in th]
    [x.join() for x in th]
    assert not errors, errors[:4]
    st = L.implicit_cache_stats()
    assert st["uploads"] == up0, st      # no re-registration of the large vector


def check_sharded_base_set(L, oc, n, spacing=0, kind=0, seed=61):
    """h2b_register_bases_sharded: rows split over the devices; whole-set, prefix and offset MSMs and batched columns."""
    s, P = edge_msm_inputs(L, oc, n, kind, seed)
    if spacing:
        L.set_msm_precomp(spacing)
    try:
        h = L.register_bases_sharded(P)
    finally:
        L.set_msm_precomp(0)
    try:
        D = L.device_count()
        info = L.base_set_info(h)
        if D > 1 and info["n_tables"] >= 1:
            assert info["device_bytes"] <= info["n_tables"] * ((n + D - 1) // D + 1) * 64
        for off, m in ((0, n), (0, n // 3), (n // 5, n // 2), (n - 1, 1), (n // 2, 0)):
            got = affine_of(oc, L.msm_registered(s[:m], h, off))
            assert (got == affine_of(oc, oc.best_multiexp(s[:m], P[off:off + m]))).all(), (off, m)
        cols = [oc.random_fr(seed + 20 + j, n - 11 * j) for j in range(3)]
        got = L.msm_batch_registered(cols, h)
        for j, c in enumerate(cols):
            assert (affine_of(oc, got[j]) == affine_of(oc, oc.best_multiexp(c, P[:c.shape[0]]))).all(), j
    finally:
        L.unregister_bases(h)


def check_batched_columns(L, oc, n, ncols, spacing=0, kinds=(0, 1), window=0, seed=71):
    """h2b_msm_bn254_g1_batch_registered / _dev_batch_registered: columns of different lengths and distributions (uniform,
    witness-like, all zero, one scalar everywhere) through ONE kernel sequence == single calls == the oracle."""
    P = oc.gen_points(seed, n)
    cols = []
    for j in range(ncols):
        m = n - (j * 37) % (n // 2 + 1)
        c = L.gen_scalars(seed + 1 + j, m, kinds[j % len(kinds)]) if hasattr(L, "gen_scalars") else oc.random_fr(seed + 1 + j, m)
        if j == 2:
            c = np.zeros((m, 4), dtype=np.uint64)
        if j == 3:
            c = np.repeat(oc.fr_to_mont(np.array([[5, 0, 0, 0]], dtype=np.uint64)), m, axis=0)
        cols.append(np.ascontiguousarray(c))
    cols.append(np.zeros((0, 4), dtype=np.uint64))
    want = [affine_of(oc, oc.best_multiexp(c, P[:c.shape[0]])) for c in cols]
    if spacing:
        L.set_msm_precomp(spacing)
    try:
        h = L.register_bases(P)
    finally:
        L.set_msm_precomp(0)
    try:
        L.L.h2b_set_msm_window(window)
        got = L.msm_batch_registered(cols, h)
        for j in range(len(cols)):
            assert (affine_of(oc, got[j]) == want[j]).all(), ("host batch", j)
            assert (affine_of(oc, L.msm_registered(cols[j], h, 0)) == want[j]).all(), ("single", j)
        # device-resident columns
        d_cols = []
        for c in cols:
            p = L.dev_alloc(0, max(c.nbytes, 32))
            if c.nbytes:
                L.h2d(0, p, c)
            d_cols.append(p)
        d_out = L.dev_alloc(0, 224 * len(cols))
        L.msm_dev_batch_registered(0, d_cols, [c.shape[0] for c in cols], h, d_out)
        L.dev_sync(0)
        out = np.zeros((len(cols), 28), dtype=np.uint64)
        L.d2h(0, out, d_out)
        for j in range(len(cols)):
            assert (affine_of(oc, out[j, :12]) == want[j]).all(), ("device batch", j)
        for p in d_cols + [d_out]:
            L.dev_free(0, p)
    finally:
        L.L.h2b_set_msm_window(0)
        L.unregister_bases(h)


def check_batched_ntts(L, oc, k, count, seed=81):
    """h2b_ntt_bn254_fr_batch / _dev_batch: `count` transforms sharing every pass launch == single calls == the oracle"""
    for inverse in (False, True):
        w = omega_words(oc, k, inverse)
        polys = [oc.random_fr(seed + j, 1 << k) for j in range(count)]
        want = [oc.best_fft(a, w, k) for a in polys]
        host = [a.copy() for a in polys]
        L.ntt_batch(host, w, k)
        assert all((a == b).all() for a, b in zip(host, want)), ("host batch", k, inverse)
        ptrs = []
        for a in polys:
            p = L.dev_alloc(0, a.nbytes)
            L.h2d(0, p, a)
            ptrs.append(p)
        L.ntt_dev_batch(0, ptrs, w, k)
        L.dev_sync(0)
        for p, b in zip(ptrs, want):
            got = np.zeros_like(b)
            L.d2h(0, got, p)
            assert (got == b).all(), ("device batch", k, inverse)
            L.dev_free(0, p)


def check_column_pipeline(L, oc, j, k, seed=91):
    """h2b_column_pipeline (commit_lagrange -> lagrange_to_coeff -> coeff_to_extended, one upload) == the three separate steps of the oracle"""
    import halo2_scaffold_b200 as h2
    from halo2_scaffold_b200.domain import fr_to_words
    dom, ref = h2.EvaluationDomain(j, k, lib=L), o.EvaluationDomain(j, k)
    n, en = 1 << k, 1 << ref.extended_k
    col = L.gen_scalars(seed, n, 1)
    gl = oc.gen_points(seed + 1, n)
    h = L.register_bases(gl)
    try:
        zs = np.stack([fr_to_words(1), fr_to_words(ref.g_coset), fr_to_words(ref.g_coset_inv)])
        r = L.column_pipeline(col, h, k, ref.extended_k, fr_to_words(ref.omega_inv), fr_to_words(ref.ifft_divisor), fr_to_words(ref.extended_omega), zs,
                              keep_on_device=True)
        want_commit = affine_of(oc, oc.best_multiexp(col, gl))
        assert (affine_of(oc, r["commitment"]) == want_commit).all()
        want_coeff = oc.fr_scale(oc.best_fft(col, fr_to_words(ref.omega_inv), k), fr_to_words(ref.ifft_divisor))
        assert (r["coeff"] == want_coeff).all()
        e = np.zeros((en, 4), dtype=np.uint64)
        e[:n] = oc.field_op("fr", "mul", want_coeff, np.ascontiguousarray(np.tile(zs, ((n + 2) // 3, 1))[:n]))
        want_ext = oc.best_fft(e, fr_to_words(ref.extended_omega), ref.extended_k)
        assert (r["extended"] == want_ext).all()
        back = np.zeros((en, 4), dtype=np.uint64)
        L.d2h(0, back, r["d_extended"])
        L.dev_free(0, r["d_extended"])
        assert (back == want_ext).all()
        # the same answers as the mirrored three-call path
        assert (dom.lagrange_to_coeff(col) == r["coeff"]).all() and (dom.coeff_to_extended(r["coeff"]) == r["extended"]).all()
        r2 = L.column_pipeline(col, h, k, ref.extended_k, fr_to_words(ref.omega_inv), fr_to_words(ref.ifft_divisor), fr_to_words(ref.extended_omega), zs,
                               want_coeff=False, want_extended=False)
        assert (affine_of(oc, r2["commitment"]) == want_commit).all() and r2["coeff"] is None
    finally:
        L.unregister_bases(h)
