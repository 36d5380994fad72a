"""The device-resident entry points of the C ABI (include/pcdgpu.h: "device-resident polynomials", the `_dev` MSMs and
the xyzz partial-sum helpers) against plain big-integer references, one header clause at a time: aliasing, zeros in
batch inversion, the gather sentinel, the untouched quotient of a division by a larger vanishing polynomial, NULL
outputs, empty inputs, the key bound of shifted commitments, Montgomery-form MSM scalars and xyzz inputs in more than
one projective representation.  Field elements are compared as canonical integers (every device output must also be
below p); points as affine limbs."""
import ctypes

import numpy as np
import pytest

import c_oracle as co
import codec
import kzg_oracle as ko
import marlin_oracle as mo
import synth

FIELDS = [0, 1]
CURVES = [0, 1, 2, 3]
P = codec.FIELD_P
ADD, SUB, MUL, RSUB = 0, 1, 2, 3
NONE = 0xFFFFFFFF
E_ARG = -1
GEN = {0: 10, 1: 17}                  # multiplicative generators (the NTT's coset shifts)
COORD_FIELD = {0: 1, 1: 1, 2: 0, 3: 0}  # MNT4 points have q4 coordinates, MNT6 points r4 ones
K = 256                               # poly.cu's chunk length (and chunks per super-chunk)


# ---- references and encodings (plain Python integers) ----------------------------------------------------------
def _mont(vals, field):
    p = P[field]
    R = (1 << 320) % p
    b = b"".join((v % p * R % p).to_bytes(40, "little") for v in vals)
    return np.frombuffer(b, dtype="<u8").copy().reshape(-1, 5)


def _unmont(limbs, field, canonical=True):
    """Montgomery limbs -> canonical integers; a limb vector >= p (a non-canonical output) fails here unless
    `canonical` is off (xyzz coordinates carry no such promise)"""
    p = P[field]
    Rinv = pow((1 << 320) % p, -1, p)
    raw = np.ascontiguousarray(limbs, dtype="<u8").tobytes()
    out = []
    for i in range(0, len(raw), 40):
        v = int.from_bytes(raw[i:i + 40], "little")
        assert v < p or not canonical, "non-canonical element %#x at %d" % (v, i // 40)
        out.append(v * Rinv % p)
    return out


def _rand(n, field, seed):
    p = P[field]
    raw = np.random.Generator(np.random.Philox(seed)).bytes(40 * n)
    return [int.from_bytes(raw[40 * i:40 * i + 40], "little") % p for i in range(n)]


def _omega(field, N):
    """generator of the multiplicative subgroup of order N (N | p - 1)"""
    p = P[field]
    assert (p - 1) % N == 0
    return pow(GEN[field], (p - 1) // N, p)


def _edges(field):
    p = P[field]
    return [0, 1, p - 1, p - 2]


def _sparse_eval(p, terms, z):
    return sum(c * pow(z, i, p) for i, c in terms) % p


def _xyzz(curve, aff, lam):
    """an affine point (Montgomery limbs) as the xyzz point (lam^2 x, lam^3 y, lam^2, lam^3), lam in the prime field
    under the coordinates (so every coefficient of an extension coordinate scales alike); infinity: all zero"""
    f = COORD_FIELD[curve]
    q = P[f]
    w = codec.COORD_LIMBS[curve] // 5
    a = np.asarray(aff, dtype=np.uint64)
    if not a.any():
        return np.zeros(codec.POINT_LIMBS[curve] * 2, dtype=np.uint64)
    x, y = _unmont(a[:5 * w], f), _unmont(a[5 * w:], f)
    l2, l3 = lam * lam % q, lam * lam * lam % q
    one = [1] + [0] * (w - 1)
    coords = [c * l2 for c in x] + [c * l3 for c in y] + [c * l2 for c in one] + [c * l3 for c in one]
    return _mont(coords, f).reshape(-1)


def _normalise_g1(curve, xyzz):
    """xyzz limbs of a G1 point -> affine limbs (x = X / ZZ, y = Y / ZZZ), in Python"""
    f = COORD_FIELD[curve]
    q = P[f]
    X, Y, ZZ, ZZZ = _unmont(xyzz, f, canonical=False)
    if ZZ == 0:
        return np.zeros(10, dtype=np.uint64)
    return _mont([X * pow(ZZ, -1, q) % q, Y * pow(ZZZ, -1, q) % q], f).reshape(-1)


def _neg(curve, aff):
    f = COORD_FIELD[curve]
    w = codec.COORD_LIMBS[curve] // 5
    c = _unmont(aff, f)
    return _mont(c[:w] + [-v for v in c[w:]], f).reshape(-1)


# ---- CPU self-checks of the helpers above ----------------------------------------------------------------------
def test_reference_helpers():
    for field in FIELDS:
        p = P[field]
        vals = _edges(field) + _rand(20, field, 1)
        assert _unmont(_mont(vals, field), field) == vals
        for N in (2, 256, 1 << 16, 1 << 17):
            w = _omega(field, N)
            assert pow(w, N, p) == 1 and pow(w, N // 2, p) == p - 1
        terms = [(0, 5), (3, 7), (300, 11)]
        dense = [0] * 301
        for i, c in terms:
            dense[i] = c
        for z in (0, 1, p - 1, 12345):
            assert _sparse_eval(p, terms, z) == ko.poly_eval(p, dense, z)
    for N in (7 * 32, 49 * 8):  # mixed-radix domains of q4
        w = _omega(1, N)
        assert pow(w, N, P[1]) == 1 and all(pow(w, N // d, P[1]) != 1 for d in (2, 7))
    # divide_by_vanishing oracle: a = q (X^N - 1) + r at a random point, r zero-padded to N
    for field, N, n in ((0, 2, 5), (1, 224, 1123), (0, 256, 1), (1, 256, 513)):
        p = P[field]
        a = _rand(n, field, n)
        q, r = mo.p_div_vanishing(p, a, N)
        assert len(r) == min(n, N) and len(q) == max(n - N, 0)
        x = 987654321
        assert ko.poly_eval(p, a, x) == (ko.poly_eval(p, q, x) * (pow(x, N, p) - 1) + ko.poly_eval(p, r, x)) % p
    # xyzz encodings: every representation normalises back to the point; -P is on the other branch
    for curve in (0, 2):
        P0 = synth.random_points(1, curve, 3)[0]
        for lam in (1, 2, 123456789):
            assert np.array_equal(_normalise_g1(curve, _xyzz(curve, P0, lam)), P0)
        assert not np.array_equal(_neg(curve, P0), P0) and np.array_equal(_neg(curve, _neg(curve, P0)), P0)


# ---- GPU --------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    import pcd_b200
    c = pcd_b200.Context(0)
    yield c
    c.close()


def _vp(x):
    return ctypes.c_void_p(x)


def _a(arr):
    return ctypes.c_void_p(arr.ctypes.data)


def _ops(ctx, field):
    from pcd_b200 import marlin
    return marlin._Ops(ctx, field)


def _up(ctx, field, vals):
    from pcd_b200 import marlin
    return marlin.DVec.from_host(ctx, field, _mont(vals, field))


def _raw(ctx, arr):
    """an arbitrary array (point limbs, u32 indices) in device memory, as a DVec of 40-byte slots"""
    from pcd_b200 import marlin
    a = np.ascontiguousarray(arr)
    v = marlin.DVec(ctx, 0, max(1, (a.nbytes + 39) // 40))
    ctx._check(ctx.lib.pcdgpu_dev_upload(ctx.h, _vp(v.ptr), _a(a), a.nbytes))
    return v


def _down(v, field):
    return _unmont(v.host(), field)


def _err(ctx):
    return ctx.lib.pcdgpu_last_error(ctx.h).decode()


def _binop(op, p, x, y):
    return ((x + y) if op == ADD else (x - y) if op == SUB else (x * y) if op == MUL else (y - x)) % p


# 1. vec_binary / vec_scalar / vec_axpy
@pytest.mark.gpu
@pytest.mark.parametrize("field", FIELDS)
@pytest.mark.parametrize("n", [1, 255, 256, 257, 1000])
def test_vec_binary_scalar_axpy(ctx, field, n):
    from pcd_b200 import marlin
    p, lib, h = P[field], ctx.lib, ctx.h
    ops = _ops(ctx, field)
    a, b = _rand(n, field, 10 + n), _rand(n, field, 20 + n)
    pairs = [(x, y) for x in _edges(field) for y in _edges(field)]  # every pairing of edge operands first
    for i in range(min(n, len(pairs))):
        a[i], b[i] = pairs[i]
    da, db = _up(ctx, field, a), _up(ctx, field, b)
    for op in (ADD, SUB, MUL, RSUB):
        ref = [_binop(op, p, x, y) for x, y in zip(a, b)]
        out = marlin.DVec(ctx, field, n)
        ops.binary(op, out, da, db, n)
        assert _down(out, field) == ref, op
        # out aliasing a, then out aliasing b
        d = _up(ctx, field, a)
        ctx._check(lib.pcdgpu_vec_binary_dev(h, field, op, _vp(d.ptr), _vp(d.ptr), _vp(db.ptr), n))
        assert _down(d, field) == ref, op
        d = _up(ctx, field, b)
        ctx._check(lib.pcdgpu_vec_binary_dev(h, field, op, _vp(d.ptr), _vp(da.ptr), _vp(d.ptr), n))
        assert _down(d, field) == ref, op
    scalars = _edges(field) + _rand(1, field, 30 + n)
    for s in scalars:
        for op in (ADD, SUB, MUL, RSUB):
            out = marlin.DVec(ctx, field, n)
            ops.scalar(op, out, da, s)
            assert _down(out, field) == [_binop(op, p, x, s) for x in a], (op, s)
        y = _up(ctx, field, b)
        ops.axpy(y, s, da)
        assert _down(y, field) == [(yy + s * x) % p for x, yy in zip(a, b)], s
        # y aliasing x: x + s x
        x = _up(ctx, field, a)
        sl = _mont([s], field)
        ctx._check(lib.pcdgpu_vec_axpy_dev(h, field, _vp(x.ptr), _a(sl), _vp(x.ptr), n))
        assert _down(x, field) == [(1 + s) * v % p for v in a], s
    # in-place scalar op (out aliasing a)
    d = _up(ctx, field, a)
    ops.scalar(RSUB, d, d, scalars[-1])
    assert _down(d, field) == [(scalars[-1] - x) % p for x in a]


@pytest.mark.gpu
def test_vec_empty_and_argument_errors(ctx):
    from pcd_b200 import marlin
    lib, h = ctx.lib, ctx.h
    for field in FIELDS:
        s = _mont([3], field)
        assert lib.pcdgpu_vec_binary_dev(h, field, ADD, None, None, None, 0) == 0
        assert lib.pcdgpu_vec_scalar_dev(h, field, MUL, None, None, _a(s), 0) == 0
        assert lib.pcdgpu_vec_axpy_dev(h, field, None, _a(s), None, 0) == 0
        assert lib.pcdgpu_vec_inverse_dev(h, field, None, 0) == 0
        assert lib.pcdgpu_vec_powers_dev(h, field, None, _a(s), _a(s), 0) == 0
        assert lib.pcdgpu_vec_gather_dev(h, field, None, None, None, 0) == 0
        out = np.full(5, 0x1234, dtype=np.uint64)
        assert lib.pcdgpu_poly_eval_dev(h, field, None, 0, _a(s), _a(out)) == 0
        assert not out.any()  # the empty polynomial evaluates to 0
    ctx.sync()
    d = marlin.DVec.zeros(ctx, 0, 4)
    s = _mont([3], 0)
    for op in (4, -1):
        assert lib.pcdgpu_vec_binary_dev(h, 0, op, _vp(d.ptr), _vp(d.ptr), _vp(d.ptr), 4) == E_ARG
        assert _err(ctx)
        assert lib.pcdgpu_vec_scalar_dev(h, 0, op, _vp(d.ptr), _vp(d.ptr), _a(s), 4) == E_ARG
    F = 2  # no such field
    assert lib.pcdgpu_vec_binary_dev(h, F, ADD, _vp(d.ptr), _vp(d.ptr), _vp(d.ptr), 4) == E_ARG
    assert "field" in _err(ctx)
    assert lib.pcdgpu_vec_scalar_dev(h, F, ADD, _vp(d.ptr), _vp(d.ptr), _a(s), 4) == E_ARG
    assert lib.pcdgpu_vec_axpy_dev(h, F, _vp(d.ptr), _a(s), _vp(d.ptr), 4) == E_ARG
    assert lib.pcdgpu_vec_inverse_dev(h, F, _vp(d.ptr), 4) == E_ARG
    assert lib.pcdgpu_vec_powers_dev(h, F, _vp(d.ptr), _a(s), _a(s), 4) == E_ARG
    assert lib.pcdgpu_vec_gather_dev(h, F, _vp(d.ptr), _vp(d.ptr), _vp(d.ptr), 4) == E_ARG
    out = np.zeros(5, dtype=np.uint64)
    assert lib.pcdgpu_poly_eval_dev(h, F, _vp(d.ptr), 4, _a(s), _a(out)) == E_ARG
    # the rejected calls launched nothing: the vector is still zero
    assert _down(d, 0) == [0] * 4


# 2. vec_inverse
@pytest.mark.gpu
@pytest.mark.parametrize("field", FIELDS)
@pytest.mark.parametrize("n", [1, 7, 8, 9, 15, 16, 17, 1000, (1 << 16) + 3])
def test_vec_inverse(ctx, field, n):
    p = P[field]
    ops = _ops(ctx, field)
    x = _rand(n, field, 40 + n)
    if n > 2:
        x[1], x[2] = 1, p - 1
    if n >= 32:
        x[16:24] = [0] * 8  # a whole chunk of eight
    for i in (0, 7, 8, n - 1):
        if i < n:
            x[i] = 0
    dense = _rand(n, field, 50 + n)  # no zeros (with overwhelming probability; asserted)
    assert all(dense)
    for vals in (x, dense, [0] * n):
        d = _up(ctx, field, vals)
        ops.inverse_inplace(d)
        got = _down(d, field)
        bad = [i for i, (v, w) in enumerate(zip(vals, got)) if (w != 0 if v == 0 else v * w % p != 1)]
        assert not bad, bad[:10]


# 3. vec_powers
@pytest.mark.gpu
@pytest.mark.parametrize("field", FIELDS)
@pytest.mark.parametrize("n", [1, 255, 256, 257, 4096, 1 << 20])
def test_vec_powers(ctx, field, n):
    p = P[field]
    ops = _ops(ctx, field)
    N = min(n, 1 << (34, 17)[field]) if n & (n - 1) == 0 else 256  # omega_N with N = n where the field has it
    w = _omega(field, N)
    rng = np.random.Generator(np.random.Philox(60 + n))
    spots = sorted({0, 1, 255, 256, N - 1, N, n - 1} | {int(i) for i in rng.integers(0, n, 64)})
    spots = [i for i in spots if i < n]
    for base in (0, 1, p - 1, w, _rand(1, field, 61)[0]):
        for scale in (0, 1, _rand(1, field, 62)[0]):
            d = ops.powers(base, scale, n)
            raw = d.host()
            if n <= 4096:
                got, exp, acc = _unmont(raw, field), [], scale
                for _ in range(n):
                    exp.append(acc)
                    acc = acc * base % p
                assert got == exp, (base, scale)
            else:
                got = _unmont(raw[spots], field)
                assert got == [scale * pow(base, i, p) % p for i in spots], (base, scale)
            if base == w and scale == 1 and N <= n:
                last = _unmont(raw[N - 1], field)[0]
                assert last * w % p == 1


# 4. vec_gather
@pytest.mark.gpu
@pytest.mark.parametrize("field", FIELDS)
def test_vec_gather(ctx, field):
    p = P[field]
    lib, h = ctx.lib, ctx.h
    src = _rand(1000, field, 70)
    src[0] = 5
    dsrc = _up(ctx, field, src)
    rng = np.random.Generator(np.random.Philox(71))
    for n in (1, 255, 257, 1000, 3001):
        idx = rng.integers(0, len(src), n).astype(np.uint32)
        idx[rng.random(n) < 0.2] = NONE
        idx[0] = NONE
        for k, v in ((1, 0), (2, len(src) - 1), (3, 17), (4, 17), (5, 0), (n - 1, NONE)):
            if k < n:
                idx[k] = v
        didx = _raw(ctx, idx)
        out = _up(ctx, field, [p - 1] * n)  # prefilled: the sentinel must write a zero
        ctx._check(lib.pcdgpu_vec_gather_dev(h, field, _vp(out.ptr), _vp(dsrc.ptr), _vp(didx.ptr), n))
        assert _down(out, field) == [0 if j == NONE else src[j] for j in idx], n


# 5. poly_eval_dev
@pytest.mark.gpu
@pytest.mark.parametrize("field", FIELDS)
@pytest.mark.parametrize("n", [1, 2, 255, 256, 257, 65535, 65536, 65537, 2 * 65536 + 1])
def test_poly_eval_dev(ctx, field, n):
    p = P[field]
    ops = _ops(ctx, field)
    coeffs = _rand(n, field, 80 + n)
    d = _up(ctx, field, coeffs)
    for z in (0, 1, p - 1, _omega(field, 1 << 16), _rand(1, field, 81)[0]):
        assert ops.evaluate(d, z) == ko.poly_eval(p, coeffs, z), z


@pytest.mark.gpu
@pytest.mark.parametrize("field", FIELDS)
def test_poly_eval_dev_many_superchunks(ctx, field):
    """K * K + 5 coefficients (671 MB on the device): the top kernel walks 257 super-chunks.  Zero except at chunk and
    super-chunk edges, so the reference is a short sum of powers."""
    from pcd_b200 import marlin
    p = P[field]
    n = K * K * K + 5
    d = marlin.DVec.zeros(ctx, field, n)
    pos = sorted({0, 1, K - 1, K, K * K - 1, K * K, K * K + 1, 2 * K * K, 255 * K * K + 3, K ** 3 - 1, K ** 3, n - 1})
    vals = _rand(len(pos), field, 90)
    for i, v in zip(pos, vals):
        limbs = _mont([v], field)
        ctx._check(ctx.lib.pcdgpu_dev_upload(ctx.h, _vp(d.ptr + i * 40), _a(limbs), 40))
    ops = _ops(ctx, field)
    for z in (0, 1, p - 1, _omega(field, 1 << 16), _rand(1, field, 91)[0]):
        assert ops.evaluate(d, z) == _sparse_eval(p, zip(pos, vals), z), z


# 6. poly_divide_vanishing_dev
@pytest.mark.gpu
@pytest.mark.parametrize("field,N", [(f, N) for f in FIELDS for N in (1, 2, 256)] + [(1, 7 * 32), (1, 49 * 8)])
def test_poly_divide_vanishing_dev(ctx, field, N):
    p = P[field]
    lib, h = ctx.lib, ctx.h
    SENT = p - 7
    for n in sorted({1, N - 1, N, N + 1, 2 * N, 2 * N + 1, 5 * N + 3} - {0}):
        a = _rand(n, field, 100 + n)
        dp = _up(ctx, field, a)
        q_ref, r_ref = mo.p_div_vanishing(p, a, N)
        r_ref = r_ref + [0] * (N - len(r_ref))
        dq = _up(ctx, field, [SENT] * max(n - N, 1))
        dr = _up(ctx, field, [SENT] * N)
        ctx._check(lib.pcdgpu_poly_divide_vanishing_dev(h, field, _vp(dp.ptr), n, N, _vp(dq.ptr), _vp(dr.ptr)))
        assert _down(dr, field) == r_ref, n
        assert _down(dq, field) == (q_ref if n > N else [SENT]), n
        if n <= N:  # no quotient: q may be NULL
            dr = _up(ctx, field, [SENT] * N)
            ctx._check(lib.pcdgpu_poly_divide_vanishing_dev(h, field, _vp(dp.ptr), n, N, None, _vp(dr.ptr)))
            assert _down(dr, field) == r_ref, n
        else:  # through the Python mirror
            q, r = _ops(ctx, field).divide_by_vanishing(dp, N)
            assert _down(q, field) == q_ref and _down(r, field) == r_ref, n


# 7. poly_divide_linear_dev
@pytest.mark.gpu
@pytest.mark.parametrize("field", FIELDS)
@pytest.mark.parametrize("n", [1, 256, 257, 65537])
def test_poly_divide_linear_dev(ctx, field, n):
    p = P[field]
    lib, h = ctx.lib, ctx.h
    ops = _ops(ctx, field)
    coeffs = _rand(n, field, 110 + n)
    d = _up(ctx, field, coeffs)
    for z in (0, 1, _rand(1, field, 111)[0]):
        q_ref, v_ref = ko.poly_divide_linear(p, coeffs, z)
        # out_eval = NULL: asynchronous; the download that follows is ordered after it on the stream
        q = ops.divide_by_linear(d, z)
        assert _down(q, field) == q_ref, z
        dq = _up(ctx, field, [p - 1] * max(n - 1, 1))
        ev = np.zeros(5, dtype=np.uint64)
        zl = _mont([z], field)
        ctx._check(lib.pcdgpu_poly_divide_linear_dev(h, field, _vp(d.ptr), n, _a(zl), _vp(dq.ptr) if n > 1 else None,
                                                     _a(ev)))
        assert _unmont(ev, field) == [v_ref], z
        if n > 1:
            assert _down(dq, field) == q_ref, z


# 8. csr_upload / csr_matvec
def _csr(rows):
    ptr, col, val = [0], [], []
    for r in rows:
        for c, v in r:
            col.append(c)
            val.append(v)
        ptr.append(len(col))
    return np.array(ptr, dtype=np.uint32), np.array(col, dtype=np.uint32), val


@pytest.mark.gpu
@pytest.mark.parametrize("field", FIELDS)
def test_csr_matvec(ctx, field):
    p = P[field]
    lib, h = ctx.lib, ctx.h
    ops = _ops(ctx, field)
    ncols = 50
    rng = np.random.Generator(np.random.Philox(120 + field))
    big = [(int(c), v) for c, v in zip(rng.integers(0, ncols, 300), _rand(300, field, 121))]
    for k in range(0, 300, 7):  # Montgomery one (the fast path), zero and two among the values
        big[k] = (big[k][0], (1, 0, 2)[k % 3])
    matrices = [
        [[(ncols - 1, 1), (0, p - 1)]],  # m = 1
        [[]],                            # m = 1, empty
        [[], [(0, 1), (ncols - 1, 2), (3, 0), (3, 5), (3, 1)], big, [], [(ncols - 1, 1)], []],
    ]
    x = _rand(ncols, field, 122)
    dx = _up(ctx, field, x)
    for rows in matrices:
        ptr, col, val = _csr(rows)
        m = len(rows)
        vl = _mont(val, field) if val else np.zeros((1, 5), dtype=np.uint64)
        c = ctypes.c_void_p()
        ctx._check(lib.pcdgpu_csr_upload(h, field, m, ncols, _a(ptr), _a(col) if col.size else None, _a(vl),
                                         ctypes.byref(c)))
        try:
            out = ops.matvec(c, dx, m)
            assert _down(out, field) == [sum(v * x[j] for j, v in r) % p for r in rows]
            # the same into a prefilled buffer: empty rows must write a zero
            out = _up(ctx, field, [p - 1] * m)
            ctx._check(lib.pcdgpu_csr_matvec_dev(h, c, _vp(dx.ptr), _vp(out.ptr)))
            assert _down(out, field) == [sum(v * x[j] for j, v in r) % p for r in rows]
        finally:
            lib.pcdgpu_csr_free(c)
    one = _mont([1, 1, 1], field)

    def upload(f, m, ptr, col):
        c = ctypes.c_void_p()
        ptr, col = np.array(ptr, dtype=np.uint32), np.array(col, dtype=np.uint32)
        rc = lib.pcdgpu_csr_upload(h, f, m, 4, _a(ptr), _a(col), _a(one), ctypes.byref(c))
        if rc == 0:
            lib.pcdgpu_csr_free(c)
        return rc

    assert upload(field, 1, [0, 2], [0, 3]) == 0
    assert upload(field, 1, [1, 2], [0, 3]) == E_ARG and "row_ptr[0]" in _err(ctx)
    assert upload(field, 3, [0, 2, 1, 3], [0, 1, 2]) == E_ARG and "monotone" in _err(ctx)
    assert upload(field, 1, [0, 2], [0, 4]) == E_ARG and "column" in _err(ctx)
    assert upload(2, 1, [0, 2], [0, 3]) == E_ARG and "field" in _err(ctx)


# 9. kzg_commit_dev
@pytest.mark.gpu
@pytest.mark.parametrize("pairing,pre", [(0, False), (0, True), (1, False), (1, True)])
def test_kzg_commit_dev(ctx, pairing, pre):
    from pcd_b200 import kzg
    field = pairing
    p = P[field]
    g1 = codec.G1_OF[pairing]
    G = synth.generator_limbs(g1)
    beta, gamma = pow(3, 217, p), pow(5, 61, p)
    deg = 64
    pg, pgg = ko.setup(pairing, deg, beta, gamma, G, 8)
    powers = kzg.Powers(ctx, pairing, pg, pgg, precompute=pre)
    nk, nkg = pg.shape[0], pgg.shape[0]
    lib, h = ctx.lib, ctx.h

    def commit(shift, n, n_rand, seed):
        c, r = _rand(n, field, seed), _rand(n_rand, field, seed + 1)
        dc = _up(ctx, field, c) if n else None
        dr = _up(ctx, field, r) if n_rand else None
        out = np.full(10, 7, dtype=np.uint64)
        rc = lib.pcdgpu_kzg_commit_dev(h, powers.powers_of_g.h, shift, _vp(dc.ptr) if dc else None, n,
                                       powers.powers_of_gamma_g.h, _vp(dr.ptr) if dr else None, n_rand, _a(out))
        return rc, out, c, r

    try:
        for shift, n, n_rand in ((0, 40, 0), (0, 40, 3), (nk - 40, 40, 0), (nk - 40, 40, 2), (nk - 1, 1, 0),
                                 (0, nk, 0), (0, nk, nkg), (5, 0, 0), (nk, 0, 0), (0, 0, 3)):
            rc, out, c, r = commit(shift, n, n_rand, 130 + shift + n)
            assert rc == 0, _err(ctx)
            log = (sum(ci * pow(beta, shift + i, p) for i, ci in enumerate(c)) +
                   gamma * ko.poly_eval(p, r, beta)) % p
            if log == 0:
                assert not out.any(), (shift, n, n_rand)  # infinity
            else:
                assert np.array_equal(out, co.fixed_base_mul(g1, G, ko._limbs([log]), 1)[0]), (shift, n, n_rand)
            parts = ([co.msm(g1, pg[shift:shift + n], ko._limbs(c))] if n else []) + \
                    ([co.msm(g1, pgg[:n_rand], ko._limbs(r))] if n_rand else [])
            ref = co.point_sum(g1, np.stack(parts)) if parts else np.zeros(10, dtype=np.uint64)
            assert np.array_equal(out, ref), (shift, n, n_rand)
        rc, out, _, _ = commit(nk - 39, 40, 0, 1)  # shift + n = powers_of_g.n + 1
        assert rc == E_ARG and "exceeds" in _err(ctx)
        assert np.all(out == 7)
        rc, _, _, _ = commit(0, 4, nkg + 1, 2)
        assert rc == E_ARG and "blinding" in _err(ctx)
    finally:
        powers.close()


# 10. msm_dev / Bases.msm_dev with Montgomery-form scalars
def _read_xyzz(ctx, curve, d_out):
    """the MSM's xyzz result read twice: summed (and normalised) by the library, and on G1 normalised in Python"""
    xyzz = ctx.xyzz_download(curve, d_out.ptr)
    got = ctx.xyzz_sum(curve, xyzz)
    if curve in (0, 2):
        assert np.array_equal(_normalise_g1(curve, xyzz), got)
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("curve", CURVES)
def test_msm_dev_mont_scalars(ctx, curve):
    from pcd_b200 import Bases, marlin
    f = codec.SCALAR_FIELD[curve]
    r = P[f]
    n = 400 if curve in (0, 2) else 120
    extra = 17
    pts = synth.random_points(n + extra, curve, 140 + curve)
    plain = [0, 1, r - 1, 2] + _rand(n - 4, f, 141)
    ref = co.msm(curve, pts[extra:], ko._limbs(plain), 8)
    dpts = _raw(ctx, pts[extra:])
    dmont = _up(ctx, f, plain)
    dplain = _raw(ctx, ko._limbs(plain))
    d_out = marlin.DVec(ctx, f, codec.POINT_LIMBS[curve] * 2 // 5)
    ctx.msm_dev(curve, dpts.ptr, dmont.ptr, n, d_out.ptr, scalars_mont=True)
    assert np.array_equal(_read_xyzz(ctx, curve, d_out), ref)
    ctx.msm_dev(curve, dpts.ptr, dplain.ptr, n, d_out.ptr, scalars_mont=False)
    assert np.array_equal(_read_xyzz(ctx, curve, d_out), ref)
    # resident bases, with and without window tables, at an offset that ends at the last point
    for pre in (False, True):
        b = Bases(ctx, curve, pts, pre)
        try:
            b.msm_dev(dmont.ptr, n, d_out.ptr, offset=extra, scalars_mont=True)
            assert np.array_equal(_read_xyzz(ctx, curve, d_out), ref), pre
            b.msm_dev(dmont.ptr + 40, n - 1, d_out.ptr, offset=extra + 1, scalars_mont=True)
            assert np.array_equal(_read_xyzz(ctx, curve, d_out), co.msm(curve, pts[extra + 1:], ko._limbs(plain[1:]), 8))
        finally:
            b.close()


# 11. xyzz_sum
@pytest.mark.gpu
@pytest.mark.parametrize("curve", CURVES)
def test_xyzz_sum(ctx, curve):
    from pcd_b200 import Bases, marlin
    lib, h = ctx.lib, ctx.h
    q = P[COORD_FIELD[curve]]
    f = codec.SCALAR_FIELD[curve]
    pts = synth.random_points(3, curve, 150 + curve)
    out = np.full(codec.POINT_LIMBS[curve], 9, dtype=np.uint64)
    ctx._check(lib.pcdgpu_xyzz_sum(h, curve, None, 0, _a(out)))
    assert not out.any()
    lam1, lam2 = 123456789, q - 3
    # one point in two representations: the sum doubles it
    two = co.fixed_base_mul(curve, pts[0], ko._limbs([2]), 1)[0]
    assert np.array_equal(ctx.xyzz_sum(curve, np.stack([_xyzz(curve, pts[0], 1), _xyzz(curve, pts[0], lam1)])), two)
    assert np.array_equal(ctx.xyzz_sum(curve, np.stack([_xyzz(curve, pts[0], lam2), _xyzz(curve, pts[0], lam1)])), two)
    # P + (-P) = infinity, in either order and representation
    neg = _neg(curve, pts[0])
    assert not ctx.xyzz_sum(curve, np.stack([_xyzz(curve, pts[0], lam1), _xyzz(curve, neg, lam2)])).any()
    assert not ctx.xyzz_sum(curve, np.stack([_xyzz(curve, neg, 1), _xyzz(curve, pts[0], 1)])).any()
    # an entry with ZZ = 0 (its other coordinates nonzero) is the point at infinity
    inf = _xyzz(curve, pts[1], lam1)
    w = codec.COORD_LIMBS[curve]
    inf[2 * w:3 * w] = 0
    parts = np.stack([_xyzz(curve, pts[0], lam1), inf, _xyzz(curve, pts[1], 1), _xyzz(curve, pts[2], lam2), inf])
    assert np.array_equal(ctx.xyzz_sum(curve, parts), co.point_sum(curve, pts))
    assert np.array_equal(ctx.xyzz_sum(curve, inf), np.zeros(codec.POINT_LIMBS[curve], dtype=np.uint64))
    # the partials of one MSM over three point ranges (the sharded prover's gather, on one GPU) sum to the MSM
    n = 600 if curve in (0, 2) else 150
    bp = synth.random_points(n, curve, 160 + curve)
    sc = synth.random_scalars(n, curve, 161 + curve, "W")
    ref = co.msm(curve, bp, sc, 8)
    ds = _raw(ctx, sc)
    xb = codec.POINT_LIMBS[curve] * 2 * 8
    d_out = marlin.DVec(ctx, f, 3 * xb // 40)
    b = Bases(ctx, curve, bp)
    try:
        cuts = [0, n // 3, n // 3 + 1, n]  # the middle range holds one point
        for k in range(3):
            lo, hi = cuts[k], cuts[k + 1]
            b.msm_dev(ds.ptr + lo * 40, hi - lo, d_out.ptr + k * xb, offset=lo)
        partials = np.stack([ctx.xyzz_download(curve, d_out.ptr + k * xb) for k in range(3)])
        assert np.array_equal(ctx.xyzz_sum(curve, partials), ref)
    finally:
        b.close()


# 12. one chain of asynchronous calls
@pytest.mark.gpu
@pytest.mark.parametrize("field", FIELDS)
def test_chained_async_sequence(ctx, field):
    """powers -> alpha - x -> batch inversion -> axpy -> pointwise product -> division by the vanishing polynomial ->
    division by X - z -> add -> evaluation, with no synchronisation between the calls; one download at the end"""
    from pcd_b200 import marlin
    p = P[field]
    lib, h = ctx.lib, ctx.h
    ops = _ops(ctx, field)
    n, N = 5000, 1024
    w = _omega(field, 8192)
    s0, c, z, zeta = _rand(4, field, 170)
    alpha = s0 * pow(w, 5, p) % p  # alpha - x_5 = 0: a zero goes through the inversion
    y0, m = _rand(n, field, 171), _rand(n, field, 172)
    dy, dm = _up(ctx, field, y0), _up(ctx, field, m)
    t = marlin.DVec(ctx, field, n)
    dq = marlin.DVec(ctx, field, n - N)
    dr = marlin.DVec(ctx, field, N)
    dq2 = marlin.DVec(ctx, field, n - N - 1)
    ctx.sync()
    # --- no synchronisation from here on until the downloads ---
    pw = ops.powers(w, s0, n)
    ops.scalar(RSUB, t, pw, alpha)
    ops.inverse_inplace(t)
    ops.axpy(dy, c, t)
    ops.binary(MUL, dy, dy, dm, n)
    ctx._check(lib.pcdgpu_poly_divide_vanishing_dev(h, field, _vp(dy.ptr), n, N, _vp(dq.ptr), _vp(dr.ptr)))
    zl = _mont([z], field)
    ctx._check(lib.pcdgpu_poly_divide_linear_dev(h, field, _vp(dq.ptr), n - N, _a(zl), _vp(dq2.ptr), None))
    ops.binary(ADD, dr, dr, dq2, N)
    got_eval = ops.evaluate(dr, zeta)
    got_r, got_q2 = _down(dr, field), _down(dq2, field)
    # the same chain in Python
    x = [s0 * pow(w, i, p) % p for i in range(n)]
    tt = [(alpha - v) % p for v in x]
    assert tt[5] == 0
    tt = [pow(v, -1, p) if v else 0 for v in tt]
    y = [(a + c * b) % p * mm % p for a, b, mm in zip(y0, tt, m)]
    q, r = mo.p_div_vanishing(p, y, N)
    q2, _ = ko.poly_divide_linear(p, q, z)
    r = [(a + (q2[i] if i < len(q2) else 0)) % p for i, a in enumerate(r)]
    assert got_q2 == q2
    assert got_r == r
    assert got_eval == ko.poly_eval(p, r, zeta)
