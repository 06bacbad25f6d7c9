"""Integer model of the BN254 pairing as csrc/fp12.cuh and csrc/pairing.cu compute it.

Fp2 = Fp[u]/(u^2 + 1), Fp6 = Fp2[v]/(v^3 - xi) with xi = 9 + u, Fp12 = Fp6[w]/(w^2 - v).  Elements are
nested tuples of ints; the formulas (sparse line product, projective Miller steps, cyclotomic squaring,
the exp-by-x chain of the hard part) are the device's, step for step, so the CPU suite pins them against
the oracle's py_ecc restatement without a GPU.
"""
P = 21888242871839275222246405745257275088696311157297823662689037894645226208583
R = 21888242871839275222246405745257275088548364400416034343698204186575808495617
X = 4965661367192848881            # BN parameter; the ate loop runs over 6x + 2
ATE = 6 * X + 2
XI = (9, 1)


# ---- Fp2
def f2(a, b=0):
    return (a % P, b % P)


def f2_add(a, b):
    return ((a[0] + b[0]) % P, (a[1] + b[1]) % P)


def f2_sub(a, b):
    return ((a[0] - b[0]) % P, (a[1] - b[1]) % P)


def f2_neg(a):
    return ((-a[0]) % P, (-a[1]) % P)


def f2_mul(a, b):
    return ((a[0] * b[0] - a[1] * b[1]) % P, (a[0] * b[1] + a[1] * b[0]) % P)


def f2_sqr(a):
    return f2_mul(a, a)


def f2_scale(a, k):
    return (a[0] * k % P, a[1] * k % P)


def f2_conj(a):
    return (a[0], (-a[1]) % P)


def f2_mul_xi(a):
    return ((9 * a[0] - a[1]) % P, (a[0] + 9 * a[1]) % P)


def f2_inv(a):
    d = pow((a[0] * a[0] + a[1] * a[1]) % P, -1, P)
    return (a[0] * d % P, (-a[1] * d) % P)


def f2_pow(a, e):
    r = (1, 0)
    while e:
        if e & 1:
            r = f2_mul(r, a)
        a = f2_mul(a, a)
        e >>= 1
    return r


F2_ZERO, F2_ONE = (0, 0), (1, 0)


# ---- Fp6
def f6_add(a, b):
    return tuple(f2_add(x, y) for x, y in zip(a, b))


def f6_sub(a, b):
    return tuple(f2_sub(x, y) for x, y in zip(a, b))


def f6_neg(a):
    return tuple(f2_neg(x) for x in a)


def f6_mul(a, b):
    t0, t1, t2 = f2_mul(a[0], b[0]), f2_mul(a[1], b[1]), f2_mul(a[2], b[2])
    c0 = f2_add(f2_mul_xi(f2_sub(f2_sub(f2_mul(f2_add(a[1], a[2]), f2_add(b[1], b[2])), t1), t2)), t0)
    c1 = f2_add(f2_sub(f2_sub(f2_mul(f2_add(a[0], a[1]), f2_add(b[0], b[1])), t0), t1), f2_mul_xi(t2))
    c2 = f2_add(f2_sub(f2_sub(f2_mul(f2_add(a[0], a[2]), f2_add(b[0], b[2])), t0), t2), t1)
    return (c0, c1, c2)


def f6_mul_v(a):
    return (f2_mul_xi(a[2]), a[0], a[1])


def f6_mul_01(a, b0, b1):
    """a * (b0 + b1 v)"""
    t0, t1 = f2_mul(a[0], b0), f2_mul(a[1], b1)
    c0 = f2_add(f2_mul_xi(f2_sub(f2_mul(f2_add(a[1], a[2]), b1), t1)), t0)
    c1 = f2_sub(f2_sub(f2_mul(f2_add(a[0], a[1]), f2_add(b0, b1)), t0), t1)
    c2 = f2_add(f2_sub(f2_mul(f2_add(a[0], a[2]), b0), t0), t1)
    return (c0, c1, c2)


def f6_inv(a):
    c0 = f2_sub(f2_sqr(a[0]), f2_mul_xi(f2_mul(a[1], a[2])))
    c1 = f2_sub(f2_mul_xi(f2_sqr(a[2])), f2_mul(a[0], a[1]))
    c2 = f2_sub(f2_sqr(a[1]), f2_mul(a[0], a[2]))
    t = f2_add(f2_mul(a[0], c0), f2_mul_xi(f2_add(f2_mul(a[2], c1), f2_mul(a[1], c2))))
    ti = f2_inv(t)
    return (f2_mul(c0, ti), f2_mul(c1, ti), f2_mul(c2, ti))


F6_ZERO = (F2_ZERO, F2_ZERO, F2_ZERO)
F6_ONE = (F2_ONE, F2_ZERO, F2_ZERO)


# ---- Fp12
ONE = (F6_ONE, F6_ZERO)


def f12_mul(a, b):
    t0, t1 = f6_mul(a[0], b[0]), f6_mul(a[1], b[1])
    c1 = f6_sub(f6_sub(f6_mul(f6_add(a[0], a[1]), f6_add(b[0], b[1])), t0), t1)
    return (f6_add(t0, f6_mul_v(t1)), c1)


def f12_sqr(a):
    # (a0 + a1 w)^2 = (a0 + a1)(a0 + v a1) - a0 a1 - v a0 a1 + 2 a0 a1 w
    m = f6_mul(a[0], a[1])
    c0 = f6_sub(f6_sub(f6_mul(f6_add(a[0], a[1]), f6_add(a[0], f6_mul_v(a[1]))), m), f6_mul_v(m))
    return (c0, f6_add(m, m))


def f12_mul_line(f, c00, c10, c11):
    """f * (c00 + c10 w + c11 w^3): the line's coefficients sit at w^0, w^1, w^3 = c0.c0, c1.c0, c1.c1"""
    t0 = tuple(f2_mul(x, c00) for x in f[0])
    t1 = f6_mul_01(f[1], c10, c11)
    c1 = f6_sub(f6_sub(f6_mul_01(f6_add(f[0], f[1]), f2_add(c00, c10), c11), t0), t1)
    return (f6_add(t0, f6_mul_v(t1)), c1)


def f12_conj(a):
    return (a[0], f6_neg(a[1]))


def f12_inv(a):
    t = f6_inv(f6_sub(f6_mul(a[0], a[0]), f6_mul_v(f6_mul(a[1], a[1]))))
    return (f6_mul(a[0], t), f6_neg(f6_mul(a[1], t)))


def frobenius_coeffs():
    """GAMMA[k-1][i] = xi^(i (p^k - 1) / 6), k = 1..3, i = 0..5 (Fp2 pairs)"""
    return [[f2_pow(XI, i * (P ** k - 1) // 6) for i in range(6)] for k in (1, 2, 3)]


GAMMA = frobenius_coeffs()


def _w_coeffs(a):
    """the Fp2 coefficients of w^0..w^5"""
    return [a[0][0], a[1][0], a[0][1], a[1][1], a[0][2], a[1][2]]


def _from_w_coeffs(g):
    return ((g[0], g[2], g[4]), (g[1], g[3], g[5]))


def f12_frobenius(a, k):
    g = _w_coeffs(a)
    if k & 1:
        g = [f2_conj(x) for x in g]
    return _from_w_coeffs([f2_mul(g[i], GAMMA[k - 1][i]) for i in range(6)])


def f12_cyclotomic_sqr(a):
    """Granger-Scott squaring, valid for elements of the cyclotomic subgroup (after the easy part)"""
    def fp4_sqr(x, y):
        t0, t1 = f2_sqr(x), f2_sqr(y)
        return f2_add(f2_mul_xi(t1), t0), f2_sub(f2_sub(f2_sqr(f2_add(x, y)), t0), t1)
    z0, z4, z3 = a[0]
    z2, z1, z5 = a[1]
    t0, t1 = fp4_sqr(z0, z1)
    z0 = f2_add(f2_scale(f2_sub(t0, z0), 2), t0)
    z1 = f2_add(f2_scale(f2_add(t1, z1), 2), t1)
    t0, t1 = fp4_sqr(z2, z3)
    t2, t3 = fp4_sqr(z4, z5)
    z4 = f2_add(f2_scale(f2_sub(t0, z4), 2), t0)
    z5 = f2_add(f2_scale(f2_add(t1, z5), 2), t1)
    t0 = f2_mul_xi(t3)
    z2 = f2_add(f2_scale(f2_add(t0, z2), 2), t0)
    z3 = f2_add(f2_scale(f2_sub(t2, z3), 2), t2)
    return ((z0, z4, z3), (z2, z1, z5))


def f12_pow(a, e):
    r = ONE
    for bit in bin(e)[2:]:
        r = f12_sqr(r)
        if bit == "1":
            r = f12_mul(r, a)
    return r


def exp_by_x(a):
    r = a
    for bit in bin(X)[3:]:
        r = f12_cyclotomic_sqr(r)
        if bit == "1":
            r = f12_mul(r, a)
    return r


def final_exponentiation(f):
    # easy part f^((p^6 - 1)(p^2 + 1))
    f = f12_mul(f12_conj(f), f12_inv(f))
    f = f12_mul(f12_frobenius(f, 2), f)
    # hard part (p^4 - p^2 + 1) / r: Scott, Benger, Charlemagne, Dominguez Perez, Kachisa (2009), section 6
    fx = exp_by_x(f)
    fx2 = exp_by_x(fx)
    fx3 = exp_by_x(fx2)
    y0 = f12_mul(f12_mul(f12_frobenius(f, 1), f12_frobenius(f, 2)), f12_frobenius(f, 3))
    y1 = f12_conj(f)
    y2 = f12_frobenius(fx2, 2)
    y3 = f12_conj(f12_frobenius(fx, 1))
    y4 = f12_conj(f12_mul(fx, f12_frobenius(fx2, 1)))
    y5 = f12_conj(fx2)
    y6 = f12_conj(f12_mul(fx3, f12_frobenius(fx3, 1)))
    t0 = f12_mul(f12_mul(f12_cyclotomic_sqr(y6), y4), y5)
    t1 = f12_mul(f12_mul(y3, y5), t0)
    t0 = f12_mul(t0, y2)
    t1 = f12_cyclotomic_sqr(f12_mul(f12_cyclotomic_sqr(t1), t0))
    t0 = f12_mul(t1, y1)
    t1 = f12_mul(t1, y0)
    t0 = f12_cyclotomic_sqr(t0)
    return f12_mul(t0, t1)


# ---- basis map to py_ecc's FQ12 = Fp[w]/(w^12 - 18 w^6 + 82), w^6 = 9 + u
def to_pyecc(a):
    g = _w_coeffs(a)
    out = [0] * 12
    for i, (x, y) in enumerate(g):
        out[i] = (x - 9 * y) % P
        out[i + 6] = y
    return out


def from_pyecc(c):
    return _from_w_coeffs([((c[i] + 9 * c[i + 6]) % P, c[i + 6] % P) for i in range(6)])


# ---- Miller loop (homogeneous projective coordinates on the D-type twist y^2 = x^3 + 3/xi)
def _dbl_step(T, xp, yp):
    X_, Y_, Z_ = T
    b3 = f2_mul((3, 0), f2_inv(XI))        # b' = 3/xi
    A = f2_mul(X_, Y_)
    B = f2_sqr(Y_)
    C = f2_sqr(Z_)
    E = f2_scale(f2_mul(b3, C), 3)          # 3 b' Z^2
    F = f2_scale(E, 3)
    H = f2_sub(f2_sqr(f2_add(Y_, Z_)), f2_add(B, C))   # 2 Y Z
    J = f2_sqr(X_)
    line = (f2_neg(f2_scale(H, yp)), f2_scale(J, 3 * xp), f2_sub(E, B))
    BF = f2_add(B, F)
    X3 = f2_scale(f2_mul(A, f2_sub(B, F)), 2)
    Y3 = f2_sub(f2_sqr(BF), f2_scale(f2_sqr(E), 12))
    Z3 = f2_scale(f2_mul(B, H), 4)
    return (X3, Y3, Z3), line


def _add_step(T, Q, xp, yp):
    X_, Y_, Z_ = T
    xq, yq = Q
    theta = f2_sub(Y_, f2_mul(yq, Z_))
    lam = f2_sub(X_, f2_mul(xq, Z_))
    C = f2_sqr(theta)
    D = f2_sqr(lam)
    E = f2_mul(lam, D)
    F = f2_mul(Z_, C)
    G = f2_mul(X_, D)
    H = f2_sub(f2_add(E, F), f2_scale(G, 2))
    X3 = f2_mul(lam, H)
    Y3 = f2_sub(f2_mul(theta, f2_sub(G, H)), f2_mul(Y_, E))
    Z3 = f2_mul(Z_, E)
    line = (f2_neg(f2_scale(lam, yp)), f2_scale(theta, xp), f2_sub(f2_mul(lam, yq), f2_mul(theta, xq)))
    return (X3, Y3, Z3), line


def twist_frobenius(Q, k):
    """pi^k on the twist: (x^(p^k) gamma_{k,2}, y^(p^k) gamma_{k,3})"""
    x, y = Q
    if k & 1:
        x, y = f2_conj(x), f2_conj(y)
    return (f2_mul(x, GAMMA[k - 1][2]), f2_mul(y, GAMMA[k - 1][3]))


def miller_loop(Q, Pt):
    if Q is None or Pt is None:
        return ONE
    xp, yp = Pt
    T = (Q[0], Q[1], F2_ONE)
    f = ONE
    for i in range(ATE.bit_length() - 2, -1, -1):
        T, l = _dbl_step(T, xp, yp)
        f = f12_mul_line(f12_sqr(f), *l)
        if (ATE >> i) & 1:
            T, l = _add_step(T, Q, xp, yp)
            f = f12_mul_line(f, *l)
    Q1 = twist_frobenius(Q, 1)
    Q2 = twist_frobenius(Q, 2)
    nQ2 = (Q2[0], f2_neg(Q2[1]))
    T, l = _add_step(T, Q1, xp, yp)
    f = f12_mul_line(f, *l)
    T, l = _add_step(T, nQ2, xp, yp)
    return f12_mul_line(f, *l)


def pairing(Q, Pt):
    return final_exponentiation(miller_loop(Q, Pt))
