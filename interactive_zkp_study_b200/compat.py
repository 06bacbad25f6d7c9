"""Field / point *types* of the boundary.

The reference returns py_ecc objects: G1 = (FQ, FQ), G2 = (FQ2, FQ2), Fr = FR(FQ) with
``field_modulus = curve_order`` (/root/reference/zkp/plonk/field.py:36-66).  When the real py_ecc is
importable (a deployment of the reference) those exact classes are used, so results interoperate
with the untouched parts of the reference (serializers, verifiers, ``bn128.is_on_curve``).  When it
is not (this image), a minimal stand-in with the same observable behaviour is defined here: these are
value containers for single elements (transcript challenges, a handful of scalars per proof), not a
compute path -- every vector / group operation goes to the GPU through ``native``.
"""

field_modulus = 21888242871839275222246405745257275088696311157297823662689037894645226208583
curve_order = 21888242871839275222246405745257275088548364400416034343698204186575808495617

try:  # pragma: no cover - exercised only where py_ecc is installed
    from py_ecc.fields import bn128_FQ as FQ, bn128_FQ2 as FQ2, bn128_FQ12 as FQ12
    from py_ecc import bn128 as _bn128
    HAVE_PY_ECC = True
    G1, G2 = _bn128.G1, _bn128.G2
except ImportError:
    HAVE_PY_ECC = False

    def _inv(a, m):
        a %= m
        return pow(a, -1, m) if a else 0  # py_ecc: inv(0) == 0

    class FQ(object):
        field_modulus = field_modulus

        def __init__(self, val):
            if isinstance(val, FQ):
                self.n = val.n
            elif isinstance(val, int):
                self.n = val % self.field_modulus
            else:
                raise TypeError("Expected an int or FQ object, but got object of type {}".format(type(val)))

        @staticmethod
        def _n(other):
            if isinstance(other, FQ):
                return other.n
            if isinstance(other, int):
                return other
            raise TypeError("Expected an int or FQ object, but got object of type {}".format(type(other)))

        def __add__(self, o):
            return type(self)(self.n + self._n(o))

        __radd__ = __add__

        def __sub__(self, o):
            return type(self)(self.n - self._n(o))

        def __rsub__(self, o):
            return type(self)(self._n(o) - self.n)

        def __mul__(self, o):
            return type(self)(self.n * self._n(o))

        __rmul__ = __mul__

        def __truediv__(self, o):
            return type(self)(self.n * _inv(self._n(o), self.field_modulus))

        def __rtruediv__(self, o):
            return type(self)(_inv(self.n, self.field_modulus) * self._n(o))

        def __pow__(self, e):
            return type(self)(pow(self.n, e, self.field_modulus))

        def __neg__(self):
            return type(self)(-self.n)

        def __eq__(self, o):
            return self.n == self._n(o)

        def __ne__(self, o):
            return not self == o

        __hash__ = None

        def __int__(self):
            return self.n

        def __repr__(self):
            return repr(self.n)

        @classmethod
        def one(cls):
            return cls(1)

        @classmethod
        def zero(cls):
            return cls(0)

    class FQ2(object):
        """a + b*u, u^2 = -1: container with the ``coeffs`` the serializers read
        (/root/reference/plonk_serializers.py:56-57)."""

        def __init__(self, coeffs):
            if len(coeffs) != 2:
                raise Exception("FQ2 takes two coefficients")
            self.coeffs = tuple(FQ(c) for c in coeffs)

        def __eq__(self, o):
            if not isinstance(o, FQ2):
                raise TypeError("Expected an FQ2 object")
            return self.coeffs[0] == o.coeffs[0] and self.coeffs[1] == o.coeffs[1]

        def __ne__(self, o):
            return not self == o

        __hash__ = None

        def __neg__(self):
            return FQ2([-self.coeffs[0].n, -self.coeffs[1].n])

        def __repr__(self):
            return repr(self.coeffs)

    class FQ12(object):
        """Element of Fp[w]/(w^12 - 18 w^6 + 82), py_ecc's pairing target: a value container for what
        zkp.pairing.pairing returns, with the product and the equality the verifiers' e(..) * e(..) == e(..)
        needs.  The pairings themselves run on the GPU (native.pairing)."""
        degree = 12

        def __init__(self, coeffs):
            if len(coeffs) != 12:
                raise Exception("FQ12 takes twelve coefficients")
            self.coeffs = tuple(FQ(c) for c in coeffs)

        def __mul__(self, o):
            if isinstance(o, (int, FQ)):
                return FQ12([c * o for c in self.coeffs])
            if not isinstance(o, FQ12):
                raise TypeError("Expected an FQ12, FQ or int")
            a = [c.n for c in self.coeffs]
            b = [c.n for c in o.coeffs]
            t = [0] * 23
            for i in range(12):
                for j in range(12):
                    t[i + j] += a[i] * b[j]
            for k in range(22, 11, -1):      # w^12 = 18 w^6 - 82
                t[k - 6] += 18 * t[k]
                t[k - 12] -= 82 * t[k]
            return FQ12(t[:12])

        __rmul__ = __mul__

        def __eq__(self, o):
            if not isinstance(o, FQ12):
                raise TypeError("Expected an FQ12 object")
            return all(x == y for x, y in zip(self.coeffs, o.coeffs))

        def __ne__(self, o):
            return not self == o

        __hash__ = None

        def __repr__(self):
            return repr(self.coeffs)

        @classmethod
        def one(cls):
            return cls([1] + [0] * 11)

        @classmethod
        def zero(cls):
            return cls([0] * 12)

    G1 = (FQ(1), FQ(2))
    G2 = (
        FQ2([10857046999023057135944570762232829481370756359578518086990519993285655852781,
             11559732032986387107991004021392285783925812861821192530917403151452391805634]),
        FQ2([8495653923123431417604973247489272438418190587263600148770280649306958101930,
             4082367875863433681332203403145435568316851327593401208105741076214120093531]),
    )


class FR(FQ):
    """Element of the BN254 scalar field, as every reference module declares it
    (zkp/plonk/field.py:36-51, zkp/groth16/poly_utils.py:12-13)."""
    field_modulus = curve_order


def g1_from_ints(p):
    return None if p is None else (FQ(p[0]), FQ(p[1]))


def g2_from_ints(p):
    return None if p is None else (FQ2([p[0][0], p[0][1]]), FQ2([p[1][0], p[1][1]]))


def is_g2(pt):
    return pt is not None and hasattr(pt[0], "coeffs")
