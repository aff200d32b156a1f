"""Parameter points between and around the named sets: the shapes the C ABI accepts (check_params in csrc/c_api.cu) that the kernel
dispatcher routes to each blind-rotation kernel, at LWE dimensions, base logs and level counts no named set has.  Shared by
test_param_range_premise.py (CPU: the lattice premise of DESIGN section 4 at every point) and test_gpu_param_range.py (every kernel
instance word for word against the exact rotation).

A point is a plain orc.Params (noise fields 0: nothing is encrypted) plus the lattice-key settings of its test.  Every point uses the
default lattice key (nnz = 8 nonzeros per polynomial, |c| <= cmax = 127); a point that needs a thinner key to keep the f64 premise
records the change and its reason here."""
from dataclasses import dataclass

# keyswitch fields of every blind-rotation point: the context needs a valid decomposition, the rotation tests never upload a KSK
_KS = dict(ks_base_log=4, ks_level=3)


@dataclass(frozen=True)
class Point:
    family: str          # "classic" (pbs_v4 / pbs_v8 / pbs_v8x2), "multibit" (pbs_multibit_v4 / v8 / v8x2), "n512", "n8192", "generic"
    n: int
    N: int
    k: int
    B: int
    l: int
    g: int = 0
    nnz: int = 8
    cmax: int = 127
    why: str = ""        # reason for a non-default nnz / cmax

    @property
    def id(self):
        g = f"_g{self.g}" if self.g else ""
        return f"{self.family}_N{self.N}_k{self.k}_n{self.n}_B{self.B}_l{self.l}{g}"

    def params(self, orc):
        p = orc.Params()
        p.lwe_dim, p.glwe_dim, p.poly_size, p.pbs_base_log, p.pbs_level = self.n, self.k, self.N, self.B, self.l
        p.ks_base_log, p.ks_level = _KS["ks_base_log"], _KS["ks_level"]
        p.grouping_factor, p.msg_mod, p.carry_mod = self.g, 4, 4
        return p


def _cross(family, ns, Bs, n0, B0, extra=(), **kw):
    """n0 with every B, B0 with every n, and the extra (n, B) pairs: not the full product"""
    pairs = [(n0, B) for B in Bs] + [(n, B0) for n in ns if n != n0] + list(extra)
    return [Point(family, n, B=B, **kw) for n, B in dict.fromkeys(pairs)]


# N = 2048, k = 1, l = 1: pbs_v4 <1..4>, pbs_v8, pbs_v8x2.  Small n sit around the key-ring depths and the 4 ring pieces per iteration
# of pbs_v4; above 742 odd and even row strides n + 1 (the fused u16 input).
CLASSIC = _cross("classic", [1, 2, 3, 4, 5, 7, 8, 11, 12, 742, 745, 1023, 1024, 4096], [2, 3, 8, 15, 16, 22, 23, 24, 29, 30], 742, 23,
                 extra=[(1, 30), (4096, 2), (4096, 30)], N=2048, k=1, l=1)
# grouping factor 3, N = 2048: pbs_multibit_v4 <1..3>, v8, v8x2
MULTIBIT = _cross("multibit", [3, 6, 9, 12, 15, 888, 4095], [2, 8, 16, 21, 24, 30], 888, 21, N=2048, k=1, l=1, g=3)
# N = 512, k = 3, l = 1: pbs_n512 <1, 4, 8>
N512 = [Point("n512", n, 512, 3, B, 1) for n in (1, 5, 684, 4096) for B in (2, 9, 18, 30)]
# N = 8192, k = 1, l = 2: pbs_n8192 while 2 B <= 31, pbs_generic above (signed_digits2 is 32-bit)
N8192 = [Point("n8192", 864, 8192, 1, B, 2) for B in (2, 8, 15, 16, 20, 26)] + [Point("n8192", n, 8192, 1, 15, 2) for n in (1, 2, 3)]
# pbs_generic: every level count at the B * l = 52 edge (l = 1 at the largest base, 30), on three (N, k); multi-bit g = 2 at N = 2048
# and g = 3 at N = 512
_EDGE = [(30, 1), (26, 2), (17, 3), (13, 4), (10, 5), (8, 6), (7, 7), (6, 8)]
GENERIC = ([Point("generic", 130, N, k, B, l) for N, k in ((256, 5), (512, 2), (1024, 2)) for B, l in _EDGE]
           + [Point("generic", n, 2048, 1, 22, 1, g=2) for n in (2, 818, 4096)]
           + [Point("generic", n, 512, 3, 18, 1, g=3) for n in (3, 765)])

ROTATION_POINTS = CLASSIC + MULTIBIT + N512 + N8192 + GENERIC


def engine_dict(orc, point):
    from helpers import engine_params
    return engine_params(point.params(orc))
