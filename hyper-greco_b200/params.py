"""BFV secret-key-encryption parameter sets (data only).

Values are the per-parameter-set constants the reference generates into
/root/reference/bfv-gkr/src/constants/sk_enc_constants_*.rs (trait `BfvSkEncryptConstans`,
/root/reference/bfv-gkr/src/constants/mod.rs:16-35). `K` = number of CRT moduli (`num_reps`).
"""
from dataclasses import dataclass
from typing import List

LIMB_BITS = 16  # sk_encryption_circuit.rs:29
C = 4           # sk_encryption_circuit.rs:30
M = 1 << LIMB_BITS  # sk_encryption_circuit.rs:31


@dataclass(frozen=True)
class BfvSkEncryptConstants:
    name: str
    N: int
    E_BOUND: int
    S_BOUND: int
    K1_BOUND: int
    R1_BOUNDS: tuple
    R2_BOUNDS: tuple
    QIS: tuple
    K0IS: tuple

    @property
    def K(self) -> int:
        return len(self.QIS)

    @property
    def N_LOG2(self) -> int:
        return self.N.bit_length() - 1

    @property
    def log2_size(self) -> int:  # sk_encryption_circuit.rs:81-83
        return self.N_LOG2 + 1


PARAMS = {
    "1024_1x27_65537": BfvSkEncryptConstants(
        name="1024_1x27_65537", N=1024, E_BOUND=19, S_BOUND=1, K1_BOUND=32768,
        R1_BOUNDS=(1246,),
        R2_BOUNDS=(41319090,),
        QIS=(82638181,),
        K0IS=(1849798,),
    ),
    "2048_1x52_65537": BfvSkEncryptConstants(
        name="2048_1x52_65537", N=2048, E_BOUND=19, S_BOUND=1, K1_BOUND=32768,
        R1_BOUNDS=(29882,),
        R2_BOUNDS=(1434875766359798,),
        QIS=(2869751532719597,),
        K0IS=(2527239722765942,),
    ),
    "4096_2x55_65537": BfvSkEncryptConstants(
        name="4096_2x55_65537", N=4096, E_BOUND=19, S_BOUND=1, K1_BOUND=32768,
        R1_BOUNDS=(25966, 19503),
        R2_BOUNDS=(13712101976447600, 13712101976447600),
        QIS=(27424203952895201, 27424203952895203),
        K0IS=(20017153978526555, 14608220699689817),
    ),
    "8192_4x55_65537": BfvSkEncryptConstants(
        name="8192_4x55_65537", N=8192, E_BOUND=19, S_BOUND=1, K1_BOUND=32768,
        R1_BOUNDS=(28014, 21551, 24676, 29416),
        R2_BOUNDS=(13712101976447600, 13712101976447600, 13712101976447602, 13712101976447604),
        QIS=(27424203952895201, 27424203952895203, 27424203952895205, 27424203952895207),
        K0IS=(20017153978526555, 14608220699689817, 17223556688605927, 21190079862835656),
    ),
    "16384_8x54_65537": BfvSkEncryptConstants(
        name="16384_8x54_65537", N=16384, E_BOUND=19, S_BOUND=1, K1_BOUND=32768,
        R1_BOUNDS=(16113, 24818, 37593, 34517, 12912, 32948, 38917, 29910),
        R2_BOUNDS=(6452516132120967, 6452516132120968, 6452516132120969, 6452516132120970, 6452516132120973, 6452516132120975, 6452516132120976, 6452516132120978),
        QIS=(12905032264241935, 12905032264241937, 12905032264241939, 12905032264241941, 12905032264241947, 12905032264241951, 12905032264241953, 12905032264241957),
        K0IS=(3119285534855982, 6547723161734179, 11578631950954274, 10367425251572977, 1858653883183236, 9749317979689080, 12100252264181577, 8552879692347062),
    ),
    "32768_16x59_65537": BfvSkEncryptConstants(
        name="32768_16x59_65537", N=32768, E_BOUND=19, S_BOUND=1, K1_BOUND=32768,
        R1_BOUNDS=(17449, 44739, 23337, 23971, 38527, 41231, 47178, 25438, 29323, 21130, 36215, 41226, 47080, 20341, 18613, 40562),
        R2_BOUNDS=(238750987231488128, 238750987231488128, 238750987231488128, 238750987231488128, 238750987231488128, 238750987231488128, 238750987231488128, 238750987231488128, 238750987231488160, 238750987231488160, 238750987231488160, 238750987231488160, 238750987231488160, 238750987231488160, 238750987231488160, 238750987231488192),
        QIS=(477501974462976263, 477501974462976265, 477501974462976267, 477501974462976269, 477501974462976271, 477501974462976277, 477501974462976283, 477501974462976289, 477501974462976293, 477501974462976299, 477501974462976301, 477501974462976307, 477501974462976311, 477501974462976313, 477501974462976317, 477501974462976361),
        K0IS=(15519160254606397, 413181248299753132, 101318987089463173, 110550337344198528, 322660099471945682, 362070023329770101, 448729597070750619, 131927434145614106, 188539582116643080, 69158624007851611, 288969678337063080, 361989877431741640, 447294256896967800, 57654044645399264, 32480946673725505, 352321367733214595),
    ),
}


def by_n(n: int) -> BfvSkEncryptConstants:
    for p in PARAMS.values():
        if p.N == n:
            return p
    raise KeyError(n)


# ----------------------------------------------------------------------------- public-key encryption
@dataclass(frozen=True)
class BfvPkEncryptConstants:
    """Bounds of the BFV public-key-encryption relation (for every modulus i, over Z[x]):
        ct0_i = pk0_i u + e0 + k0_i k1 + r1_i q_i + r2_i (x^n + 1)
        ct1_i = pk1_i u + e1           + p1_i q_i + p2_i (x^n + 1)
    Derived from the SK set of the same name (pk_from_sk)."""
    name: str
    N: int
    E_BOUND: int
    U_BOUND: int
    K1_BOUND: int
    R1_BOUNDS: tuple
    R2_BOUNDS: tuple
    P1_BOUNDS: tuple
    P2_BOUNDS: tuple
    QIS: tuple
    K0IS: tuple

    @property
    def K(self) -> int:
        return len(self.QIS)

    @property
    def N_LOG2(self) -> int:
        return self.N.bit_length() - 1

    @property
    def log2_size(self) -> int:
        return self.N_LOG2 + 1


def quotient_bound(n: int, q: int, u_bound: int, e_bound: int, extra: int = 0) -> int:
    """Bound on the q-quotient of pk u + e (+ extra) - ct: floor((n h U + E + extra + 2h) / q), h = (q - 1) / 2. With
    extra = K1_BOUND k0_i it reproduces every SK R1_BOUNDS entry; with extra = 0 it is the PK P1 bound."""
    h = (q - 1) // 2
    return (n * h * u_bound + e_bound + extra + 2 * h) // q


def pk_from_sk(sk: BfvSkEncryptConstants) -> BfvPkEncryptConstants:
    """N, QIS, K0IS, E_BOUND, K1_BOUND as they are; U_BOUND = S_BOUND; R1 = SK R1; R2 = P2 = SK R2 (kept as given: at n = 32768
    they differ from (q - 1) / 2 by the float rounding of the generator that produced them); P1 by quotient_bound."""
    return BfvPkEncryptConstants(
        name=sk.name, N=sk.N, E_BOUND=sk.E_BOUND, U_BOUND=sk.S_BOUND, K1_BOUND=sk.K1_BOUND,
        R1_BOUNDS=sk.R1_BOUNDS, R2_BOUNDS=sk.R2_BOUNDS,
        P1_BOUNDS=tuple(quotient_bound(sk.N, q, sk.S_BOUND, sk.E_BOUND) for q in sk.QIS), P2_BOUNDS=sk.R2_BOUNDS,
        QIS=sk.QIS, K0IS=sk.K0IS)


PK_PARAMS = {name: pk_from_sk(p) for name, p in PARAMS.items()}
