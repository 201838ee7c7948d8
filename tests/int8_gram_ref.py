"""
Exact references for the int8 Gram product of the Gaussian step's constant-weight SYRK (DESIGN §2, csrc/int8_gram.cu).

    A = rint(K * (2^52 / v))              0 <= A < 2^53, exact in a double (v = the kernel variance; K may exceed v by rounding)
    r_i = A mod p_i  (symmetric range)    16 pairwise coprime moduli, int8 planes
    C_i = R_i R_i^T  (int32, exact)       < 2^31 for fewer than 2^17 points per slab
    B' = CRT(C_i mod p_i)                 Garner digits + Horner, symmetric range: exact while |B'| < P / 2
    C = fl(C + fl(B') s),  s = ((alpha v) v) 2^-104     one rounding of the exact integer, one of the fused multiply-add

The NumPy functions model the scheme on small arrays.  The torch functions build what each kernel stage writes, byte for byte or
bit for bit, at the sizes the step runs; they take tensors on any device and stay exact there: every floating-point operation
on integers has all its partial sums below 2^53.
"""
import numpy as np
import torch

MODULI = [256, 255, 253, 251, 247, 241, 239, 233, 229, 227, 223, 217, 211, 199, 197, 193]
NMOD = len(MODULI)
P = int(np.prod([int(p) for p in MODULI], dtype=object))
GRID = 2.0 ** 52
MAX_POINTS = 2 ** 17 - 128   # widest slab the int32 accumulation takes (a multiple of 128 below 2^17), I8_MAX_COLS
KB_BYTES = 16384             # one 128-row x 128-byte k-block, and one 128 x 128 tile of residues


# ---- the scheme in NumPy ------------------------------------------------------------------------------------------------------
def grid(K, v):
    A = np.rint(np.asarray(K, dtype=np.float64) * (GRID / v))
    A[~np.isfinite(A)] = 0.0
    return A


def residues(A):
    """[16, rows, n] symmetric residues of the grid integers (what the int8 planes hold)."""
    Ai = A.astype(np.int64)
    out = []
    for p in MODULI:
        r = Ai % p
        r = np.where(r > (p - 1) // 2, r - p, r)   # [-128, 127] for 256, [-(p-1)/2, (p-1)/2] for odd p
        out.append(r.astype(np.int8))
    return np.stack(out)


def modular_gram(R):
    """C_i mod p_i in [0, p_i) from the int32-exact products of the residue planes."""
    out = []
    for p, r in zip(MODULI, R):
        c = r.astype(np.int64) @ r.astype(np.int64).T
        assert np.abs(c).max(initial=0) < 2 ** 31   # the tensor cores accumulate in int32
        out.append(c % p)
    return out


def crt(cs):
    """Garner's mixed-radix digits, then Horner; the integer in the symmetric range (-P/2, P/2)."""
    n = len(MODULI)
    shape = cs[0].shape
    out = np.empty(shape, dtype=object)
    inv = [[pow(MODULI[j], -1, MODULI[i]) if j < i else 0 for j in range(n)] for i in range(n)]
    for idx in np.ndindex(shape):
        v = []
        for i in range(n):
            t = int(cs[i][idx])
            for j in range(i):
                t = (t - v[j]) * inv[i][j] % MODULI[i]
            v.append(t)
        x = 0
        for i in reversed(range(n)):
            x = x * MODULI[i] + v[i]
        out[idx] = x - P if x > P // 2 else x
    return out


def exact_gram(A):
    """The exact integer A A^T from 18-bit limbs (int64 products summed exactly), combined in Python integers."""
    Ai = A.astype(np.int64)
    limbs = [(Ai >> (18 * k)) & ((1 << 18) - 1) for k in range(3)]
    out = np.zeros((A.shape[0], A.shape[0]), dtype=object)
    for a in range(3):
        for b in range(3):
            out = out + (limbs[a] @ limbs[b].T).astype(object) * (1 << (18 * (a + b)))
    return out


def to_double(B_int, v, alpha=1.0):
    return np.vectorize(lambda x: float(x))(B_int).astype(np.float64) * (alpha * v * v * 2.0 ** -104)


# ---- sizes and layout of the workspace ----------------------------------------------------------------------------------------
def plane_row_blocks(Mp):
    """Row blocks of one plane: Mp / 128 rounded up to even (the last 128 x 256 block of an odd tile row reads one past it)."""
    return (Mp // 128 + 1) & ~1


def plane_bytes(Mp, nc):
    return NMOD * (nc // 128) * plane_row_blocks(Mp) * KB_BYTES


def tile_bytes(Mp):
    nt = Mp // 128
    return NMOD * nt * (nt + 1) // 2 * KB_BYTES


def blocks_per_modulus(nt):
    """Lower 128 x 256 output blocks of one modulus: tile row i holds ceil((i + 1) / 2) of them."""
    return sum((i + 2) // 2 for i in range(nt))


def kblock_offsets():
    """[128, 128] byte offset of (row r, byte k) in a k-block: 8-row atoms of 1024 B, 16-byte chunk c of row r at c ^ (r & 7)."""
    r = np.arange(128)[:, None]
    k = np.arange(128)[None, :]
    return (r >> 3) * 1024 + (r & 7) * 128 + ((((k >> 4) ^ (r & 7)) << 4) | (k & 15))


# ---- stage references (torch) -------------------------------------------------------------------------------------------------
def grid_t(K, v):
    """The grid integers as the residue kernel forms them: rint(K * (2^52 / v)), off the grid (|A| >= 2^53, NaN) -> 0; int64."""
    t = torch.round(K * (GRID / v))   # round half to even, as rint
    return torch.where(t.abs() < 2.0 ** 53, t, torch.zeros_like(t)).to(torch.int64)


def residue_t(A, p):
    r = torch.remainder(A, p)   # [0, p)
    return torch.where(r > (p - 1) // 2, r - p, r)


def plane_image(A, nc_alloc):
    """uint8 [plane_bytes(Mp, nc_alloc)]: the residue planes of the grid integers A [Mp, ncols] as the residue kernel writes them
    after i8_planes_init.  Plane m at m * pstride holds k-block (kb, rb) at (kb * nrb + rb) * 16 KB in the kblock_offsets layout;
    the padding row block of an odd tile count and the k-blocks from ncols to nc_alloc are zero."""
    Mp, ncols = A.shape
    nrb, nkb = plane_row_blocks(Mp), ncols // 128
    off = torch.from_numpy(kblock_offsets().reshape(-1)).to(A.device)
    img = torch.zeros(NMOD, nc_alloc // 128, nrb, KB_BYTES, dtype=torch.uint8, device=A.device)
    for m, p in enumerate(MODULI):
        r = residue_t(A, p).to(torch.int8).view(torch.uint8)                      # two's complement bytes
        blocks = r.view(Mp // 128, 128, nkb, 128).permute(2, 0, 1, 3).reshape(nkb, Mp // 128, KB_BYTES)
        img[m, :nkb, :Mp // 128, off] = blocks
    return img.reshape(-1)


def residue_tiles(A):
    """uint8 [16, nt (nt + 1) / 2, 128, 128]: (R_m R_m^T) mod p_m on the lower 128-tiles (i, j <= i) at index i (i + 1) / 2 + j,
    as the products kernel writes them.  float64 products: every partial sum is an integer of magnitude < 2^31 < 2^53."""
    Mp = A.shape[0]
    nt = Mp // 128
    ii, jj = torch.tril_indices(nt, nt, device=A.device)   # row-major over the lower tiles: i (i + 1) / 2 + j
    out = torch.empty(NMOD, nt * (nt + 1) // 2, 128, 128, dtype=torch.uint8, device=A.device)
    for m, p in enumerate(MODULI):   # one modulus at a time bounds the memory
        r = residue_t(A, p).to(torch.float64)
        g = (r @ r.T).to(torch.int64)
        assert int(g.abs().max()) < 2 ** 31   # the tensor cores accumulate in int32
        g = torch.remainder(g, p).to(torch.uint8).view(nt, 128, nt, 128).permute(0, 2, 1, 3)
        out[m] = g[ii, jj]
    return out


def limbs_of(A):
    """A (int64, |A| < 2^53) = L_0 + L_1 2^18 + L_2 2^36 as float64 limbs: two 18-bit ones, the top one signed and below 2^17."""
    return [((A >> s) & ((1 << 18) - 1) if s < 36 else A >> s).to(torch.float64) for s in (0, 18, 36)]


def exact_gram_rows(limbs, r0, r1, c1):
    """The exact integers (A A^T)[r0:r1, 0:c1] as a NumPy object array of Python ints.  Each limb Gram L_a L_b^T is an exact
    float64 product (terms below 2^36, fewer than 2^17 of them); the limb Grams are combined in Python integers."""
    out = 0
    for a in range(3):
        for b in range(3):
            g = (limbs[a][r0:r1] @ limbs[b][:c1].T).to(torch.int64).cpu().numpy()
            out = out + g.astype(object) * (1 << (18 * (a + b)))
    return out


def syrk_scale(v, alpha):
    """The launcher's scale of the exact integer, in its order of evaluation."""
    return alpha * v * v * 2.0 ** -104


def fma(a, b, c):
    """fl(a b + c) with one rounding, as the device's fma: the exact sum as a ratio of integers, and Python's int / int true
    division is correctly rounded (to nearest, ties to even)."""
    (na, da), (nb, db), (nc, dc) = a.as_integer_ratio(), b.as_integer_ratio(), c.as_integer_ratio()
    return (na * nb * dc + nc * da * db) / (da * db * dc)


def syrk_model(A, C0, v, alpha):
    """float64 [Mp, ldc] (NumPy): C0 with every lower-tile entry replaced by  fl(C0 + fl(B') s)  (one rounding, fma) for the exact
    integer B' = (A A^T)[i, j] rounded once to double by Python's float(int) (to nearest, ties to even).  Other entries of C0 are
    returned as they are: the reconstruction kernel must not touch them."""
    Mp = A.shape[0]
    s = syrk_scale(v, alpha)
    out = np.array(C0, dtype=np.float64, copy=True)
    to_f = np.frompyfunc(float, 1, 1)
    fma_f = np.frompyfunc(fma, 3, 1)
    limbs = limbs_of(A)
    for i in range(Mp // 128):   # tile row i: its lower tiles and the full diagonal tile
        r0, r1, c1 = 128 * i, 128 * (i + 1), 128 * (i + 1)
        d = to_f(exact_gram_rows(limbs, r0, r1, c1)).astype(np.float64)
        c = out[r0:r1, :c1]
        nz = c != 0.0
        # C0 = 0: fma rounds the product alone, and the sum with 0 keeps IEEE's sign of zero (+0 + -0 = +0 when fl(B') s = -0)
        new = c + d * s
        new[nz] = fma_f(d[nz], s, c[nz]).astype(np.float64)
        out[r0:r1, :c1] = new
    return out


def largest_on_grid(v):
    """The largest double K with rint(K * (2^52 / v)) < 2^53, searched down from 2 v: the grid's headroom above the variance."""
    scale = GRID / v
    x = 2.0 * v
    while np.rint(x * scale) >= 2.0 ** 53:
        x = np.nextafter(x, 0.0)
    return x


def residues_of(x):
    """The 16 residues x mod p_i in [0, p_i) of a Python integer (what a reconstruction input tile holds for it)."""
    return [x % p for p in MODULI]
