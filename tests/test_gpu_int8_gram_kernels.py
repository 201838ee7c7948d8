"""
The int8 Gram product of the Gaussian step (csrc/int8_gram.cu, DESIGN §2) checked bit for bit, stage by stage, against the exact
integer references of tests/int8_gram_ref.py.  The product claims exactness: the integer A A^T is formed exactly and rounded to
double once, so every stage is compared for equality:

    residues        the int8 planes, byte for byte (every modulus, every row block, the padding block of an odd tile count)
    products        the residue tiles (R_m R_m^T) mod p_m, byte for byte (every modulus, every lower tile)
    reconstruction  C = fl(C + fl(B') s) for chosen integers B' (ties, sticky bits, the hi / lo word boundary, +-(P/2 - 1))
    launcher        i8_syrk_launch end to end: every lower-tile entry against the exact model, every other entry of C untouched

The kernels run through a small shim (tests/kernels/int8_gram_shim.cu) that this file compiles with nvcc; the refusal and size
tests need nvcc but no GPU.
"""
import ctypes
import os
import random
import shutil
import subprocess

import numpy as np
import pytest
import torch

from tests import int8_gram_ref as ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHIM = os.path.join(ROOT, "tests", "kernels", "int8_gram_shim.cu")
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC", "-shared"]   # csrc/Makefile
CUDA_ERROR_INVALID_VALUE = 1
VARIANCES = [2.0 ** -20, 1e-6, 0.6, 1.3, 7.0, 1e6]
ALPHAS = [-3.5, -1e-8, 1.0, -0.5 / 0.3]   # the last is the Gaussian step's weight -1/(2 s2) at s2 = 0.3


@pytest.fixture(scope="session")
def shim(tmp_path_factory):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not os.path.exists(nvcc):
        nvcc = shutil.which("nvcc") or nvcc
    out = str(tmp_path_factory.mktemp("int8_gram_shim") / "libi8shim.so")
    r = subprocess.run([nvcc, *NVCC_FLAGS, "-o", out, SHIM], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lib = ctypes.CDLL(out)
    vp, i, l, d, sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_long, ctypes.c_double, ctypes.c_size_t
    for name, args, res in [
        ("i8_syrk_launch", [vp, l, i, i, d, d, vp, l, vp, vp, l, vp], i),
        ("i8_planes_init", [vp, i, l, vp], i),
        ("i8_plane_bytes", [i, l], sz),
        ("i8_tile_bytes", [i], sz),
        ("i8_residue_launch", [vp, l, d, vp, sz, i, i, i, vp], i),
        ("i8_gram_launch", [vp, sz, i, i, i, vp, sz, vp], i),
        ("i8_crt_launch", [vp, sz, vp, l, d, vp], i),
    ]:
        f = getattr(lib, name)
        f.argtypes, f.restype = args, res
    return lib


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _ok(rc):
    assert rc == 0, f"CUDA error {rc}"


def _geometry(Mp, ncols, nc_alloc):
    """The arguments i8_syrk_launch derives for its three kernels."""
    nt, nrb = Mp // 128, ref.plane_row_blocks(Mp)
    return dict(nt=nt, nrb=nrb, nkb=ncols // 128, nblk=ref.blocks_per_modulus(nt),
                pstride=(nc_alloc // 128) * nrb * ref.KB_BYTES, tstride=nt * (nt + 1) // 2 * ref.KB_BYTES)


def _specials(v):
    """Entries at the edges of the grid: 0, exactly v, just above v by rounding, the largest double still below 2^53 on the grid,
    and the non-finite values that map to 0."""
    return [0.0, v, float(np.nextafter(v, np.inf)), v * (1 + 2.0 ** -50), ref.largest_on_grid(v), np.nan, np.inf, -np.inf]


def _slab(Mp, ncols, ldk, v, seed):
    """K [Mp, ldk] on the device: the skewed v u^2 of a covariance slab, rows 0-2 all at the grid's top / v / 0, row 3 cycling
    through the special entries, 2% of the rest special too.  Columns from ncols to ldk hold v * 0.77: read, they would count."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    u = torch.rand(Mp, ncols, generator=g, device="cuda", dtype=torch.float64)
    K = v * u * u
    sp = torch.tensor(_specials(v), device="cuda", dtype=torch.float64)
    K[0], K[1], K[2] = sp[4], v, 0.0
    K[3] = sp[torch.arange(ncols, device="cuda") % len(sp)]
    pick = torch.rand(Mp, ncols, generator=g, device="cuda") < 0.02
    pick[:4] = False
    K[pick] = sp[torch.randint(0, len(sp), (int(pick.sum()),), generator=g, device="cuda")]
    out = torch.full((Mp, ldk), v * 0.77, device="cuda", dtype=torch.float64)
    out[:, :ncols] = K
    return out


def _int32_bound_slab(Mp, ncols, seed):
    """v = 2^-20 (K 2^72 exact): rows 0-3 have A = 256 k + 128, residue -128 mod 256 in every column, so their mod-256 products
    reach ncols 2^14 = 2^31 - 2^21 at ncols = I8_MAX_COLS; the other rows are a covariance slab with the special entries."""
    v = 2.0 ** -20
    K = _slab(Mp, ncols, ncols, v, seed)
    g = torch.Generator(device="cuda").manual_seed(seed + 1)
    k = torch.randint(0, 2 ** 44, (4, ncols), generator=g, device="cuda", dtype=torch.int64)
    K[:4] = (256 * k + 128).to(torch.float64) * 2.0 ** -72
    return K, v


def _lower_mask(Mp, ldc, device="cuda"):
    """The entries the product writes: lower 128-tiles, diagonal tiles in full, no column at or past Mp."""
    r = torch.arange(Mp, device=device)[:, None] // 128
    c = torch.arange(ldc, device=device)[None, :]
    return (c < Mp) & (c // 128 <= r)


def _sentinel_C(Mp, ldc, seed, lower=None):
    """C0 [Mp, ldc]: tiny distinct values outside the lower tiles (any write to them shows), `lower` (default 0) on them."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    C = (1.0 + torch.rand(Mp, ldc, generator=g, device="cuda", dtype=torch.float64)) * 2.0 ** -1000
    m = _lower_mask(Mp, ldc)
    C[m] = 0.0 if lower is None else lower[m]
    return C


def _assert_bitwise(got, want, Mp, what):
    got, want = np.ascontiguousarray(got), np.ascontiguousarray(want)
    bad = np.argwhere(got.view(np.int64) != want.view(np.int64))
    if len(bad):
        ldc = got.shape[1]
        lower = lambda i, j: j < Mp and j // 128 <= i // 128
        where = [(int(i), int(j), "lower" if lower(i, j) else "untouched", float(got[i, j]), float(want[i, j])) for i, j in bad[:8]]
        n_low = int(((bad[:, 1] < Mp) & (bad[:, 1] // 128 <= bad[:, 0] // 128)).sum())
        pytest.fail(f"{what}: {len(bad)} of {got.size} entries differ ({n_low} in lower tiles, ldc {ldc}); first (row, col, region, "
                    f"got, want): {where}")


def _syrk(shim, K, Mp, ncols, v, alpha, planes, nc_alloc, tiles, C, stream):
    _ok(shim.i8_syrk_launch(K.data_ptr(), K.stride(0), Mp, ncols, v, alpha, planes.data_ptr(), nc_alloc, tiles.data_ptr(),
                            C.data_ptr(), C.stride(0), stream))


def _workspace(shim, Mp, nc_alloc, stream):
    """Planes and tiles filled with 0xA5 first: nothing may rely on memory that i8_planes_init and the kernels do not write."""
    planes = torch.full((ref.plane_bytes(Mp, nc_alloc),), 0xA5, dtype=torch.uint8, device="cuda")
    tiles = torch.full((ref.tile_bytes(Mp),), 0xA5, dtype=torch.uint8, device="cuda")
    torch.cuda.current_stream().synchronize()
    _ok(shim.i8_planes_init(planes.data_ptr(), Mp, nc_alloc, stream))
    return planes, tiles


# ---- without a GPU: sizes and refusals ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("Mp", [128, 256, 384, 1536, 1664, 4096, 8192])
def test_workspace_sizes(shim, Mp):
    for nc in (128, 640, 16384, ref.MAX_POINTS):
        assert shim.i8_plane_bytes(Mp, nc) == ref.plane_bytes(Mp, nc)
    assert shim.i8_tile_bytes(Mp) == ref.tile_bytes(Mp)


@pytest.mark.parametrize("Mp,ncols,nc_alloc,ldk,ldc", [
    (256, 0, 1024, 1024, 256), (256, -128, 1024, 1024, 256), (256, 200, 1024, 1024, 256),       # ncols <= 0, not a multiple of 128
    (256, ref.MAX_POINTS + 128, 1 << 17, 1 << 17, 256),                                          # above I8_MAX_COLS
    (256, 512, 384, 1024, 256),                                                                  # above nc_alloc
    (200, 512, 1024, 1024, 256),                                                                 # Mp % 128 != 0
    (256, 512, 1024, 1023, 256), (256, 512, 1024, 1024, 257),                                    # odd ldk, odd ldc
], ids=["ncols_0", "ncols_negative", "ncols_not_128", "ncols_above_max", "ncols_above_alloc", "Mp_not_128", "ldk_odd", "ldc_odd"])
def test_launcher_refuses_bad_arguments(shim, Mp, ncols, nc_alloc, ldk, ldc):
    # the launcher checks its arguments before any CUDA call: host buffers stand in for the device ones, and C stays as it was
    K = np.full(16, 0.5)
    planes, tiles = np.zeros(16, np.int8), np.zeros(16, np.uint8)
    C = np.random.default_rng(0).standard_normal(64)
    C0 = C.copy()
    rc = shim.i8_syrk_launch(K.ctypes.data, ldk, Mp, ncols, 1.3, -3.5, planes.ctypes.data, nc_alloc, tiles.ctypes.data,
                             C.ctypes.data, ldc, None)
    assert rc == CUDA_ERROR_INVALID_VALUE
    assert np.array_equal(C.view(np.int64), C0.view(np.int64))


def test_references_agree_with_the_numpy_model():
    # the torch stage references against the NumPy model of the scheme (test_int8_gram_cpu.py), on the CPU
    v = 0.6
    rng = np.random.default_rng(5)
    K = v * rng.uniform(0, 1, (384, 256)) ** 2
    K[0, :8] = _specials(v)
    K[5] = 0.0   # exact zero entries: with alpha < 0 the product is -0, and fl(0 + -0) = +0
    A = ref.grid_t(torch.from_numpy(K), v)
    An = ref.grid(K, v)
    assert np.array_equal(A.numpy(), An.astype(np.int64))
    R = ref.residues(An)
    img = ref.plane_image(A, 384).view(ref.NMOD, 3, 4, 128 * 128).numpy()
    off = ref.kblock_offsets()
    for m in range(ref.NMOD):
        for kb in range(2):
            for rb in range(3):
                assert np.array_equal(img[m, kb, rb][off].view(np.int8), R[m, 128 * rb:128 * rb + 128, 128 * kb:128 * kb + 128])
    assert not img[:, :, 3].any() and not img[:, 2].any()   # the padding row block and the k-block beyond ncols
    tiles = ref.residue_tiles(A).numpy()
    mg = ref.modular_gram(R)
    for m in range(ref.NMOD):
        for t, (i, j) in enumerate((i, j) for i in range(3) for j in range(i + 1)):
            assert np.array_equal(tiles[m, t], mg[m][128 * i:128 * i + 128, 128 * j:128 * j + 128])
    C = ref.syrk_model(A, np.zeros((384, 384)), v, -3.5)
    want = 0.0 + ref.to_double(ref.exact_gram(An), v, alpha=-3.5)   # C0 + fl(B') s with C0 = 0
    low = _lower_mask(384, 384, "cpu").numpy()
    assert np.array_equal(C[low].view(np.int64), want[low].view(np.int64)) and not C[~low].any()
    zeros = C[low][C[low] == 0.0]
    assert len(zeros) and not np.signbit(zeros).any()
    assert ref.largest_on_grid(v) > v and np.rint(np.nextafter(ref.largest_on_grid(v), np.inf) * (ref.GRID / v)) >= 2.0 ** 53


def test_reference_fma_rounds_once():
    # the model of the reconstruction's C + fl(B') s against exact rational arithmetic, and distinct from two roundings
    from fractions import Fraction
    rng = np.random.default_rng(9)
    a, b, c = (rng.uniform(-1, 1, 2000) * 2.0 ** rng.integers(-60, 60, 2000) for _ in range(3))
    got = [ref.fma(float(x), float(y), float(z)) for x, y, z in zip(a, b, c)]
    assert got == [float(Fraction(x) * Fraction(y) + Fraction(z)) for x, y, z in zip(a, b, c)]
    assert ref.fma(1.0 + 2.0 ** -30, 1.0 - 2.0 ** -30, -1.0) == -(2.0 ** -60) != (1.0 + 2.0 ** -30) * (1.0 - 2.0 ** -30) - 1.0


def test_cases_separate_the_scale_orders():
    # the end-to-end cases include (alpha, v) pairs where alpha (v v) 2^-104 differs from the launcher's ((alpha v) v) 2^-104
    pairs = {(v, a) for _, _, _, _, v, a in E2E_CASES}
    assert {v for v, _ in pairs} == set(VARIANCES) and {a for _, a in pairs} == set(ALPHAS)
    assert any(a * v * v * 2.0 ** -104 != a * (v * v) * 2.0 ** -104 for v, a in pairs)


# ---- stage 1: residues ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("Mp,ncols,nc_alloc,v", [(128, 384, 640, 1.3), (384, 640, 640, 2.0 ** -20), (1536, 512, 512, 7.0),
                                                 (1664, 1024, 1280, 1e-6)])
def test_residue_planes_are_the_reference_image(shim, Mp, ncols, nc_alloc, v):
    s = _stream()
    K = _slab(Mp, ncols, nc_alloc, v, seed=Mp + ncols)
    planes, _ = _workspace(shim, Mp, nc_alloc, s)
    g = _geometry(Mp, ncols, nc_alloc)
    _ok(shim.i8_residue_launch(K.data_ptr(), nc_alloc, ref.GRID / v, planes.data_ptr(), g["pstride"], g["nrb"], g["nkb"], g["nt"], s))
    torch.cuda.synchronize()
    want = ref.plane_image(ref.grid_t(K[:, :ncols], v), nc_alloc)
    bad = torch.nonzero(planes != want)
    if len(bad):
        m, rest = divmod(int(bad[0]), g["pstride"])
        kb, rest = divmod(rest, g["nrb"] * ref.KB_BYTES)
        pytest.fail(f"{len(bad)} plane bytes differ; first at modulus {m}, k-block {kb}, row block {rest // ref.KB_BYTES}, "
                    f"byte {rest % ref.KB_BYTES}")


# ---- stage 2: products ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("Mp,ncols", [(128, 128), (128, 640), (256, 384), (256, 512), (384, 640), (1664, 2048), (4096, 512)])
def test_residue_tiles_are_the_exact_modular_products(shim, Mp, ncols):
    # planes from the reference image (this stage alone); one k-block past ncols holds garbage the products must not read
    s = _stream()
    nc_alloc = ncols + 128
    A = ref.grid_t(_slab(Mp, ncols, ncols, 1.3, seed=7 * Mp + ncols), 1.3)
    A[-1] = 256 * (A[-1] // 256) + 128   # residue -128 mod 256 along a whole row
    g = _geometry(Mp, ncols, nc_alloc)
    planes = ref.plane_image(A, nc_alloc).view(ref.NMOD, nc_alloc // 128, g["nrb"], ref.KB_BYTES)
    planes[:, -1] = torch.randint(0, 256, planes[:, -1].shape, dtype=torch.uint8, device="cuda")
    tiles = torch.full((ref.tile_bytes(Mp),), 0xA5, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    _ok(shim.i8_gram_launch(planes.data_ptr(), g["pstride"], g["nrb"], g["nkb"], g["nblk"], tiles.data_ptr(), g["tstride"], s))
    torch.cuda.synchronize()
    want = ref.residue_tiles(A)
    got = tiles.view(want.shape)
    bad = torch.nonzero(got != want)
    if len(bad):
        m, t, r, c = (int(x) for x in bad[0])
        i = int((np.sqrt(8 * t + 1) - 1) // 2)
        pytest.fail(f"{len(bad)} residue bytes differ; first at modulus {m}, tile ({i}, {t - i * (i + 1) // 2}), row {r}, col {c}: "
                    f"{int(got[m, t, r, c])} != {int(want[m, t, r, c])}")


# ---- stage 3: reconstruction ---------------------------------------------------------------------------------------------------
P2 = ref.P // 2
CRT_INTEGERS = [
    0, 1, -1,
    2 ** 53 - 1, -(2 ** 53 - 1), 2 ** 53, -(2 ** 53),
    2 ** 53 + 1,                        # a tie: rounds to even, down
    2 ** 53 + 3,                        # a tie: rounds to even, up
    2 ** 64 - 1, 2 ** 64,               # the hi / lo word boundary
    2 ** 64 + 2 ** 11,                  # a tie, round bit in the low word
    2 ** 64 + 2 ** 11 + 1,              # ... decided by the bit shifted out of the low word (sticky)
    2 ** 100 + 2 ** 47,                 # an exact tie: rounds down to even
    2 ** 100 + 2 ** 47 + 1,             # the only bit that decides is in the shifted-out low word
    -(2 ** 100 + 2 ** 47 + 1),
    2 ** 100 + 2 ** 48 + 2 ** 47,       # a tie: rounds up to even
    P2 - 1, -(P2 - 1),                  # the ends of the symmetric range
    ref.MAX_POINTS * (2 ** 53 - 1) ** 2,   # the largest Gram entry of the widest slab
]


@pytest.mark.gpu
def test_reconstruction_rounds_the_exact_integer_once(shim):
    # synthetic residue tiles at nt = 64 (2080 tiles): the chosen integers in tiles at both ends and in the middle, random integers
    # of 54 to 123 bits in three tiles, and elsewhere a value that names its tile and entry, so the tile decoding is checked too.
    # scale 1 and C0 = 0: the output is Python's float(x)
    Mp = 8192
    nt = Mp // 128
    T = nt * (nt + 1) // 2
    base = torch.arange(T * ref.KB_BYTES, device="cuda", dtype=torch.int64).view(T, ref.KB_BYTES) + 1
    base[1::2] = -base[1::2]
    ints = {}
    for t in (0, 1, T // 2, T - 2, T - 1):
        for e, x in enumerate(CRT_INTEGERS):
            ints[(t, 977 * e % ref.KB_BYTES)] = x
    rnd = random.Random(3)
    for t in (2, T // 3, T - 3):
        for e in range(ref.KB_BYTES):
            x = rnd.getrandbits(rnd.randint(54, 123))
            ints[(t, e)] = -x if rnd.random() < 0.5 else x
    tiles = torch.stack([torch.remainder(base, p) for p in ref.MODULI]).to(torch.uint8)   # [16, T, 16384]
    want_t = base.to(torch.float64)   # |base| < 2^26: exact
    keys = list(ints)
    ti = torch.tensor([k[0] for k in keys], device="cuda")
    te = torch.tensor([k[1] for k in keys], device="cuda")
    tiles[:, ti, te] = torch.tensor([ref.residues_of(ints[k]) for k in keys], dtype=torch.uint8, device="cuda").T
    want_t[ti, te] = torch.tensor([float(ints[k]) for k in keys], dtype=torch.float64, device="cuda")
    C = _sentinel_C(Mp, Mp, seed=1)
    want = C.clone()
    ii, jj = torch.tril_indices(nt, nt, device="cuda")
    W = want.view(nt, 128, nt, 128).permute(0, 2, 1, 3)
    W[ii, jj] = want_t.view(T, 128, 128)
    torch.cuda.synchronize()
    _ok(shim.i8_crt_launch(tiles.data_ptr(), T * ref.KB_BYTES, C.data_ptr(), Mp, 1.0, _stream()))
    torch.cuda.synchronize()
    _assert_bitwise(C.cpu().numpy(), want.cpu().numpy(), Mp, "reconstruction")


# ---- end to end ----------------------------------------------------------------------------------------------------------------
def _small_cases():
    out = []
    for n, (Mp, ncols) in enumerate((Mp, nc) for Mp in (128, 256, 384) for nc in (128, 384, 512, 640)):
        ldk = ncols + 256 if n % 3 == 2 else ncols
        ldc = Mp + 6 if n % 2 else Mp
        out.append((Mp, ncols, ldk, ldc, VARIANCES[n % 6], ALPHAS[n % 4]))
    return out


# (Mp, ncols, ldk, ldc, v, alpha)
E2E_CASES = _small_cases() + [
    (1536, 16384, 16384, 1536, 1.3, ALPHAS[3]),     # the step's smallest int8 shape
    (1536, 16128, 16384, 1538, 0.6, -3.5),          # ragged: 16 384 - 300 points rounded up to 128
    (1664, 16384, 16384, 1664, 7.0, -1e-8),         # odd tile count: the padding row block
    (1664, 16128, 16384, 1674, 1e6, 1.0),
    (2048, 16384, 16384, 2048, 1e-6, -3.5),         # cfg3's M
    (4096, 16384, 16384, 4096, 2.0 ** -20, ALPHAS[3]),   # cfg4's M
    (8192, 16384, 16384, 8192, 1.3, -3.5),          # many units per persistent CTA
]


def _e2e_id(c):
    return f"Mp{c[0]}-n{c[1]}-ldk{c[2]}-ldc{c[3]}-v{c[4]:g}-a{c[5]:g}"


@pytest.mark.gpu
@pytest.mark.parametrize("Mp,ncols,ldk,ldc,v,alpha", E2E_CASES, ids=[_e2e_id(c) for c in E2E_CASES])
def test_syrk_launch_is_the_exact_product_rounded_once(shim, Mp, ncols, ldk, ldc, v, alpha):
    s = _stream()
    K = _slab(Mp, ncols, ldk, v, seed=Mp * 7 + ncols)
    planes, tiles = _workspace(shim, Mp, ldk, s)
    C = _sentinel_C(Mp, ldc, seed=Mp + ldc)
    C0 = C.cpu().numpy()
    _syrk(shim, K, Mp, ncols, v, alpha, planes, ldk, tiles, C, s)
    torch.cuda.synchronize()
    want = ref.syrk_model(ref.grid_t(K[:, :ncols], v), C0, v, alpha)
    _assert_bitwise(C.cpu().numpy(), want, Mp, f"Mp {Mp} ncols {ncols}")


@pytest.mark.gpu
def test_widest_slab_at_the_int32_bound(shim):
    # 130 944 columns (I8_MAX_COLS) with rows of residue -128 mod 256: the int32 sums come within 2^21 of 2^31
    Mp, ncols = 256, ref.MAX_POINTS
    s = _stream()
    K, v = _int32_bound_slab(Mp, ncols, seed=11)
    A = ref.grid_t(K, v)
    assert bool((torch.remainder(A[:4], 256) == 128).all())
    planes, tiles = _workspace(shim, Mp, ncols, s)
    C = _sentinel_C(Mp, Mp, seed=12)
    C0 = C.cpu().numpy()
    _syrk(shim, K, Mp, ncols, v, -3.5, planes, ncols, tiles, C, s)
    torch.cuda.synchronize()
    _assert_bitwise(C.cpu().numpy(), ref.syrk_model(A, C0, v, -3.5), Mp, "widest slab")


@pytest.mark.gpu
def test_accumulation_and_workspace_reuse(shim):
    # a 16 384-column slab, then a 384-column one on the same planes and tiles (ldk 16 384): (C0 + r1) + r2, with C0 != 0,
    # each sum rounded once with its product (fma)
    Mp, ldk, v, alpha = 1664, 16384, 0.6, ALPHAS[3]
    s = _stream()
    K1 = _slab(Mp, 16384, ldk, v, seed=21)
    K2 = _slab(Mp, 384, ldk, v, seed=22)
    planes, tiles = _workspace(shim, Mp, ldk, s)
    g = torch.Generator(device="cuda").manual_seed(23)
    lower = alpha * v * v * 16384 * 0.25 * torch.randn(Mp, Mp, generator=g, device="cuda", dtype=torch.float64)
    C = _sentinel_C(Mp, Mp, seed=24, lower=lower)
    C0 = C.cpu().numpy()
    assert C0[_lower_mask(Mp, Mp).cpu().numpy()].all()
    _syrk(shim, K1, Mp, 16384, v, alpha, planes, ldk, tiles, C, s)
    _syrk(shim, K2, Mp, 384, v, alpha, planes, ldk, tiles, C, s)
    torch.cuda.synchronize()
    want = ref.syrk_model(ref.grid_t(K1, v), C0, v, alpha)
    want = ref.syrk_model(ref.grid_t(K2[:, :384], v), want, v, alpha)
    _assert_bitwise(C.cpu().numpy(), want, Mp, "two slabs")


@pytest.mark.gpu
def test_non_default_stream(shim):
    Mp, ncols, v, alpha = 384, 2048, 7.0, -3.5
    K = _slab(Mp, ncols, ncols, v, seed=31)
    C = _sentinel_C(Mp, Mp, seed=32)
    C0 = C.cpu().numpy()
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        planes, tiles = _workspace(shim, Mp, ncols, st.cuda_stream)
        _syrk(shim, K, Mp, ncols, v, alpha, planes, ncols, tiles, C, st.cuda_stream)
    st.synchronize()
    _assert_bitwise(C.cpu().numpy(), ref.syrk_model(ref.grid_t(K, v), C0, v, alpha), Mp, "side stream")
