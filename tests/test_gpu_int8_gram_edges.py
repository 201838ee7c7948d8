"""
Edge cases of the int8 Gram product's integer arithmetic (csrc/int8_gram.cu, DESIGN §2), bit for bit against tests/int8_gram_ref.py.

    residues        the grid integer t enters as u = t + 2^53, split into three 18-bit limbs; each residue is a limb combination
                    below 2^27 reduced by one multiply-high.  Checked at the limb boundaries, at +-(2^53 - 1), at exact multiples
                    of every modulus and next to them, at both ends of every symmetric range, and on the grid's edge entries.
    reconstruction  Garner's digits with one reduction each (a sum of constant multiples of the lower digits).  Checked on
                    residue vectors drawn uniformly (every integer of [0, P) equally likely) and on structured ones: every
                    residue 0 or p_i - 1, one non-zero residue, every digit at its largest.

The CPU tests replay the same integer arithmetic in NumPy (uint32, wrapping as on the device) against the references.
"""
import numpy as np
import pytest
import torch

from tests import int8_gram_ref as ref
from tests.test_gpu_int8_gram_kernels import _assert_bitwise, _geometry, _ok, _sentinel_C, _specials, _stream, _workspace, shim  # noqa: F401

ODD = ref.MODULI[1:]


def _edge_integers():
    """Grid integers where the limb and modular arithmetic has its edges, both signs."""
    xs = {0, 1, 2 ** 53 - 1, 2 ** 53 - 2, 2 ** 52, 2 ** 54 // 3}
    for b in (2 ** 18, 2 ** 36):
        xs |= {b - 1, b, b + 1, 2 * b - 1, (2 ** 18 - 1) * b}
    xs |= {2 ** 53 - 2 ** 36, 2 ** 53 - 2 ** 18, 2 ** 36 + 2 ** 18 + 1, (2 ** 17 - 1) * 2 ** 36 + (2 ** 18 - 1) * (1 + 2 ** 18)}
    for p in ref.MODULI:
        h = (p - 1) // 2
        for k in (1, 2 ** 18 // p, 2 ** 36 // p, 2 ** 45 // p, (2 ** 53 - 1) // p):
            for d in (-h - 1, -h, -1, 0, 1, h, h + 1):
                if 0 <= k * p + d < 2 ** 53:
                    xs.add(k * p + d)
    xs = sorted(x for x in xs if x < 2 ** 53)
    return xs + [-x for x in xs if x]


def _residues_np(t):
    """The residue kernel's arithmetic in NumPy: int64 grid integers -> [16, n] residue bytes (uint8)."""
    u = (np.asarray(t, dtype=np.int64) + (1 << 53)).astype(np.uint64)
    l0, l1, l2 = ((u >> np.uint64(s)) & np.uint64((1 << 18) - 1) for s in (0, 18, 36))
    out = [(u & np.uint64(0xFF)).astype(np.uint8)]
    for p in ODD:
        h = (p - 1) // 2
        off = (h - 2 ** 53) % p
        x = (l2 * np.uint64(2 ** 36 % p) + l1 * np.uint64(2 ** 18 % p) + l0 + np.uint64(off)).astype(np.uint32)
        assert int(x.max()) < 2 ** 27
        m = np.uint64(-(-2 ** 36 // p))
        q = ((x.astype(np.uint64) * m) >> np.uint64(32)).astype(np.uint32) >> np.uint32(4)   # __umulhi, then >> 4
        r = (x - q * np.uint32(p) - np.uint32(h)).astype(np.uint32)
        out.append((r & np.uint32(0xFF)).astype(np.uint8))
    return np.stack(out)


def _garner_np(r):
    """The reconstruction's digits in NumPy: [16, n] residues -> [16, n] Garner digits, one multiply-high reduction each."""
    r = np.asarray(r, dtype=np.uint32)
    v = [r[0]]
    for i, p in enumerate(ref.MODULI[1:], start=1):
        pre = [int(np.prod([int(q) for q in ref.MODULI[:j]], dtype=object)) % p for j in range(i + 1)]
        inv = pow(pre[i], -1, p)
        s = r[i] * np.uint32(inv)
        for j in range(i):
            s = s + v[j] * np.uint32((-pre[j] * inv) % p)
        assert int(s.max()) < 2 ** 28
        q = ((s.astype(np.uint64) * np.uint64(-(-2 ** 36 // p))) >> np.uint64(32)).astype(np.uint32) >> np.uint32(4)
        v.append((s - q * np.uint32(p)).astype(np.uint32))
    return np.stack(v)


def _residue_vectors(n, seed):
    """[16, n] residue vectors: structured ones first, then uniform draws."""
    rng = np.random.default_rng(seed)
    p = np.array(ref.MODULI)[:, None]
    rows = [np.zeros(16, int), p[:, 0] - 1, np.array(ref.residues_of(ref.P // 2)), np.array(ref.residues_of(ref.P // 2 + 1))]
    for i in range(16):
        for val in (1, ref.MODULI[i] - 1):
            e = np.zeros(16, int)
            e[i] = val
            rows.append(e)
    big = 0   # every Garner digit at its largest: x = P - 1 ... and the integer just below each partial product
    for i, q in enumerate(ref.MODULI):
        big = big + (q - 1) * int(np.prod([int(m) for m in ref.MODULI[:i]], dtype=object))
        rows.append(np.array(ref.residues_of(big)))
    fixed = np.stack(rows, axis=1)
    return np.concatenate([fixed, rng.integers(0, p, (16, n - fixed.shape[1]))], axis=1)


# ---- without a GPU: the arithmetic itself ---------------------------------------------------------------------------------------
def test_residue_arithmetic_matches_the_reference():
    t = np.array(_edge_integers() + list(np.random.default_rng(1).integers(-2 ** 53 + 1, 2 ** 53, 20000)), dtype=np.int64)
    got = _residues_np(t)
    want = np.stack([ref.residue_t(torch.from_numpy(t), p).to(torch.int8).view(torch.uint8).numpy() for p in ref.MODULI])
    assert np.array_equal(got, want)


def test_lazy_garner_digits_match_the_reference():
    r = _residue_vectors(3000, seed=2)
    v = _garner_np(r)
    p = np.array(ref.MODULI)[:, None]
    assert (v < p).all()
    x = np.zeros(r.shape[1], dtype=object)
    for i in reversed(range(16)):
        x = x * ref.MODULI[i] + v[i].astype(object)
    x = np.where(x > ref.P // 2, x - ref.P, x)
    assert list(x) == list(ref.crt([ri for ri in r]))


# ---- on the GPU: the kernels --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("v", [1.0, 2.0 ** -20, 1.3])
def test_residue_planes_at_the_arithmetic_edges(shim, v):
    # Mp 384 (odd tile count: the padding row block), 3 k-blocks.  For v a power of two, K = t v 2^-52 is exact and the grid
    # integer is t itself; every edge integer appears in several rows and k-blocks, the rest is a covariance slab with the grid's
    # edge entries (just above v, the grid's top, +-Inf, NaN), negated in alternate rows
    Mp, ncols, nc_alloc = 384, 384, 512
    s = _stream()
    edges = torch.tensor(_edge_integers(), dtype=torch.int64)
    g = torch.Generator().manual_seed(5)
    u = torch.rand(Mp, ncols, generator=g, dtype=torch.float64)
    K = v * u * u
    sp = torch.tensor(_specials(v), dtype=torch.float64)
    K[::7] = sp[torch.randint(0, len(sp), (K[::7].numel(),), generator=g)].view(K[::7].shape)
    K[1::2] = -K[1::2]
    if v in (1.0, 2.0 ** -20):
        flat = K.view(-1)
        idx = torch.randperm(flat.numel(), generator=g)[: 4 * len(edges)]
        flat[idx] = edges.repeat(4).to(torch.float64) * (v * 2.0 ** -52)
        assert torch.equal(ref.grid_t(flat[idx], v), edges.repeat(4))
    Kd = torch.full((Mp, nc_alloc), 0.5 * v, dtype=torch.float64)
    Kd[:, :ncols] = K
    Kd = Kd.cuda()
    planes, _ = _workspace(shim, Mp, nc_alloc, s)
    geo = _geometry(Mp, ncols, nc_alloc)
    _ok(shim.i8_residue_launch(Kd.data_ptr(), nc_alloc, ref.GRID / v, planes.data_ptr(), geo["pstride"], geo["nrb"], geo["nkb"],
                               geo["nt"], s))
    torch.cuda.synchronize()
    want = ref.plane_image(ref.grid_t(Kd[:, :ncols], v), nc_alloc)
    bad = torch.nonzero(planes != want)
    assert len(bad) == 0, f"{len(bad)} plane bytes differ; first at byte {int(bad[0])} of {planes.numel()}"


@pytest.mark.gpu
def test_reconstruction_of_every_residue_pattern(shim):
    # Mp 256: three lower tiles, 49 152 entries, each a residue vector; scale 1 and C0 = 0, so the output is float(x) of the
    # symmetric-range integer x
    Mp = 256
    nt = Mp // 128
    T = nt * (nt + 1) // 2
    r = _residue_vectors(T * ref.KB_BYTES, seed=3)
    x = ref.crt([ri for ri in r])
    tiles = torch.from_numpy(r.astype(np.uint8)).view(16, T, ref.KB_BYTES).cuda()
    want_t = torch.tensor([float(xi) for xi in x], dtype=torch.float64).view(T, 128, 128).cuda()
    C = _sentinel_C(Mp, Mp, seed=4)
    want = C.clone()
    ii, jj = torch.tril_indices(nt, nt, device="cuda")
    W = want.view(nt, 128, nt, 128).permute(0, 2, 1, 3)
    W[ii, jj] = want_t
    torch.cuda.synchronize()
    _ok(shim.i8_crt_launch(tiles.data_ptr(), T * ref.KB_BYTES, C.data_ptr(), Mp, 1.0, _stream()))
    torch.cuda.synchronize()
    _assert_bitwise(C.cpu().numpy(), want.cpu().numpy(), Mp, "reconstruction of residue patterns")
