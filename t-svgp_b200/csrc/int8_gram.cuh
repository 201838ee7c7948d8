// The Gaussian step's constant-weight SYRK  C += alpha K K^T  (lower 128-tiles) as an exact integer Gram product on the INT8
// tensor cores (DESIGN §2): K is rounded once to the fixed-point grid  A = rint(K 2^52 / v),  A A^T is formed exactly from its
// residues modulo 16 pairwise coprime moduli (int8 x int8 -> int32, tcgen05.mma kind::i8) and rebuilt by the Chinese remainder
// theorem, then rounded once to double.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace tsvgp {

constexpr int I8_NMOD = 16;
// widest slab the int32 accumulation holds exactly: |r_i r_j| <= 2^14 per point, fewer than 2^17 points
constexpr long I8_MAX_COLS = (1L << 17) - 128;

// bytes of the residue planes of one Mp x nc slab: 16 int8 images of [nc / 128 k-blocks][Mp / 128 rounded up to even][16 KB]
size_t i8_plane_bytes(int Mp, long nc);
// bytes of the per-modulus residues of the lower 128-tiles of an Mp x Mp product
size_t i8_tile_bytes(int Mp);

// C[Mp x Mp] (row-major, ldc; lower 128-tiles, diagonal tiles in full) += alpha * K K^T over ncols (multiple of 128, <= I8_MAX_COLS)
// columns of K[Mp][ldk], whose entries lie in [0, var] up to rounding.  `planes` and `tiles` are workspace of the sizes above; the
// planes' row-block padding must be zero (i8_planes_init).  Three launches on `s`: residues, products, reconstruction.
int i8_syrk_launch(const double* K, long ldk, int Mp, int ncols, double var, double alpha, int8_t* planes, long nc_alloc,
                   uint8_t* tiles, double* C, long ldc, cudaStream_t s);
int i8_planes_init(int8_t* planes, int Mp, long nc_alloc, cudaStream_t s);

}  // namespace tsvgp
