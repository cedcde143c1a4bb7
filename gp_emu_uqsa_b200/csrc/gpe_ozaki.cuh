// FP64 GEMM emulated on the INT8 tensor cores (tcgen05.mma kind::i8) by integer modular arithmetic -- "Ozaki scheme II".
//
// sm_100a has no FP64 tcgen05 kind: DMMA.8x8x4 peaks at the DFMA rate (37.2 TFLOP/s measured), and the big products of
// the factorisation (gpe_api.cu:potrf_inv_rec) and LAUUM already run at 0.86 of that.  This family is the way past that
// roof: C = op(A) op(B) is evaluated as
//   1. oz_convert_kernel: each row of op(A) / column of op(B) is scaled by a power of two, truncated to a `bits`-bit
//      integer and reduced modulo nmod pairwise coprime moduli p <= 256 -> unsigned 8-bit residue planes, K-major;
//   2. oz_gemm_kernel: one exact u8 x u8 -> s32 GEMM per modulus on the tensor cores -- TMA (128B-swizzled tensor maps)
//      feeds a 4-stage shared-memory ring, one thread issues tcgen05.mma into a double-buffered TMEM accumulator, four
//      epilogue warps read it back with tcgen05.ld, reduce mod p and store 8-bit residues;
//   3. oz_combine_kernel: Chinese remainder theorem in 96-bit fixed point (V/P = frac(sum_i r_i y_i / p_i)), centred,
//      scaled back, rounded once to FP64, C = alpha * V (+ C).
// Step 2 is exact, so the only error is the truncation of step 1: relative to (row max of A) x (column max of B), about
// K 2^(1-bits); bits = 63 (nmod = 18), 59-60 (17), 56 (16).  The reference arithmetic this replaces is NumPy's float64
// matmul / LAPACK inside np.linalg.cholesky and solve (_emulatoroptimise.py:313-335, 425-441); the parity bar (llh 1e-10,
// gradient 1e-9 against the real reference at n = 4096) is what decides nmod.  oracle/ozaki2_oracle.py restates the
// arithmetic limb for limb.  The default (nmod = 16) for products of 1024 and more in every dimension (GPE_OZAKI_MIN);
// GPE_OZAKI=<nmod> sets the number of moduli, GPE_OZAKI=0 keeps every product on DMMA.
#pragma once
#include "gpe_gemm.cuh"

namespace gpe {

constexpr int OZ_MAXMOD = 20;
constexpr int OZ_BM = 128, OZ_BN = 256, OZ_BK = 128;   // tile of the residue GEMM; BK in bytes = elements

// scratch of one stream: residue planes of the operands and of the product, scale exponents
struct OzWs {
    uint8_t *PA = nullptr, *PB = nullptr, *PD = nullptr;
    int *sA = nullptr, *sB = nullptr;
    size_t capA = 0, capB = 0, capD = 0, capS = 0;
    // what PA / sA hold: a caller that knows the source is unchanged since the previous product on this stream may ask for
    // the planes to be used again (the factorisation: L21 is an operand of two consecutive products)
    struct Key {
        const double* src; int ld; long long stride; int R, K, batch, nmod, bits, tri, kc;
        bool operator==(const Key& o) const {
            return src == o.src && ld == o.ld && stride == o.stride && R == o.R && K == o.K && batch == o.batch && nmod == o.nmod &&
                   bits == o.bits && tri == o.tri && kc == o.kc;
        }
    };
    Key key_a{};
    unsigned long long tag_a = 0; // caller's generation of the source (0: none)
    bool have_a = false;
    bool grew = false;           // set when a buffer was reallocated: captured graphs that used the old one are stale
    void release();
};

// What the caller of one product knows about its operands (all zero: nothing).
struct OzHint {
    // the planes of operand A left on this stream by the previous product may be used again if they describe the same operand
    // and carry the same tag (the caller vouches that the source has not changed)
    bool reuse_a = false;
    unsigned long long a_tag = 0;
    double b_bound = 0.0;        // |B| <= b_bound everywhere: operand B takes one scale and its maxima are not searched
};

bool oz_supported(const GemmP& p, int epi);
// largest operand width with K 2^(2 bits) < P/2
int oz_operand_bits(int nmod, int K);
// optional per-phase hook for event timing (phase 0 residue conversion, 1 residue GEMM, 2 CRT)
struct OzHook {
    void* ctx = nullptr;
    void (*fn)(void* ctx, int phase, bool begin, cudaStream_t st) = nullptr;
    void operator()(int phase, bool begin, cudaStream_t st) const { if (fn) fn(ctx, phase, begin, st); }
};

// column norms (EPI_SUMSQ, k <= i) evaluated with the roles swapped -- Z^T = B^T A^T, row norms: the output is then ONE row of
// partial sums, C[0 .. N), instead of M / 128 rows
bool oz_sumsq_swapped(const GemmP& p, int epi);
// makes sure `ws` can hold the planes of `p` (allocates: must not be called during stream capture when it has to grow); a
// reallocation sets ws.grew and forgets the planes of operand A
cudaError_t oz_reserve(OzWs& ws, const GemmP& p, int layout, int nmod);
// C = alpha op(A) op(B) (+ C), same meaning of every field of p, of `layout` and of `epi` as launch_gemm (EPI_SUMSQ: batch 1).
cudaError_t oz_gemm(const GemmP& p, int layout, int epi, int nmod, OzWs& ws, cudaStream_t st, const OzHint& hint = OzHint(),
                    const OzHook& hook = OzHook());

}  // namespace gpe
