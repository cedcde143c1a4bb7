// Dispatch for the batched DMMA GEMM family (see gpe_gemm.cuh).
#include "gpe_gemm.cuh"

namespace gpe {

template <bool A_KC, bool B_KC>
static cudaError_t dispatch_tiles(const GemmP& p, int epi, cudaStream_t st) {
    if (p.M == 32 || p.M == 16) {   // skinny-M panel product (prediction: [e | Gm K^-T]^T C; 16 rows when q + 1 <= 16)
        if (epi != EPI_STORE || p.N % 128) return cudaErrorInvalidValue;
        if (p.M == 16) return launch_gemm_cfg<16, 128, 1, 8, A_KC, B_KC, EPI_STORE>(p, st);
        return launch_gemm_cfg<32, 128, 1, 8, A_KC, B_KC, EPI_STORE>(p, st);
    }
    if (p.N == 32) {
        if (epi != EPI_STORE) return cudaErrorInvalidValue;
        // few items: 128-row tiles would leave most SMs idle behind up to K/16 serial k-steps (n = 1000, one guess:
        // 8 CTAs, 51 us); 32-row tiles give four times the CTAs, each a quarter of the work.  Same k order per
        // output element, so the values do not depend on the tile shape.
        if ((long long)(p.M / 128) * p.batch < NUM_SMS && p.M % 32 == 0)
            return launch_gemm_cfg<32, 32, 2, 2, A_KC, B_KC, EPI_STORE>(p, st);
        return launch_gemm_cfg<128, 32, 4, 2, A_KC, B_KC, EPI_STORE>(p, st);
    }
    if (epi == EPI_SUMSQ) {
        // column norms are accumulated per 128-row tile: the partial buffer is sized for BM = 128.  The ragged last row
        // tile exists in the one-CTA kernel only.
        if (p.M % 128 == 0) return launch_gemm_ws2<A_KC, B_KC, EPI_SUMSQ>(p, st);
        return launch_gemm_ws<A_KC, B_KC, EPI_SUMSQ>(p, st);
    }
    // the two-CTAs-per-SM 128x64 kernel for the machine-filling launches of the factorisation (see gpe_gemm.cuh): a
    // consistent +0.6 % on the n = 4096 step over the one-CTA 128x128 kernel in same-box A/B runs (75.01 -> 74.53 ms,
    // 74.81 -> 74.42 ms)
    if (gemm_fills_machine(p)) return launch_gemm_ws2<A_KC, B_KC, EPI_STORE>(p, st);
    // latency regime (one or two guesses at n <= 2000): 64x64 tiles would occupy under half of the SMs
    long long t64 = (long long)(p.M / 64) * (p.N / 64) * p.batch;
    if (p.lower) t64 = t64 / 2 + (p.M / 64) * p.batch / 2;
    if (t64 < NUM_SMS / 2 && p.M % 32 == 0 && p.N % 32 == 0)
        return launch_gemm_cfg<32, 32, 2, 2, A_KC, B_KC, EPI_STORE>(p, st);
    return launch_gemm_cfg<64, 64, 2, 2, A_KC, B_KC, EPI_STORE>(p, st);
}

bool gemm_fills_machine(const GemmP& p) {
    if (p.M % 128 || p.N % 128) return false;
    long long t128 = (long long)(p.M / 128) * (p.N / 128) * p.batch;
    if (p.lower) t128 = t128 / 2 + (p.M / 128) * p.batch / 2;
    return t128 >= 120;
}

cudaError_t launch_gemm(const GemmP& p, int layout, int epi, cudaStream_t st) {
    switch (layout) {
        case GEMM_NT: return dispatch_tiles<true, true>(p, epi, st);
        case GEMM_NN: return dispatch_tiles<true, false>(p, epi, st);
        case GEMM_TN: return dispatch_tiles<false, false>(p, epi, st);
        default: return cudaErrorInvalidValue;
    }
}

}  // namespace gpe
