// G1-point NTTs.  The inverse one is the Lagrange-basis SRS  L_i = (1/n) * sum_j w^(-ij) * SRS_j  (natural order),
// replacing KZG::g1_ifft (reference prover/src/kzg.rs:263-285: ark-poly `ifft` over G1Projective, then
// n un-batched into_affine).  The commitment path never needs it (MSM(IFFT_G1(SRS), f) ==
// MSM(SRS, IFFT_Fr(f))); it is public API and is pinned by the reference's lagrangeG1SRS.txt fixture.  The forward
// one serves the proofs at every root of the domain (allroots.cu).
//
// Radix-2 decimation in frequency on XYZZ points in global memory, one thread per butterfly and
// stage:  (P, Q) -> (P + Q, (P - Q) * w^(+-t)), the twiddle product being a 254-bit scalar multiplication
// (~4000 Fq multiplications; the integer pipe is the bound, each point moves 2 x 128 B per stage).
// The last kernel scales, converts to affine (one safegcd inversion per point) and writes to
// the bit-reversed index so the output is in natural order.
#include "kzgb_internal.hpp"

namespace kzgb {

// r = k * p, k a canonical (non-Montgomery) 256-bit scalar; exact for every input
__device__ __forceinline__ void xyzz_mul_scalar(XYZZ& r, const XYZZ& p, const Fr& k) {
    XYZZ acc; xyzz_set_inf(acc);
    bool started = false;
    for (int w = 7; w >= 0; w--) {
        uint32_t word = k.l[w];
        if (!started && word == 0) continue;
        for (int b = 31; b >= 0; b--) {
            if (started) xyzz_dbl(acc, acc);
            if ((word >> b) & 1u) { xyzz_add(acc, p); started = true; }
        }
    }
    r = acc;
}

__global__ void __launch_bounds__(128) k_g1_from_affine(const Affine* __restrict__ in, XYZZ* __restrict__ out, uint32_t n) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    XYZZ p;
    xyzz_from_affine(p, aff_load_ro(&in[i]));
    xyzz_store(&out[i], p);
}

// one DIF stage with butterfly span 2^(s+1).  Forward twiddle w^t = tw[t * 2^(logN-1-s)], multiplied by the signed-window
// routine; inverse twiddle w^-t = -tw[(N/2) - t * 2^(logN-1-s)], multiplied by xyzz_mul_scalar (the Lagrange tables' path).
template <bool INV>
__global__ void __launch_bounds__(128) k_g1_ntt_stage(XYZZ* __restrict__ pts, int logn, int s, const Fr* __restrict__ tw,
                                                       int logN) {
    uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= (1u << (logn - 1))) return;
    const uint32_t h = 1u << s;
    const uint32_t t = b & (h - 1u);
    const uint32_t i = ((b >> s) << (s + 1)) | t;
    const uint32_t j = i + h;
    XYZZ P = xyzz_load(&pts[i]), Q = xyzz_load(&pts[j]);
    XYZZ sum = P;
    xyzz_add(sum, Q);
    XYZZ nq; xyzz_neg(nq, Q);
    XYZZ dif = P;
    xyzz_add(dif, nq);
    xyzz_store(&pts[i], sum);
    const uint32_t idx = t << (logN - 1 - s);
    if (idx != 0) {
        Fr w;
        if (INV) {
            w = fe_load_ro(&tw[(1u << (logN - 1)) - idx]);
            fe_neg(w, w);
        } else {
            w = fe_load_ro(&tw[idx]);
        }
        fe_from_mont(w, w);
        XYZZ r;
        if (INV) xyzz_mul_scalar(r, dif, w);
        else xyzz_mul_scalar_w4(r, dif, w);
        dif = r;
    }
    xyzz_store(&pts[j], dif);
}

// out[bitrev(i)] = affine(scale * pts[i])
__global__ void __launch_bounds__(128) k_g1_ntt_finish(const XYZZ* __restrict__ pts, Affine* __restrict__ out, int logn,
                                                        Fr scale_canon) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (1u << logn)) return;
    XYZZ p = xyzz_load(&pts[i]), r;
    xyzz_mul_scalar(r, p, scale_canon);
    Affine a;
    xyzz_to_affine(a, r);
    uint32_t o = logn ? (__brev(i) >> (32 - logn)) : 0u;
    aff_store(&out[o], a);
}

void g1_ntt_stages_launch(XYZZ* pts, int logn, bool inverse, const Fr* tw, int logN, cudaStream_t st) {
    const uint32_t nb = (1u << logn) / 2;
    for (int s = logn - 1; s >= 0; s--) {
        if (inverse) k_g1_ntt_stage<true><<<(nb + 127) / 128, 128, 0, st>>>(pts, logn, s, tw, logN);
        else k_g1_ntt_stage<false><<<(nb + 127) / 128, 128, 0, st>>>(pts, logn, s, tw, logN);
        g_launch_count++;
    }
}

void g1_ntt_finish_launch(const XYZZ* pts, Affine* out, int logn, const Fr* scale_canon_host, cudaStream_t st) {
    const uint32_t n = 1u << logn;
    k_g1_ntt_finish<<<(n + 127) / 128, 128, 0, st>>>(pts, out, logn, *scale_canon_host);
    g_launch_count++;
}

void g1_intt_launch(const Affine* srs, int logn, XYZZ* work, Affine* out, const Fr* tw, int logN,
                    const Fr* ninv_canon_host, cudaStream_t st) {
    const uint32_t n = 1u << logn;
    k_g1_from_affine<<<(n + 127) / 128, 128, 0, st>>>(srs, work, n);
    g_launch_count++;
    g1_ntt_stages_launch(work, logn, true, tw, logN, st);
    g1_ntt_finish_launch(work, out, logn, ninv_canon_host, st);
}

}  // namespace kzgb
