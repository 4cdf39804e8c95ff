// Proofs at every root of the domain (KZG::compute_proof_with_known_z_fr_index, prover/src/kzg.rs:187-207, at all n
// indices) by the Feist-Khovratovich method, single-point form: with c = IFFT_n(evals) and S = SRS,
//   pi = DFT_n(H),   H_i = sum_{m <= n-2-i} c_{i+1+m} S_m  (i <= n-2),  H_{n-1} = identity,
// and H is a linear convolution:  u = IDFT_2n(DFT_2n(c || 0) / 2n  (.)  s_hat),  s_hat = DFT_2n(r),
// r_t = S_{n-2-t} for t <= n-2, zero up to 2n;  then H_i = u_{i+n-1}.  s_hat depends only on the SRS and n
// (cached per size by the host).  The G1 transforms are g1ntt.cu's stages; this file holds the kernels around them.
#include "kzgb_internal.hpp"

namespace kzgb {

// out[t] = S_{n-2-t} for t <= n-2, the identity for n-2 < t < 2n  (XYZZ, natural order)
__global__ void __launch_bounds__(128) k_allroots_embed(const Affine* __restrict__ srs, XYZZ* __restrict__ out, uint32_t n) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= 2 * n) return;
    XYZZ p;
    if (t + 2 <= n) xyzz_from_affine(p, aff_load_ro(&srs[n - 2 - t]));
    else xyzz_set_inf(p);
    xyzz_store(&out[t], p);
}

// u_k = (c_hat_k * scale) * s_hat_k, one thread per element (c_hat Montgomery, s_hat affine, both natural order)
__global__ void __launch_bounds__(128) k_allroots_hadamard(const Fr* __restrict__ chat, Fr scale_mont,
                                                           const Affine* __restrict__ shat, XYZZ* __restrict__ u, uint32_t m) {
    uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= m) return;
    Fr s = fe_load_ro(&chat[k]);
    fe_mul(s, s, scale_mont);
    fe_from_mont(s, s);
    XYZZ p, r;
    xyzz_from_affine(p, aff_load_ro(&shat[k]));
    xyzz_mul_scalar_w4(r, p, s);
    xyzz_store(&u[k], r);
}

// H_i = u_{i+n-1} (i <= n-2), H_{n-1} = identity; u is the bit-reversed output of the 2n-point DIF, H natural order
__global__ void __launch_bounds__(128) k_allroots_extract(const XYZZ* __restrict__ u, XYZZ* __restrict__ H, int logn) {
    const uint32_t n = 1u << logn;
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    XYZZ p;
    if (i + 1 < n) p = xyzz_load(&u[__brev(i + n - 1) >> (31 - logn)]);
    else xyzz_set_inf(p);
    xyzz_store(&H[i], p);
}

void allroots_embed_launch(const Affine* srs, int logn, XYZZ* out, cudaStream_t st) {
    const uint32_t m = 2u << logn;
    k_allroots_embed<<<(m + 127) / 128, 128, 0, st>>>(srs, out, 1u << logn);
    g_launch_count++;
}

void allroots_hadamard_launch(const Fr* chat, const Fr* scale_mont_host, const Affine* shat, XYZZ* u, int logm, cudaStream_t st) {
    const uint32_t m = 1u << logm;
    k_allroots_hadamard<<<(m + 127) / 128, 128, 0, st>>>(chat, *scale_mont_host, shat, u, m);
    g_launch_count++;
}

void allroots_extract_launch(const XYZZ* u, XYZZ* H, int logn, cudaStream_t st) {
    const uint32_t n = 1u << logn;
    k_allroots_extract<<<(n + 127) / 128, 128, 0, st>>>(u, H, logn);
    g_launch_count++;
}

}  // namespace kzgb
