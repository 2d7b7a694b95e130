// gpa.cuh -- O(N^2) kernels of the latent-GP (GPA) target and gradient (see gpa.cu).
// Buffers follow the engine's layout (gpb200.cu): F / G row-major with leading dimension ld, L in F's lower triangle,
// W' = L^-T in G's strictly-upper tiles after the inverse merges, DinvT / Zd compact [Npad x 128] diagonal tiles.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

// out = L x (trans = false) or out = L' x (trans = true); x, out: Npad (x zero past N).
// part: [Npad/128 x Npad] scratch of per-tile partial sums, reduced in a fixed order.
cudaError_t gpa_trmv(const double* F, int64_t ld, int64_t Npad, bool trans, const double* x, double* part, double* out,
                     cudaStream_t st, int64_t* launches);

// Z' of the closed-form reverse-mode Cholesky, Z'[b,k] = w_k (sum_{l<k} v_l W'[b,l] + v_k W'[b,k] / 2):
// strictly-upper tiles into F (scratch once the inverse merges are done), diagonal tiles into Zd [Npad x 128].
// tsum: [Npad/128 x Npad] scratch (per-tile row sums, then their exclusive prefix along each row).
cudaError_t gpa_row_scan(const double* G, int64_t ld, const double* DinvT, const double* v, const double* w, int64_t Npad,
                         double* tsum, double* F, double* Zd, cudaStream_t st, int64_t* launches);
