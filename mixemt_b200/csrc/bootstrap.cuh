// Resampling of the nonparametric bootstrap (bootstrap.cu): the fragments a replicate draws,
// as counts per signature row.  The EM side of a bootstrap lives in em.cu (mxb_em_bootstrap).
#pragma once

#include <stdint.h>

#include <vector>

struct mxb_ctx;

namespace mxb {

// Checks that the weights are finite, non-negative, integral and sum to 1 <= W < 2^32
// (MXB_ERR_VALUE otherwise) and forms their inclusive prefix sums.
int boot_prefix(const double *weights, int64_t n_rows, std::vector<int64_t> &cumw, uint64_t &total);

// counts[k][i] += draws of row i by replicate boot0 + k, k < n_boot (counts must start at zero):
// one thread per fragment, W fragments per replicate, integer atomics.  cumw on the device.
int boot_draw(mxb_ctx *ctx, const int64_t *cumw, int64_t n_rows, uint64_t total, uint64_t seed,
              int64_t boot0, int64_t n_boot, uint32_t *counts);

// w[i] = counts[i] as fp64, and counts[i] = 0 again for the next draw.
int boot_take_counts(mxb_ctx *ctx, uint32_t *counts, int64_t n_rows, double *w);

}  // namespace mxb
