/* magprop_band.h -- C ABI of the credible band of the light curve on the device: exact order statistics of many
 * columns at once.  An extension of magprop_b200.h: same conventions, same library (libmagprop_b200.so), same return
 * codes; MP_ABI_VERSION covers it too.
 *
 * A band is np.percentile(curves, q, axis=0) over S posterior draws' curves [S][3][Gs] (mp_model_curves_device): at
 * every node, two neighbouring order statistics of the S values, interpolated by NumPy's rule on the host.
 */
#ifndef MAGPROP_BAND_H
#define MAGPROP_BAND_H

#include "magprop_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Exact order statistics of many columns at once: what a credible band of light curves needs at every node
 * (np.percentile(curves, q, axis=0) over posterior draws).  d_x holds n rows on `device`; element (row i, column c)
 * is d_x[i*ld + c], ld >= n_cols (a curve buffer [S][3][Gs] is n = S rows of 3*Gs columns).  d_out is a DEVICE array
 * [n_ranks][n_cols]: d_out[r][c] = the ranks[r]-th smallest value (0-based) of column c, in the total order of
 * mp_chain_order_statistics (-0.0 before +0.0, every NaN last, a NaN returned with its sign bit cleared).  ranks is a
 * HOST array, in any order, duplicates allowed.  Exact, so the result is the same bits on any stream.
 * MP_ERR_BAD_ARG before any device work: a null d_x, d_out or ranks; n outside 1..MP_COLUMN_SELECT_MAX; n_cols < 1;
 * ld < n_cols; n_ranks < 1; a rank outside [0, n); d_out's range overlapping the range d_x spans.  Stream-ordered on
 * `stream`: no allocation and no synchronisation.  One block sorts one column in shared memory (8 bytes per row,
 * rounded up to a power of two), which is what bounds n.                                                    */
#define MP_COLUMN_SELECT_MAX 16384
int mp_columns_order_statistics(const double* d_x, int64_t n, int64_t n_cols, int64_t ld,
                                const int64_t* ranks, int32_t n_ranks, double* d_out,
                                int32_t device, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MAGPROP_BAND_H */
