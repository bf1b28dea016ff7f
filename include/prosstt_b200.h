/* prosstt_b200.h - C ABI of the B200 (sm_100a) implementation of PROSSTT's
 * simulation hot path.
 *
 * The reference (soedinglab/prosstt 1.2.0) is pure Python and has no FFI of its
 * own; the boundary its users see is the Python module API.  Each entry point
 * below replaces the body of one reference function (cited as
 * prosstt/<file>:<lines>); the Python host layer in prosstt_b200/ keeps the
 * reference signatures and calls these through ctypes (see INTEGRATION.md).
 *
 * Conventions
 *  - plain C types only; every pointer is a DEVICE pointer unless named h_*;
 *  - the caller owns all buffers; nothing here allocates, frees or synchronises;
 *  - every call is stream-ordered on `stream` (a cudaStream_t passed as void*);
 *  - return value: 0 ok, <0 invalid argument, >0 cudaError_t; message via
 *    pst_last_error() (thread-local);
 *  - tree positions are "packed rows": branches in tree.branches order, branch b
 *    owns rows [row_base[b], row_base[b]+T_b); P = sum T_b.  This is also the
 *    concatenation order of sample_density (simulation.py:454-461);
 *  - matrices are row-major: W[P][K], H[K][G], rel/means[P][G], X[N][G];
 *  - every random quantity is a pure function of (seed, stream tag, global
 *    cell/row index[, gene]) through Philox4x32-10, never of thread, block,
 *    launch shape or rank: results are bit-identical for any partition of the
 *    cells over calls, streams or GPUs.
 */
#ifndef PROSSTT_B200_H
#define PROSSTT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)   /* the library is built with -fvisibility=hidden */
#endif

#define PST_ABI_VERSION 2

/* bits of the device-side status word written by the sampling kernels */
#define PST_FLAG_DOMAIN   1u  /* mu <= 0, non-finite, or alpha*mu+beta-1 <= 0: scipy's
                                 "Domain error in arguments" (SURVEY.md Q9)            */
#define PST_FLAG_ROW      2u  /* row_of_cell outside [0,P)                              */
#define PST_FLAG_CLAMPED  4u  /* a count exceeded INT32_MAX and was clamped             */
#define PST_FLAG_NOZONE   8u  /* pseudotime outside every timezone (pick_branch)        */
#define PST_FLAG_SCRATCH  16u /* the scratch list of pst_draw_counts was too small      */

/* which per-count algorithm pst_draw_counts runs */
#define PST_SAMPLER_GAMMA_POISSON 0  /* Marsaglia-Tsang gamma, PTRS / inversion Poisson  */
#define PST_SAMPLER_HYBRID        1  /* direct NB inversion for small means + the above  */

int         pst_abi_version(void);
const char *pst_last_error(void);
/* number of kernels launched by this library in this process (bench "gpu_launches") */
uint64_t    pst_launch_count(void);

/* ---- counter-based draws (replace the global MT19937 of the reference) ------- */
/* out[i] = uniform double in [0,1), 53 bits, element index = first + i.
 * Replaces random_sample inside np.random.choice (simulation.py:464, sim_utils.py:399). */
int pst_uniform_f64(uint64_t seed, uint32_t tag, int64_t first, int64_t n,
                    double *out, void *stream);
/* out[i] = loc + scale * N(0,1).  Replaces scipy.stats.norm.rvs call sites
 * (simulation.py:409, sim_utils.py:495).  loc/scale: per-element device arrays, or NULL
 * to use the scalars loc0/scale0. */
int pst_normal_f64(uint64_t seed, uint32_t tag, int64_t first, int64_t n, double loc0,
                   double scale0, const double *loc, const double *scale, double *out,
                   void *stream);
/* raw Philox4x32-10 words, out[4*i..4*i+3] for counter (first+i, tag, 0) - test hook */
int pst_philox_words(uint64_t seed, uint32_t tag, int64_t first, int64_t n,
                     uint32_t *out, void *stream);

/* ---- lineage: simulation.py:21-124, 215-286; sim_utils.py:129-142, 611-640 ---- */
/* Draws of `diffusion` (simulation.py:107-117) for nb branches x K programs, keyed
 * by (seed, branch_id, attempt, k, t): u0~U(0,1.5), v0~N(0,0.2), eta~U(0,1),
 * eps[t]~N(0,2/T).  Layout: u0/v0/eta [nb*K]; eps for branch j starts at
 * eps_off[j] and is [K][T_j-1]; max_T = max_j T[j] (host copy, sizes the grid). */
int pst_walk_draws(uint64_t seed, int32_t nb, int32_t K, int32_t max_T,
                   const int32_t *branch_id, const int32_t *attempt, const int32_t *T,
                   const int64_t *eps_off, double *u0, double *v0, double *eta, double *eps,
                   void *stream);
/* Momentum walk of every (branch, program): walk[0]=log(u0); walk[t+1]=walk[t]+v[t];
 * v[t+1]=eta*v[t]+eps[t] as a warp-shuffle scan (affine-map scan for v, prefix sum
 * for walk).  Writes W[(row_base[j]+t)*K + k].  Replaces simulation.py:21-124. */
int pst_walk_scan(int32_t nb, int32_t K, const int32_t *row_base, const int32_t *T,
                  const int64_t *eps_off, const double *u0, const double *v0,
                  const double *eta, const double *eps, double *W, void *stream);
/* Parent carry in topological order: for i in 0..n_order-1, child=order_child[i],
 * W[child rows] -= (W[child first row] - W[parent last row]).  order_parent_last[i]
 * is the packed row of the parent's last time point, or -1 for a root.
 * Replaces sim_utils.py:129-142, 611-640. */
int pst_walk_carry(int32_t n_order, int32_t K, const int32_t *order_row_base,
                   const int32_t *order_T, const int32_t *order_parent_last,
                   double *W, void *stream);
/* rel = W[row0:row0+nrows] . H  (simulation.py:269, sim_utils.py:190-213), fused with
 * M = exp(rel) * gene_scale (tree.py:180-183) and the per-gene maximum of rel
 * (simulation.py:270; sim_utils.py:406-426 since exp is monotone).  Any of the
 * outputs may be NULL.  out_rel/out_mean64/out_mean32 are indexed from row 0 of the
 * packed table (row r goes to out[r*G..]).  out_colmax[G] must be initialised by the
 * caller (-inf); it is max-merged. */
int pst_rel_means(const double *W, const double *H, const double *gene_scale,
                  int64_t row0, int64_t nrows, int32_t K, int64_t G,
                  double *out_rel, double *out_mean64, float *out_mean32,
                  double *out_colmax, void *stream);
/* Number of genes whose Pearson r between columns of A[0:n] and B[0:n] is < 0
 * (sim_utils.py:145-168, 249-251).  out_count is one int32, caller zeroes it. */
int pst_pearson_anticorr(const double *A, const double *B, int64_t nrows, int64_t G,
                         int32_t *out_count, void *stream);
/* The acceptance tests of simulate_lineage (simulation.py:270-272) for a batch of candidate
 * branches in one launch.  rel is the packed rel table (candidates live in rows behind the P tree
 * rows).  Candidate i (i < n_slots) owns rows [slot_row[i], slot_row[i]+slot_T[i]): out_slot_max[i]
 * is max-merged with the maximum of those rows (caller initialises it to -inf) - the
 * rel_exp_cutoff test.  Pair p compares the first pair_n[p] rows from pair_a[p] and from pair_b[p]:
 * out_pair_neg[p] (caller zeroes it) receives the number of genes with Pearson r < 0, the
 * sibling-divergence test (sim_utils.py:145-168, 249-251; same arithmetic as pst_pearson_anticorr). */
int pst_lineage_checks(const double *rel, int64_t G, int32_t n_slots, const int64_t *slot_row,
                       const int32_t *slot_T, int32_t n_pairs, const int64_t *pair_a,
                       const int64_t *pair_b, const int32_t *pair_n, double *out_slot_max,
                       int32_t *out_pair_neg, void *stream);
/* fp64 -> fp32 table conversion for means supplied by the user (tree.add_genes).  Positive
 * values below min_positive (pass 1e-30; 0 disables) are raised to it so that a mean that is
 * positive in fp64 never underflows to 0 in the fp32 table (pst_rel_means does the same). */
int pst_f64_to_f32(const double *in, int64_t n, double min_positive, float *out, void *stream);

/* ---- samplers' index maps: simulation.py:319-548, sim_utils.py:342-403 -------- */
/* idx[i] = searchsorted(cdf, u[i], side='right') clipped to P-1; row_of_cell = idx
 * (packed rows are in the same order), pt[i] = pos_pt[idx]; branch[i] = pos_branch[idx].
 * Replaces np.random.choice(p=...) + the gathers at simulation.py:464-467. */
int pst_density_index(const double *cdf, int32_t P, const double *u, int64_t n,
                      const int32_t *pos_pt, const int32_t *pos_branch,
                      int32_t *row_of_cell, int64_t *pt, int32_t *branch, void *stream);
/* pt[i] = clip(trunc(z[i]), 0, max_time-1): draw_times, simulation.py:409-413, given
 * z = norm.rvs(loc=t, scale=std). */
int pst_times_from_normals(const double *z, int64_t n, int32_t max_time, int64_t *pt,
                           void *stream);
/* pick_branch (sim_utils.py:367-403) with one uniform u[i] per cell: zone = first
 * timezone containing pt[i]; weights density[b][pt - zone_start] (sic, SURVEY.md Q5)
 * over the zone's candidate branches; p = w/sum(w) (numpy summation order); legacy
 * choice: cdf = cumsum(p)/cumsum(p)[-1], searchsorted right.  zone_lo/zone_hi [nz];
 * cand_off[nz+1] indexes cand_branch[]; max_cand = largest candidate list (<= 64);
 * branch_start/row_base/T are per branch [B]; density is packed [P].
 * Outputs branch[n] (index into tree.branches) and row_of_cell[n]; a pseudotime
 * outside every zone (the reference returns None there) sets PST_FLAG_NOZONE. */
int pst_pick_branch(const int64_t *pt, const double *u, int64_t n, int32_t nz,
                    const int32_t *zone_lo, const int32_t *zone_hi, const int32_t *cand_off,
                    const int32_t *cand_branch, int32_t max_cand, const int32_t *branch_start,
                    const int32_t *row_base, const int32_t *T, const double *density,
                    int32_t *branch, int32_t *row_of_cell, uint32_t *flags, void *stream);
/* row_of_cell[i] = row_base[b] + pt[i] - branch_start[b] for caller-supplied branches
 * (draw_counts, simulation.py:634-640); out-of-range sets PST_FLAG_ROW. */
int pst_rows_from_branch(const int64_t *pt, const int32_t *branch, int64_t n, int32_t B,
                         const int32_t *branch_start, const int32_t *row_base,
                         const int32_t *T, int32_t *row_of_cell, uint32_t *flags, void *stream);
/* sample_whole_tree (simulation.py:510-513): cell first+i takes entry (first+i)/n_factor
 * of the cover_whole_tree enumeration (cover_pt/cover_branch/cover_row [n_cover]). */
int pst_whole_tree_index(const int32_t *cover_pt, const int32_t *cover_branch,
                         const int32_t *cover_row, int64_t n_cover, int64_t n_factor,
                         int64_t first, int64_t n, int64_t *pt, int32_t *branch,
                         int32_t *row_of_cell, void *stream);
/* scalings = exp(z) in fp64 (returned to the user) and fp32 (consumed by the draw
 * kernel); z=NULL writes ones (scale=False).  Replaces sim_utils.py:494-498. */
int pst_scalings(const double *z, int64_t n, double *out64, float *out32, void *stream);

/* per-gene base expression exp(N(gene_mean, gene_std)), redrawn while base * cap[g] > abs_max
 * (cap = max over the tree of exp(relative mean), from pst_rel_means' out_colmax).  Replaces
 * sim_utils.py:463-469; attempt a of gene g uses the normal at element a*G + g.  out_tries
 * (optional) = draws consumed per gene; PST_FLAG_DOMAIN is set in flags[0] if a gene is still
 * above abs_max after max_tries draws. */
int pst_base_gene_exp(uint64_t seed, uint32_t tag, const double *cap, int64_t G, double abs_max,
                      double gene_mean, double gene_std, int32_t max_tries, double *out_base,
                      int32_t *out_tries, uint32_t *flags, void *stream);

/* ---- count model: count_model.py:131-161 ------------------------------------- */
/* fp64 (p, r) of get_pr_umi for mu[n_cells][G] with per-gene alpha/beta - parity hook
 * for the parameterisation that pst_draw_counts fuses in fp32. */
int pst_nb_params(const double *alpha, const double *beta, const double *mu,
                  int64_t n_cells, int64_t G, double *out_p, double *out_r, void *stream);

/* The SAME parameterisation in fp32, evaluated by the __device__ functions that pst_draw_counts
 * inlines (MUFU rcp/lg2, the small-theta series), in the same operation order: element i has the
 * means-table value M[i], library size scaling[i] and per-element alpha[i], beta_m1[i] = beta-1.
 * Outputs: mu = M s, theta = (alpha M) s + beta-1 (gamma scale; scipy's p = 1/(1+theta)), r = mu/theta
 * (gamma shape, scipy's n), q = theta/(1+theta) = get_pr_umi's p, a = q r, log2 P(X=0) =
 * -r log2(1+theta), and the route the hybrid sampler takes.  Parity hook on the arithmetic that
 * actually runs (count_model.py:156-161). */
#define PST_ROUTE_MIXTURE       0   /* gamma-Poisson mixture                                  */
#define PST_ROUTE_INVERSION     1   /* inversion of the NB cdf: mean <= 32, sd <= 20, theta <= 32, shape <= 48
                                       (or theta < 0.1), decided as s <= s_max(M, alpha, beta-1) */
#define PST_ROUTE_DOMAIN_ERROR  2   /* sets PST_FLAG_DOMAIN in the sampler                    */
int pst_nb_params_f32(const float *M, const float *scaling, const float *alpha, const float *beta_m1,
                      int64_t n, float *out_mu, float *out_theta, float *out_r, float *out_q,
                      float *out_a, float *out_log2p0, int32_t *out_route, void *stream);

/* ---- the hot loop: draw_counts, simulation.py:602-651 ------------------------- */
/* X[i][g] ~ NB(mean mu = means[row_of_cell[i]][g]*scaling[i],
 *              var  alpha[g]*mu^2 + beta[g]*mu)        i in [0,n), g in [0,G)
 * as a gamma-Poisson mixture: gamma shape r = mu/theta, scale theta = alpha*mu +
 * (beta-1)  (== scipy nbinom(n=r, p=1/(1+theta)), count_model.py:156-161).
 * Random numbers: Philox4x32-10 keyed by seed with counter (gene, global cell =
 * cell0+i, draw index) - independent of how cells are split over calls/GPUs.
 * beta_m1[g] = beta[g]-1 formed in fp64 by the caller.  X row stride is ldx
 * elements (>= G).  flags: FOUR uint32 words, zeroed once by the caller: word 0 is OR-ed
 * with PST_FLAG_*; words 1-3 are reserved (the work-scheduler words live in the library,
 * one set per (device, stream), so concurrent launches on different streams are safe).
 * scratch: pst_draw_scratch_words(n, G, P) uint32 words, 16-byte aligned, private to this call
 * until it has completed; content on entry is ignored.  It holds (a) the visiting order of the
 * cells - grouped by tree row (counting sort) and cut into groups of at most 64 cells of one row,
 * so that everything depending on (row, gene) is formed once per group and concurrently running
 * warps share means rows; built by four small kernels in front of the draw, it never changes the
 * counts - and (b) the list of the counts whose uniform lies in the top 2^-14 (about 6e-5 n G
 * entries of 16 bytes), which a last small kernel inverts with a 64-bit uniform against a cdf
 * accumulated in fp64: that is what resolves the upper tail beyond the 1 - 1e-7 quantile.
 * gene_sum / gene_sumsq / gene_zeros (all three or all NULL; G entries each, ADDED to: the caller
 * zeroes them): per-gene sum, sum of squares and number of zeros of this call's counts, fused into
 * the draw (each warp sums its tile of X from L2 right after writing it) - the per-gene half of
 * pst_count_stats without the second pass over the matrix, bit-identical to it. */
int64_t pst_draw_scratch_words(int64_t n, int64_t G, int64_t P);
/* Word offsets inside that scratch (debugging / tests): h_out[0] = capacity of the tail list (entries
 * of 4 words from word 4; word 0 counts them), [1] = order[n] (cells in visiting order), [2] =
 * bins[P+1], [3] = gstart[P+1], [4] = groups (4 words each: first position in order, cells, tree row,
 * 0; word 1 of the scratch counts them), [5] = most groups the layout has room for. */
int pst_draw_scratch_layout(int64_t n, int64_t G, int64_t P, int64_t *h_out);
int pst_draw_counts(const float *means, int64_t P, int64_t G,
                    const int32_t *row_of_cell, const float *scaling,
                    const float *alpha, const float *beta_m1,
                    uint64_t seed, int64_t cell0, int64_t n,
                    int32_t *X, int64_t ldx, uint32_t *flags, int32_t sampler,
                    uint32_t *scratch, int64_t scratch_words,
                    uint64_t *gene_sum, uint64_t *gene_sumsq, uint64_t *gene_zeros, void *stream);

/* One streaming pass over a count matrix X[n][ldx] (first G columns): per-cell total counts and
 * zero counts, per-gene sum, sum of squares and zero counts.  These are the summaries the
 * reference's notebooks compute with NumPy after sampling (library sizes X.sum(axis=1), zero
 * fractions, per-gene mean/variance, e.g. examples/compare_axolotl.ipynb) and the full-size
 * distribution check of the sampler.  All outputs are ADDED to (the caller zeroes them; any may be
 * NULL).  Counts are taken as unsigned.  HBM-read bound, 4 B per count. */
int pst_count_stats(const int32_t *X, int64_t n, int64_t G, int64_t ldx, uint64_t *cell_total,
                    uint32_t *cell_zeros, uint64_t *gene_sum, uint64_t *gene_sumsq,
                    uint64_t *gene_zeros, void *stream);

/* ---- epilogues over the count matrix (SURVEY.md 8f rows 3-4) ------------------- */
#define PST_TRANSFORM_NORMALIZE        0   /* X / scaling            (compare_axolotl.ipynb cell 14) */
#define PST_TRANSFORM_NORMALIZE_LOG1P  1   /* log(X / scaling + 1)                                   */
#define PST_TRANSFORM_LOG1P            2   /* log(X + 1)             (minimal_example.ipynb cell 6)  */
/* out[i][g] = f(X[i][g], scaling[i]) as fp32, row strides ldx / ldo elements.  scaling may be
 * NULL for PST_TRANSFORM_LOG1P. */
int pst_transform_counts(const int32_t *X, int64_t n, int64_t G, int64_t ldx, const float *scaling,
                         int32_t mode, float *out, int64_t ldo, void *stream);
/* Compact the dense (n, G) matrix into CSR: for row i the nonzero columns (ascending) and values
 * go to indices/data[indptr[i] .. indptr[i+1]).  indptr (n+1 entries, device) is the exclusive
 * scan of the per-row nonzero counts, i.e. G - cell_zeros from pst_count_stats.  Sets
 * PST_FLAG_ROW in flags[0] if indptr does not match the matrix (nothing is written past a
 * row's end).  Replaces the dense text dump of tree_utils.py:111-121 as the exchange format. */
int pst_csr_fill(const int32_t *X, int64_t n, int64_t G, int64_t ldx, const int64_t *indptr,
                 int32_t *indices, int32_t *data, uint32_t *flags, void *stream);
/* Sizes of the CSR form of X[n][ldx] (first G columns), pass 1 of the samplers' out="csr" path:
 * row_nnz[i] = number of nonzeros of row i (written), *sat_count += number of elements >= 65535,
 * the uint16 saturation value of pst_csr_pack (ADDED to: the caller zeroes it; may be NULL).
 * One streaming read of X, HBM-read bound, 4 B per count. */
int pst_csr_row_counts(const int32_t *X, int64_t n, int64_t G, int64_t ldx, int32_t *row_nnz,
                       uint64_t *sat_count, void *stream);
/* Row pointer from the row sizes: indptr[0] = 0, indptr[i+1] = row_nnz[0] + ... + row_nnz[i]
 * (n+1 int64 entries).  One CTA; n is one shard's cells. */
int pst_csr_row_offsets(const int32_t *row_nnz, int64_t n, int64_t *indptr, void *stream);
/* Pass 2 of out="csr": pst_csr_fill for a chunk of rows, writing narrow streams into a window.
 * indptr holds the chunk's n+1 GLOBAL row offsets (from pst_csr_row_offsets); nonzero number p
 * (indptr[0] <= p < indptr[n]) goes to indices[p - base] and data[p - base], columns ascending in
 * each row.  index_bits 16 (uint16, needs G <= 65536), 32 (int32) or 64 (int64).  data_bits 32 / 64:
 * exact int32 / int64 values (64-bit widths pair with 32- or 64-bit ones: the final bytes of a file's
 * indices and data, no re-pack); data_bits 16: uint16 min(v, 65535), and every v >= 65535 is also listed as
 * (ovf_pos = p, ovf_value = v), appended at atomicAdd(ovf_count, 1) when that slot is < ovf_cap
 * (ovf_count keeps counting past the cap; pst_csr_row_counts' sat_count is the exact size needed).
 * Sets PST_FLAG_ROW in flags[0] if a row's nonzeros do not match indptr (nothing is written past
 * a row's end). */
int pst_csr_pack(const int32_t *X, int64_t n, int64_t G, int64_t ldx, const int64_t *indptr,
                 int64_t base, void *indices, int32_t index_bits, void *data, int32_t data_bits,
                 int64_t *ovf_pos, int32_t *ovf_value, int64_t ovf_cap, uint64_t *ovf_count,
                 uint32_t *flags, void *stream);

/* The indptr member of a streamed CSR file, one chunk at a time: out[i] = *running + indptr[i+1] for
 * i < n, as int32 (out_bits 32) or int64 (64), then *running += indptr[n].  indptr: the chunk's local
 * row pointer (n+1 entries from 0, pst_csr_row_offsets); running: one device int64 the caller zeroes
 * before the first chunk.  The file's leading 0 is not written here. */
int pst_csr_indptr_bytes(const int64_t *indptr, int64_t n, int64_t *running, void *out, int32_t out_bits,
                         void *stream);

/* Matrix Market text of a chunk of cells (the 10x matrix.mtx.gz, genes x cells): row i of the int32
 * chunk X is cell col0 + i + 1 of the file, and each nonzero X[i][g] = v is the line
 * "<g+1> <col0+i+1> <v>\n", genes ascending.  pst_mtx_row_bytes writes each row's text length,
 * row_bytes[i] = nnz_i (digits(col0+i+1) + 3) + sum over the nonzeros of digits(g+1) + digits(v) (int32;
 * G <= 2^31 / 42); pst_csr_row_offsets scans it into the chunk's text pointer (n+1 int64 entries).
 * pst_mtx_format writes row i's lines at out + text_ptr[i] (out 16-byte aligned), or nothing at all when
 * text_ptr[n] > cap, so a text pointer made on the device needs no host read: the caller sees text_ptr[n]
 * later and formats again into a larger buffer. */
int pst_mtx_row_bytes(const int32_t *X, int64_t n, int64_t G, int64_t ldx, int64_t col0, int32_t *row_bytes,
                      void *stream);
int pst_mtx_format(const int32_t *X, int64_t n, int64_t G, int64_t ldx, int64_t col0, const int64_t *text_ptr,
                   int64_t cap, char *out, void *stream);

/* ---- raw DEFLATE (RFC 1951) on the device: the compressed CSR file (pst_deflate.cu) ---------------
 * The input is cut into blocks of `block` bytes (a multiple of 1024, at most 32768).  Each block becomes
 * one dynamic-Huffman block over the literals 0-255 and end-of-block (no length or distance codes; the
 * one distance code has length 1), followed by an empty stored block (zlib's Z_SYNC_FLUSH marker
 * 00 00 FF FF), so it ends on a byte boundary; a block whose Huffman form is not smaller is one stored
 * block.  No block is final: append 03 00 (an empty final fixed block) to end the stream, and any
 * concatenation of such outputs is one stream.  Codes are at most 15 bits, deterministic for given
 * bytes.
 * Input length: (*count) * scale bytes when count (a device int64) is not NULL, else max_bytes; it is
 * clamped to max_bytes, which sizes the launch, so a length made on the device needs no host read.
 * out (device, pst_deflate_bound(max_bytes, block) bytes) receives the blocks back to back, *out_bytes
 * (device int64) their size and *crc (device) the CRC-32 of the input (zlib.crc32).  work: device
 * workspace of pst_deflate_workspace_bytes(max_bytes, block) bytes. */
int64_t pst_deflate_bound(int64_t n, int32_t block);
int64_t pst_deflate_workspace_bytes(int64_t n, int32_t block);
int pst_deflate_blocks(const void *in, const int64_t *count, int64_t scale, int64_t max_bytes, int32_t block,
                       void *out, int64_t *out_bytes, uint32_t *crc, void *work, int64_t work_bytes,
                       void *stream);
/* LZ77 + Huffman (`compression="lz77"`): the contract of pst_deflate_blocks, with the full DEFLATE
 * alphabet in each dynamic block - literal/length symbols 0-285 and distance codes 0-29, both at most 15
 * bits.  Matches (3-258 bytes) reach back at most to the start of their own block, so each block still
 * decodes on its own and the same framing, bound and CRC hold.  The match search is deterministic: the
 * nearest-first hash chain of each position, at most 8 candidates, and a greedy parse of 512-byte
 * segments (a match is cut at its segment's end).  The same bytes and block give the same output.
 * work: device workspace of pst_deflate_lz_workspace_bytes(max_bytes, block) bytes (that of
 * pst_deflate_blocks plus 2 bytes per input byte for the tokens). */
int64_t pst_deflate_lz_workspace_bytes(int64_t n, int32_t block);
int pst_deflate_lz_blocks(const void *in, const int64_t *count, int64_t scale, int64_t max_bytes, int32_t block,
                          void *out, int64_t *out_bytes, uint32_t *crc, void *work, int64_t work_bytes,
                          void *stream);
/* *crc = CRC-32 (zlib.crc32) of the n device bytes at in; crc is a device word. */
int pst_crc32(const void *in, int64_t n, uint32_t *crc, void *stream);

/* Narrow transfer formats for the device->host path (PCIe is the bound at 4 B per count):
 * out[i][g] = min(X[i][g], SAT) as uint8 (out_bits 8, SAT 255) or uint16 (out_bits 16, SAT 65535),
 * row stride ldo elements.  Every element that reads SAT also gets an entry in the overflow
 * list: ovf_index = (row0 + i)*G + g (flat index in the caller's full matrix), ovf_value = the
 * exact count, appended at atomicAdd(ovf_count, 1) when that slot is < ovf_cap.  ovf_count keeps
 * counting past ovf_cap, so the caller can detect a list that was too small.  Entry order is
 * not deterministic; sort by index.  (The reference returns int64; simulation.py:651.) */
int pst_narrow_counts(const int32_t *X, int64_t n, int64_t G, int64_t ldx, void *out, int64_t ldo,
                      int32_t out_bits, int64_t row0, int64_t *ovf_index, int32_t *ovf_value,
                      int64_t ovf_cap, uint64_t *ovf_count, void *stream);

/* Measurement hook: out[0..n) = value with 128-bit streaming stores (n a multiple of 4, out 16-byte
 * aligned).  Timed by tools/store_ceiling.py, it gives the write-only HBM ceiling that the count
 * write of pst_draw_counts is quoted against beside the read+write copy peak (SURVEY.md 8d). */
int pst_store_fill(int32_t *out, int64_t n, int32_t value, void *stream);

/* ---- host side of the device->host path (HOST pointers; multi-threaded; no CUDA calls) ------
 * The count matrix crosses PCIe in a narrow format (pst_narrow_counts) or as int32 into pinned
 * staging buffers; these routines expand a staged chunk into the caller's matrix - int32, or the
 * int64 the reference returns (simulation.py:651) - while the GPU samples the next chunk.
 * dst[i] = (dst type) src[i], i in [0,n): src_bits 8 / 16 (unsigned) or 32 (signed); dst_bits 32 or
 * 64 (signed).  threads <= 0 uses every hardware thread.  Returns 0, or -1 for an unsupported pair. */
int pst_host_widen(const void *h_src, int32_t src_bits, void *h_dst, int32_t dst_bits, int64_t n,
                   int32_t threads);
/* The same expansion with non-temporal 64-byte stores (AVX-512; ordinary stores elsewhere and on the
 * unaligned edges; 32 -> 32 bits is a streaming copy): for a destination that is NOT in cache - a
 * pinned or re-used result matrix - the lines are written without being read first, which halves the
 * host-memory traffic of the expansion.  A freshly allocated (never touched) destination is better
 * served by pst_host_widen: its pages are zeroed into the cache by the first-touch fault. */
int pst_host_widen_stream(const void *h_src, int32_t src_bits, void *h_dst, int32_t dst_bits, int64_t n,
                          int32_t threads);
/* 1 when pst_host_widen_stream uses non-temporal stores on this CPU, 0 when it falls back to ordinary
 * stores (no AVX-512): the default device->host transport is chosen from this and the thread count. */
int pst_host_stream_stores(void);
/* Advise transparent huge pages for a freshly allocated, still untouched result buffer (the fresh
 * int64 array the reference-shaped call returns): first-touch page faults are what bounds the host
 * expansion into pageable memory.  0 = advice given, 1 = not available; never an error. */
int pst_host_prepare(void *h_buffer, int64_t bytes);
/* h_dst[index[i] - base] = value[i] for base <= index[i] < base + n: writes the exact values of the
 * elements that saturated a narrow format (overflow list of pst_narrow_counts) into a widened chunk. */
int pst_host_apply_overflow(void *h_dst, int32_t dst_bits, int64_t base, int64_t n,
                            const int64_t *h_index, const int32_t *h_value, int64_t entries);
/* sum of the buffer read as uint32 words: the cheapest consumer that touches every byte (the sink
 * of the streamed many-cells benchmark; a transfer checksum). */
uint64_t pst_host_checksum(const void *h_src, int64_t bytes, int32_t threads);
/* zlib's crc32_combine: the CRC-32 of A || B from crc1 = crc32(A), crc2 = crc32(B) and len2 = |B|. */
uint32_t pst_host_crc32_combine(uint32_t crc1, uint32_t crc2, int64_t len2);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* PROSSTT_B200_H */
