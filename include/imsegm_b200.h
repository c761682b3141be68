/*
 * imsegm_b200.h -- C-ABI of the B200-native SLIC -> descriptors -> GraphCut hot path of Borda/pyImSegm.
 *
 * Every entry point takes plain DEVICE pointers (unless a parameter says "host"), sizes and a CUDA stream
 * (cudaStream_t passed as void*), returns 0 on success or a negative isb_status, never allocates what it
 * returns and never throws.  isb_last_error() gives the message of the last failure on the calling thread.
 * The caller owns all buffers; `ws` is scratch the caller sizes with the matching *_workspace_bytes().
 * All launches are asynchronous on `stream` unless a parameter is documented as a host output.
 *
 * Each declaration names the reference interface it replaces (file:line under the reference repository).
 */
#ifndef IMSEGM_B200_H
#define IMSEGM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* isb_stream_t; /* cudaStream_t */

enum isb_status {
    ISB_OK = 0,
    ISB_ERR_ARG = -1,      /* bad argument (null pointer, non-positive size, unsupported dtype...) */
    ISB_ERR_CUDA = -2,     /* a CUDA runtime call failed; see isb_last_error() */
    ISB_ERR_CAPACITY = -3, /* a caller-sized table was too small (edge table, candidate list); retry larger */
    ISB_ERR_UNSUPPORTED = -4
};

enum isb_dtype { ISB_U8 = 0, ISB_U16 = 1, ISB_F32 = 2, ISB_F64 = 3 };

const char* isb_last_error(void);
int isb_abi_version(void);
/* number of kernels this library has launched since load (bench.py's gpu_launches) */
long long isb_launch_count(void);
/* a caller that replays a captured CUDA graph of this library's kernels reports the kernels of one replay here, so that
 * isb_launch_count() keeps counting kernels, not graph launches */
int isb_note_graph_replay(long long n_kernels);
/* per-stage device timers: CUDA events recorded on the launching stream around each stage's kernels while enabled.
 * isb_profile_collect() synchronises the recorded events and returns, per stage id, the summed milliseconds and
 * the number of timed launches (arrays of isb_profile_stage_count() entries); it clears the record list. */
int isb_profile_enable(int on);
int isb_profile_stage_count(void);
const char* isb_profile_stage_name(int id);
int isb_profile_collect(double* ms_out /* host */, long long* count_out /* host */);

/* ------------------------------------------------------------------------------------------------------------------
 * (i) SLIC -- replaces skimage.segmentation.slic as called from imsegm/superpixels.py:61-63
 *     slic(img f64[H,W,3] in [0,1], n_segments, compactness, sigma=1, enforce_connectivity=True, slic_zero)
 * ------------------------------------------------------------------------------------------------------------------ */

/* min-max rescale to [0,1] (imsegm/superpixels.py:53-54), gaussian pre-blur (scipy.ndimage semantics: symmetric
 * 1-D correlate, mode reflect, depth(len 1) -> rows -> cols), rgb2lab, multiply by ratio = 1/compactness.
 *   img        : [H,W,C] interleaved, C in {1,3} (gray is replicated, superpixels.py:50-51), dtype = isb_dtype
 *   w_half     : HOST pointer, radius+1 doubles, w_half[0] = centre tap (radius <= 8; radius 0 = no blur)
 *   lab_planar : out, [3,H,W] f64
 *   minmax_out : out, 4 doubles (device) -- [0] min and [1] max of the raw image ([2..3] scratch); max == min makes
 *                the result NaN
 *   rescale    : 1 = apply the reference wrapper's min-max rescale when (min != 0 or max != 1); 0 = never;
 *                2 = as 1 with the extrema the caller left in minmax_out[0..1] (row-band mode: the extrema of the whole
 *                image, merged by a collective from isb_image_minmax of every band) */
int isb_slic_prepare(const void* img, int dtype, int H, int W, int C, const double* w_half, int radius, double ratio,
                     int rescale, double* lab_planar, double* minmax_out /* room for 4 doubles */, isb_stream_t stream);

/* minimum and maximum of n samples (NaN ignored) -> minmax_out[0..1]; [2..3] scratch */
int isb_image_minmax(const void* img, int dtype, long long n, double* minmax_out /* room for 4 doubles */, isb_stream_t stream);

size_t isb_slic_kmeans_workspace_bytes(int H, int W, int n_seeds, int step_y, int step_x);

/* k-means sweeps of _slic_cython: window +-2*step about each centroid, lowest index wins ties, centroid = raster
 * order sequential double sums / count.  Bit-exact with oracle/slic_oracle.c by construction.
 *   seeds_yx  : [n_seeds,2] f64 (row, col) regular grid (device)
 *   labels    : out [H,W] i32;  centroids : optional out [n_seeds,5] f64 (y,x,L,a,b) */
int isb_slic_kmeans(const double* lab_planar, int H, int W, const double* seeds_yx, int n_seeds, int step_y, int step_x,
                    double step, int max_iter, int slic_zero, int32_t* labels, double* centroids, void* ws, size_t ws_bytes,
                    isb_stream_t stream);

/* Row-band form of the sweeps: one image taller than a GPU wants to hold (BASELINE config 5, SURVEY.md section 8e) is cut into
 * row bands, one per GPU.  The cluster state (centres, windows, bins) is replicated in every band's workspace and lives in
 * the coordinates of the whole image; a band holds pixel memory for its owned rows plus a halo of >= 2*step_y rows on either
 * side, assigns every row of that slab and sums the clusters whose centre row it owns (all their members are inside the slab;
 * a member further away -- an orphan that no window covers -- is counted in xchg[6 n_seeds] and the caller must then fall back
 * to one GPU).  Per sweep:
 *     isb_slic_band_assign -> isb_slic_band_update(xchg) -> [sum xchg as int64 over the bands] -> isb_slic_band_import(xchg)
 *     -> (SLICO: [max of maxdc_xchg as int64/uint64 over the bands]) -> isb_slic_band_finalize
 * xchg is [6*n_seeds + 1] int64: per cluster the bit patterns of (cy, cx, c0, c1, c2) and a state word (1 alive, 2 died),
 * all zero in every band but the owner's, so the integer sum is an exact merge (and keeps -0.0 and NaN payloads).  The labels
 * of the owned rows are bit-identical to isb_slic_kmeans on the whole image.  Workspace: isb_slic_kmeans_workspace_bytes of
 * the WHOLE image (image_rows, width). */
typedef struct isb_slic_band {
    int32_t slab_rows, width;   /* pixel memory held by this band: rows [y_off, y_off + slab_rows) of the image */
    int32_t image_rows, y_off;
    int32_t own_lo, own_hi;     /* global rows whose clusters this band sums; the bands' [own_lo, own_hi) partition the image */
    int32_t halo;               /* >= 2*step_y; the slab covers [own_lo - halo, own_hi + halo) clipped to the image */
    int32_t n_seeds, step_y, step_x, slic_zero;
    double step;
    const double* lab_slab;     /* plane c, slab row y, column x at lab_slab[c*plane_stride + y*width + x] */
    size_t plane_stride;
    const double* seeds_yx;     /* [n_seeds,2] seeds of the whole image */
    int32_t* labels_slab;       /* [slab_rows, width] */
    void* ws; size_t ws_bytes;
} isb_slic_band_t;
int isb_slic_band_begin(const isb_slic_band_t* band, isb_stream_t stream);
int isb_slic_band_assign(const isb_slic_band_t* band, isb_stream_t stream);
int isb_slic_band_update(const isb_slic_band_t* band, int64_t* xchg, isb_stream_t stream);
int isb_slic_band_import(const isb_slic_band_t* band, const int64_t* xchg, uint64_t* maxdc_xchg /* [n_seeds], SLICO only */,
                         isb_stream_t stream);
int isb_slic_band_finalize(const isb_slic_band_t* band, const uint64_t* maxdc_xchg, isb_stream_t stream);

size_t isb_connectivity_workspace_bytes(int H, int W);


/* _enforce_label_connectivity_cython: raster-order relabel of 4-connected components, BFS truncated at max_size,
 * components < min_size merged into the last already-labelled neighbour seen.  Bit-exact with the oracle.
 *   n_labels_out : device int32, number of output labels (labels are 0..n-1) */
int isb_enforce_connectivity(const int32_t* labels, int H, int W, int min_size, int max_size, int32_t* out,
                             int32_t* n_labels_out, void* ws, size_t ws_bytes, isb_stream_t stream);

/* SLIC of a single-channel VOLUME -- replaces skimage.segmentation.slic(vol, n_segments, compactness, multichannel=False,
 * spacing=space, sigma=1) as called from imsegm/superpixels.py:104-106 (segment_slic_img3d_gray).  Bit-exact with
 * oracle/slic3d_oracle.c.  Written for generality (the reference's volumes are small), see csrc/slic3d.cu.
 *   isb_slic3d_prepare : dtype -> f64 (img_as_float scale for the integer types), scipy gaussian_filter along z, y, x with the
 *                        DEVICE half kernels w_* (radius + 1 weights, [0] = centre; radius 0 / weight 1 = axis not blurred),
 *                        then * ratio (= 1 / compactness).  tmp: scratch of D*H*W doubles
 *   isb_slic3d_kmeans  : the sweeps of _slic_cython; seeds_zyx [n,3] (device); spacing_host: 3 HOST doubles (z, y, x) */
int isb_slic3d_prepare(const void* vol, int dtype, int D, int H, int W, const double* w_z, int r_z, const double* w_y, int r_y,
                       const double* w_x, int r_x, double ratio, double* tmp, double* out, isb_stream_t stream);
size_t isb_slic3d_kmeans_workspace_bytes(int D, int H, int W, int n_seeds);
int isb_slic3d_kmeans(const double* vol_scaled, int D, int H, int W, const double* seeds_zyx, int n_seeds, int step_z, int step_y,
                      int step_x, double step, const double* spacing_host, int max_iter, int32_t* labels, void* ws, size_t ws_bytes,
                      isb_stream_t stream);
/* _enforce_label_connectivity_cython on a volume (6 neighbours in the order x+1, x-1, y+1, y-1, z+1, z-1) */
size_t isb_connectivity3d_workspace_bytes(int D, int H, int W, int max_size);
int isb_enforce_connectivity3d(const int32_t* labels, int D, int H, int W, int min_size, int max_size, int32_t* out,
                               int32_t* n_labels_out, void* ws, size_t ws_bytes, isb_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * (ii) descriptors -- replaces imsegm/features_cython.pyx (the reference's only native module)
 * ------------------------------------------------------------------------------------------------------------------ */

/* computeColorImage2dMean :81, ...Energy :101, ...Variance :122 and normColorFeatures :59 in one launch family,
 * plus the centroids of imsegm/superpixels.py:205-224.  Pixels are converted to f32 (descriptors.py:233),
 * accumulated in f64.
 *   img     : [H,W,3] interleaved, dtype = isb_dtype (NaN -> 0 as descriptors.py:824)
 *   seg     : [H,W] i32 in [0, nb)
 *   flags   : bit0 mean, bit1 std, bit2 energy  -> feature columns in that order, 3 channels each
 *   feat    : out [nb, ld] f64, columns written at col0.. ; absent labels give 0
 *   centres : optional out [nb,2] f64 (row, col), (-1,-1) for absent labels;  counts: optional out [nb] i32 */
size_t isb_segment_stats_workspace_bytes(int nb);
int isb_segment_stats_2d(const void* img, int dtype, const int32_t* seg, int H, int W, int nb, int flags, double* feat,
                         int ld, int col0, double* centres, int32_t* counts, void* ws, size_t ws_bytes, isb_stream_t stream);

/* The same statistics with caller-owned accumulators, so that row bands of one image can be merged by a collective between
 * the calls: acc [nb,6] f64 (sum c0..c2, sum of squares c0..c2), iacc [nb,3] i64 (count, sum row, sum col), var [nb,3] f64
 * (squared deviations from the f32 mean).  accumulate / deviation ADD into acc+iacc / var (the caller zeroes them);
 * rows are global rows [y_off, y_off + H) of the image for the row sums. */
int isb_segment_stats_accumulate(const void* img, int dtype, const int32_t* seg, int H, int W, int y_off, int nb, double* acc,
                                 int64_t* iacc, isb_stream_t stream);
int isb_segment_stats_deviation(const void* img, int dtype, const int32_t* seg, int H, int W, int nb, const double* acc,
                                const int64_t* iacc, float* meanf_scratch /* [nb,3] */, double* var, isb_stream_t stream);
int isb_segment_stats_finish(int nb, int flags, const double* acc, const double* var, const int64_t* iacc, double* feat, int ld,
                             int col0, double* centres, int32_t* counts, isb_stream_t stream);

/* computeGrayImage3dMean :144 / Energy :169 / Variance :194 of features_cython.pyx: one channel, any rank (n voxels).
 *   flags bit0 mean, bit1 std, bit2 energy -> columns col0.. of feat [nb, ld] in that order */
size_t isb_gray_stats_workspace_bytes(int nb);
int isb_gray_stats(const void* img, int dtype, const int32_t* seg, long long n, int nb, int flags, double* feat, int ld, int col0,
                   void* ws, size_t ws_bytes, isb_stream_t stream);

/* computeLabelHistogram2d (features_cython.pyx:222): hist[l] = #{p : segm_select[p] == l >= 0 and struc_elem[p] == 1} */
int isb_label_hist_2d(const int16_t* segm_select, const int16_t* struc_elem, int H, int W, int nb_labels, uint32_t* hist,
                      isb_stream_t stream);

/* histogram_regions_labels_counts (imsegm/labeling.py:208-240, a per-pixel Python loop in the reference): joint histogram
 * hist[a][b] = #{p : slic[p] == a and annot[p] == b}, hist is [nb_slic, nb_annot] u32; labels must be in range */
int isb_region_label_hist(const int32_t* slic, const int32_t* annot, int H, int W, int nb_slic, int nb_annot, uint32_t* hist,
                          isb_stream_t stream);

/* compute_img_filter_response2d / 3d (imsegm/descriptors.py:951-983): per slice of img [n_slices, H, W] f64 the maximum over a
 * battery of kernels [n_kernels, kh, kw] f64 (odd sizes) of scipy.ndimage.convolve(slice, kernel) -- true convolution, mode
 * 'reflect'.  Generic FP64 utility for the gray-volume texture path; colour images use isb_lm_texture. */
int isb_filter_response_2d(const double* img, int n_slices, int H, int W, const double* kernels, int n_kernels, int kh, int kw,
                           double* out, isb_stream_t stream);

/* scipy.ndimage.gaussian_filter of every slice of img [n_slices, H, W] f64 (rows, then columns; symmetric 1-D correlate, mode
 * 'reflect'), what image_subtract_gauss_smooth (:986-1000) subtracts.  w_half: DEVICE, radius + 1 weights, [0] = centre;
 * tmp: scratch of the image's size */
int isb_gaussian_filter_2d(const double* img, int n_slices, int H, int W, const double* w_half, int radius, double* tmp, double* out,
                           isb_stream_t stream);

/* compute_label_histograms_positions (imsegm/descriptors.py:1288-1352) in one launch: for every position (row, col) and every
 * diameter d the histogram of the labels under the disc dy^2 + dx^2 <= d^2 (skimage.morphology.disk(d)) clipped to the image,
 * i.e. what compute_label_hist_segm (:1396) returns for the pair, and the pixel count of the clipped disc.
 *   segm  : [H, W] i32 labels, values outside [0, nb_labels) ignored;  or proba [H, W, nb_labels] f64 (then segm may be NULL):
 *           hist[l] = sum of proba[.., l] under the disc (compute_label_hist_proba :1501)
 *   positions [n_pos, 2] i32 (row, col), diameters [n_diam] i32;  hist out [n_pos, n_diam, nb_labels] f64, sizes out [n_pos, n_diam] f64
 *   selem : optional explicit structuring element [mh, mw] u8 (1 = inside) used instead of the discs (then n_diam must be 1,
 *           diameters may be NULL); mask pixel (iy, ix) lies on image pixel (row - mh/2 + iy, col - mw/2 + ix) as in
 *           adjust_bounding_box_crop (:1355) */
int isb_disc_label_hist(const int32_t* segm, const double* proba, int H, int W, const int32_t* positions, int n_pos,
                        const int32_t* diameters, int n_diam, const uint8_t* selem, int mh, int mw, int nb_labels, double* hist,
                        double* sizes, isb_stream_t stream);

/* computeRayFeaturesBinary2d (features_cython.pyx:239) for n_pos positions at once: out [n_pos, n_ang] f32, -1 where the ray
 * leaves the image, 0 where the position lies inside the border label (edge 'up').  sin_a / cos_a: the f32 sines and cosines
 * of the ray angles as the reference forms them (np.deg2rad of the f32 angle, stored to float).  edge: 1 'up', -1 'down'. */
int isb_ray_features_2d(const int8_t* seg_binary, int H, int W, const int32_t* positions, int n_pos, const float* sin_a,
                        const float* cos_a, int n_ang, int edge, float* out, isb_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * (iii) graph + energies + alpha-expansion
 * ------------------------------------------------------------------------------------------------------------------ */

/* make_graph_segm_connect_grid2d_conn4 (imsegm/superpixels.py:157-177) for labels already in [0, nb):
 * unique 4-connected label pairs (a < b) sorted by (b, a).
 *   edges : out [cap,2] i32;  n_edges_out : device int32 (if > cap the call reports ISB_ERR_CAPACITY lazily:
 *           the host must check n_edges_out <= cap) */
size_t isb_adjacency_workspace_bytes(int nb, int cap);
int isb_adjacency_edges(const int32_t* seg, int H, int W, int nb, int32_t* edges, int cap, int32_t* n_edges_out, void* ws,
                        size_t ws_bytes, isb_stream_t stream);

/* the same for a label VOLUME [D, H, W]: 6-connectivity (make_graph_segm_connect_grid3d_conn6, superpixels.py:180-202); same
 * workspace as isb_adjacency_edges.  isb_centroids_3d: centre (z, y, x) of every label, (-1,-1,-1) when absent
 * (superpixel_centers on a volume); ws: 4 * nb uint64 */
int isb_adjacency_edges_3d(const int32_t* seg, int D, int H, int W, int nb, int32_t* edges, int cap, int32_t* n_edges_out, void* ws,
                           size_t ws_bytes, isb_stream_t stream);
int isb_centroids_3d(const int32_t* seg, int D, int H, int W, int nb, double* centres, void* ws, size_t ws_bytes, isb_stream_t stream);

/* compute_unary_cost (imsegm/graph_cuts.py:523-540), compute_edge_weights / compute_edge_model / compute_spatial_dist
 * (:574-657, :383-439, :303-336), create_pairwise_matrix_uniform (:442-456), and pyGCO's float->int conversion.
 *   proba [N,K] f64, edges [E,2] i32 (n_edges read from device n_edges_dev when non-null, else E), centres [N,2] f64
 *   metric : 0 = constant 1, 1 = lT (max_k dp^2), 2 = l1, 3 = l2   -> w = exp(-d / (2 std(d)^2))
 *   spatial: 1 = divide by the relative centroid distance (the reference does so for edge_type 'model' and
 *            'spatial' exactly, not for 'model_l1' / 'model_l2', graph_cuts.py:646)
 *   out: unary [N,K] f64, edge_w [E] f64, and the integerised (unary_i [N,K], edge_wi [E], smooth_i [K,K]) i32 */
int isb_gc_energies(const double* proba, int N, const int32_t* n_nodes_dev /* optional device N */, int K, const int32_t* edges, int E,
                    const int32_t* n_edges_dev,
                    const double* centres, int metric, int spatial, double edge_cost, const double* pairwise /* [K,K] device */,
                    double* unary, double* edge_w, int32_t* unary_i, int32_t* edge_wi, int32_t* smooth_i, void* ws,
                    size_t ws_bytes, isb_stream_t stream);
size_t isb_gc_energies_workspace_bytes(int N, int K, int E);

/* gco.cut_general_graph(..., algorithm='expansion', n_iter) on integer energies (imsegm/graph_cuts.py:735-744).
 * One CTA cluster per graph; push-relabel max-flow; a site keeps its label iff it can reach the sink in the
 * residual graph (BK's SINK segment) so labels are identical to the oracle's.
 *   labels : in/out [N] i32 (initial labeling, zeros for the reference call);  energy_out : device int64 */
size_t isb_alpha_expansion_workspace_bytes(int N, int K, int E);
int isb_alpha_expansion(int N, const int32_t* n_nodes_dev /* optional device N */, int K, int E, const int32_t* n_edges_dev,
                        const int32_t* edges, const int32_t* edge_wi,
                        const int32_t* unary_i, const int32_t* smooth_i, int n_iter, int32_t* labels, int64_t* energy_out,
                        int32_t* stats_out /* optional [8]: moves, flows, sweeps, global relabels, BFS levels, smem flag, 0, 0 */, void* ws, size_t ws_bytes,
                        isb_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * class model -- replaces the host round trip of estim_class_model / predict_proba (imsegm/graph_cuts.py:73-163 default
 * 'GMM', imsegm/pipelines.py:95-96): StandardScaler + sklearn-style full-covariance GaussianMixture EM, n_init
 * restarts run concurrently (one CTA each), best lower bound wins.
 *   feat [N, ld] f64 (first D columns used), n_dev: optional device int32 with the real row count (<= N)
 *   init_labels: optional [n_init, N] i32 hard assignments (deterministic start); else k-means++/Lloyd from `seed`
 *   proba: out [N, K];  params_out: optional, isb_gmm_params_len(D, K) doubles:
 *     scaler mean[D] | scaler scale[D] | weights[K] | means[K,D] | covariances[K,D,D] | precisions_cholesky[K,D,D] |
 *     lower_bound | n_iter | converged | ok | best_init
 * ------------------------------------------------------------------------------------------------------------------ */
size_t isb_gmm_workspace_bytes(int N, int D, int K, int n_init);
int isb_gmm_params_len(int D, int K);
int isb_gmm_fit_predict(const double* feat, int N, int D, int ld, const int32_t* n_dev, int K, int n_init, int max_iter, double tol,
                        double reg_covar, int use_scaler, unsigned long long seed, const int32_t* init_labels, double* proba,
                        double* params_out, void* ws, size_t ws_bytes, isb_stream_t stream);

/* predict_proba of a GIVEN fitted mixture (GaussianMixture / BayesianGaussianMixture, any covariance type, optionally behind a
 * StandardScaler), packed on the host into one device vector of isb_gmm_model_len(D, K) doubles:
 *     shift[D] | scale[D] | U[K,D,D] | b[K,D] | c[K]
 *   U_k: upper-triangular precision Cholesky factor (row-major, zeros below the diagonal), b_k = means_k U_k,
 *   c_k: every term of log N_k + log weight_k that does not depend on the sample.
 * For each row n < min(N, *n_dev): x = (f - shift) / scale with NaN features taken as 0, q_k = |x U_k - b_k|^2,
 * lw_k = -(D log 2pi + q_k) / 2 + c_k, proba[n, k] = exp(lw_k - logsumexp(lw)).  Rows at or beyond the count are not written.
 * D <= 16 needs no workspace; 16 < D <= 232 runs the batched FP64 GEMM of the fit (K <= 8). */
int isb_gmm_model_len(int D, int K);
size_t isb_gmm_predict_workspace_bytes(int N, int D, int K);
int isb_gmm_predict(const double* feat, int N, int D, int ld, const int32_t* n_dev, int K, const double* model, double* proba, void* ws,
                    size_t ws_bytes, isb_stream_t stream);

/* compute_texture_desc_lm_img2d_clr (imsegm/descriptors.py:1041-1106): sigma-150 background subtraction (reflect, all three
 * axes), Leung-Malik filter bank (33x33 kernels) as an implicit GEMM on the tensor cores (tcgen05.mma kind::tf32 with the 3xTF32
 * split, FP32 accumulators in tensor memory, operands staged by TMA), max over the orientations of a battery, clip at 1e6,
 * log-norm scaling, per-superpixel mean / std / energy -- the responses never leave the SM.
 *   bg_weights : device, 2*bg_radius+1 doubles (scipy's gaussian kernel, sigma 150 -> radius 600); bg_radius 0 = no background
 *   chmix_host : HOST, 3x3 doubles: the same kernel folded onto the reflected length-3 channel axis
 *   w_tc       : device f32 [33 kernel rows][hi | lo][10 k-chunks][NP/8][8 filters][4 taps]: correlation-form (flipped) kernels in
 *                the operand layout of the contraction (K-major 8 x 16-byte core matrices), tf32-rounded value and tf32-rounded
 *                remainder, taps 33..39 and padding filters zero.  Filter (column) order: oriented batteries first (edge s0 |
 *                bar s0 | edge s1 | ..., `orient` filters each), then gauss / LoG / LoG2 per sigma
 *   (orient, NP, n_batt) = (8, 80, 20) full bank | (4, 48, 15) short bank;  flags as isb_segment_stats_2d
 *   feat       : out [nb, ld]: columns col0 + battery*3*nflags + stat*3 + channel (the reference's order) */
size_t isb_lm_workspace_bytes(int H, int W, int nb, int n_batt);
int isb_lm_texture(const void* img, int dtype, const int32_t* seg, int H, int W, int nb, const double* bg_weights, int bg_radius,
                   const double* chmix_host, const float* w_tc, int NP, int orient, int n_batt, int flags,
                   double* feat, int ld, int col0, void* ws, size_t ws_bytes, isb_stream_t stream);
/* The same descriptor for ONE image cut into row bands over several GPUs (SURVEY 8(e), "one huge image"): every band runs
 * isb_lm_texture_accumulate on its slab [slab_rows, W, 3] = the rows it owns, [y_first, y_end) in slab coordinates, plus a halo of
 * bg_radius + 16 rows on every side that is not an image border (at a border the slab ends and reflects like the image); seg points
 * at the slab's first row of the label map.  The sums of the owned rows are ADDED to acc (isb_lm_acc_doubles(nb, n_batt) doubles:
 * sum r | sum r^2 | per-battery global sum r^2) and counts [nb] -- the caller zeroes them, sums them over the bands (all_reduce),
 * and isb_lm_texture_finish forms the same features isb_lm_texture writes. */
size_t isb_lm_acc_doubles(int nb, int n_batt);
int isb_lm_texture_accumulate(const void* img, int dtype, const int32_t* seg, int slab_rows, int W, int y_first, int y_end, int nb,
                              const double* bg_weights, int bg_radius, const double* chmix_host, const float* w_tc, int NP, int orient,
                              int n_batt, double* acc, int32_t* counts, void* ws, size_t ws_bytes, isb_stream_t stream);
int isb_lm_texture_finish(int nb, int n_batt, int flags, const double* acc, const int32_t* counts, double* feat, int ld, int col0,
                          isb_stream_t stream);

/* known-answer test of the tensor-core plumbing (tests/test_gpu_umma.py): D[128, N] = A[128, K] * B[N, K]^T with tcgen05.mma
 * kind::tf32 in one CTA; A, B row-major f32 holding tf32-representable values, N % 16 == 0 (<= 256), K % 8 == 0 (<= 64).
 * variant 0 = the descriptor convention the library uses; 1 = leading/stride byte offsets swapped (diagnostic only);
 * 2 = A written into tensor memory with tcgen05.st and read from there by the instruction (the form the contraction uses). */
int isb_umma_selftest(const float* A, const float* B, int N, int K, int variant, float* D, isb_stream_t stream);
/* profiling aid: clocks that `reps` back-to-back tcgen05.mma kind::tf32 instructions (M 128, K 8, the given N) take on each of `ctas`
 * CTAs; mode bit 0 = rotate over several accumulators, bit 1 = A operand from tensor memory.  cycles: device, [ctas] int64 */
int isb_umma_rate(int N, int reps, int mode, int ctas, long long* cycles, isb_stream_t stream);
/* profiling aid: clocks per dependent FP64 add / multiply / fma (one warp, chains of n operations); out: device, 4 doubles */
int isb_fp64_latency(int n, double* out, isb_stream_t stream);

/* per-segment, per-channel median -- numpy_img2d_color_median (imsegm/descriptors.py:420-455, channels = 3, n_px = H*W) and
 * numpy_img3d_gray_median (:651-676, channels = 1, n_px = D*H*W); np.median semantics (mean of the two middle values for an even
 * count), NaN for a label without pixels.
 *   img : [n_px, channels] interleaved, dtype = isb_dtype;  seg : [n_px] labels in [0, nb);  out : [nb, channels] f64 */
size_t isb_segment_median_workspace_bytes(long long n_px, int nb);
int isb_segment_median(const void* img, int dtype, const int32_t* seg, long long n_px, int channels, int nb, double* out, void* ws,
                       size_t ws_bytes, isb_stream_t stream);

/* skimage.morphology.opening(mask, disk(radius)) of a binary mask as imsegm/descriptors.py:1873-1876 applies it before tracing Ray
 * features: erosion then dilation with a disc, borders reflected.  mask / tmp / out : [H, W] uint8 (0 / 1) */
int isb_binary_opening_disk(const uint8_t* mask, int H, int W, int radius, uint8_t* tmp, uint8_t* out, isb_stream_t stream);

/* dst[0..n) = value (initial labeling of isb_alpha_expansion and similar small fills) */
int isb_fill_i32(int32_t* dst, long long n, int32_t value, isb_stream_t stream);

/* dst[i] = dst[i] (op) src[i] over n 8-byte words; op 0 int64 sum, 1 int64 max, 2 f64 min, 3 f64 max, 4 f64 sum.  What a
 * collective does between GPUs in row-band mode, for several bands held by one GPU. */
int isb_combine(void* dst, const void* src, long long n, int op, isb_stream_t stream);

/* final LUT gathers of imsegm/pipelines.py:104,109:  segm = graph_labels[slic], segm_soft = proba[slic]
 *   lut_i [nb] i32 (optional), lut_p [nb,K] f64 (optional); outputs [H,W] i32 / [H,W,K] f64 */
int isb_gather(const int32_t* seg, long long npx, const int32_t* lut_i, const double* lut_p, int K, int32_t* out_i,
               double* out_p, isb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* IMSEGM_B200_H */
