/* dctp.h - C ABI of libdctp.so: the B200 (sm_100a) DCT importance-score path.
 *
 * Drop-in boundary for the importance-generation hot path of semchan/DCT_Pruning.  The reference
 * has no native layer; each entry point below names the Python it replaces (file:line under
 * /root/reference).  A maintainer binds these with ctypes (see INTEGRATION.md); the shipped Python
 * host side (dct_pruning_b200/_lib.py) does exactly that.
 *
 * Conventions
 *   - plain pointers and sizes only; every `stream` is a cudaStream_t passed as void* (0 = default stream)
 *   - pointers named x / accum / scores / out ... are DEVICE pointers owned by the caller unless the
 *     name ends in _host; the library allocates only its cached cosine bases, a status word and the
 *     scratch of the *_host convenience entry, all released by dctp_shutdown()
 *   - return value: 0 on success, a negative DCTP_E_* code otherwise; dctp_last_error() gives the text
 *   - no C++ exception crosses the boundary, nothing calls exit(), there is NO CPU fallback:
 *     without a CUDA device every compute entry returns DCTP_E_CUDA
 *   - one host thread per process drives the library (forward hooks fire on the forward thread);
 *     calls are asynchronous on `stream` unless stated otherwise
 *   - the tensor-core score kernels are launched with programmatic stream serialization: their prologue may overlap
 *     the tail of the preceding kernel on the stream, but they wait for that kernel (and its memory) to complete
 *     before the first activation byte is read - ordinary stream semantics for the caller; DCTP_PDL=0 in the
 *     environment falls back to plain launches
 */
#ifndef DCTP_H
#define DCTP_H

#ifdef __cplusplus
extern "C" {
#endif

#define DCTP_VERSION 100          /* 0.1.0 */

#define DCTP_OK            0
#define DCTP_E_INVALID    -1      /* bad argument (null pointer, non-positive size, window out of range) */
#define DCTP_E_CUDA       -2      /* CUDA runtime error; text in dctp_last_error() */
#define DCTP_E_UNSUPPORTED -3     /* shape / layout the requested kernel path does not take */
#define DCTP_E_DEVICE     -4      /* a kernel reported a fault in the device status word (tensor-core wait timed out,
                                     channel index out of range in dctp_gather_weight) */

/* kernel path for dctp_score_accum */
#define DCTP_PATH_AUTO   0        /* the fastest tensor-core kernel the shape allows, CUDA cores otherwise */
#define DCTP_PATH_UMMA   1        /* tcgen05/TMEM bf16x3 kernel, operands in shared memory; square maps, side <= 128, contiguous maps */
#define DCTP_PATH_SIMT   2        /* fp32 CUDA-core kernels; any H x W, strided rows */
#define DCTP_PATH_TMEM   3        /* tcgen05 kernel with TMEM-resident operands; dense square maps, side 5..64 (odd sides up to 13) */
#define DCTP_PATH_LARGE  4        /* tiled tcgen05 kernel; dense square maps, side 80..320, side % 16 == 0 */
#define DCTP_PATH_STACK  5        /* warp-specialised tcgen05 kernel, TMA-staged tiles, stacked hi/lo basis in TMEM; dense square maps,
                                     even side 10..64 (above 32: multiples of 4).  AUTO's choice for these shapes */
#define DCTP_PATH_KRON   6        /* single-stage Kronecker tcgen05 kernel (C_N (x) C_N resident in shared memory, one map per TMEM
                                     lane, TMA-staged tiles); dense square maps of side <= 8.  AUTO's choice for these shapes */

int dctp_version(void);
const char* dctp_last_error(void);

/* Bind to the current CUDA device, set kernel attributes, allocate the status word.  Idempotent. */
int dctp_init(void);
/* Free every cached basis / scratch buffer.  The library can be re-initialised afterwards. */
int dctp_shutdown(void);

/* Build and upload the cosine bases an H x W map needs (synchronous, cached per size).  Called
 * implicitly by dctp_score_accum on first use of a size; call it ahead of time when the scoring
 * calls must stay asynchronous / CUDA-graph capturable. */
int dctp_prepare(int H, int W);

/* Fused hook kernel.  Replaces get_feature_hook / get_feature_hook_densenet /
 * get_feature_hook_u2net_input (utils/common.py:262-277, :280-293, :296-309) up to the per-channel
 * batch sum `c.view(a,-1).sum(0)` (:273-274):
 *
 *   accum[j] += sum_{b < B} sum_{u,v} DCT2_ortho(x[b, c_begin + j])[u,v]^2        j in [0, c_count)
 *
 * x           fp32 activation, element (b, c, h, w) at x[b*stride_b + c*stride_c + h*stride_h + w]
 *             (strides in elements, innermost stride 1)
 * c_begin/c_count  scored channel window (DenseNet variant: the last 12 channels, common.py:285)
 * accum       fp64 [c_count], caller-zeroed before the first batch, accumulated across calls
 * energy_out  optional fp32 [B * c_count]: per-(image, channel) energies, image-major (may be NULL)
 * coeff_out   optional fp32 [B * c_count * H * W]: the DCT coefficients themselves (debug / parity; NULL in production)
 * path        DCTP_PATH_*
 *
 * Non-finite input.  Call a map non-finite if one of its elements is NaN or +-Inf.  As in the reference, which scores every
 * (image, channel) slice on its own, a non-finite map changes only its own channel:
 *   1. a channel with a non-finite map gets a non-finite accum entry, and the map a non-finite energy_out entry (NaN or Inf);
 *   2. every other channel and map gets the value it would get without that map; a dead map (all +0.0 or all -0.0) scores
 *      exactly 0, also in the same tile as a non-finite map;
 *   3. DCTP_OP_DCT3: values_out[b] is non-finite exactly for the images with a non-finite map inside the window;
 *   4. the call sets no status word for it: dctp_check returns DCTP_OK, also when every map is non-finite.
 * The tensor-core kernels that put several maps into one MMA test every contribution to accum / energy_out for finiteness and
 * recompute a non-finite one in fp64 from the map in global memory.  A finite map whose fp32 energy overflows (elements of about
 * 1e18 and more) is outside these rules: depending on the kernel its channel gets Inf or an fp64 value.  coeff_out of a map that
 * shares a tile with a non-finite map is not specified: it is a debug dump. */
int dctp_score_accum(const float* x, int B, int H, int W,
                     long long stride_b, long long stride_c, long long stride_h,
                     int c_begin, int c_count,
                     double* accum, float* energy_out, float* coeff_out,
                     int path, void* stream);

/* Element type of an activation (dctp_score_accum_ex, dctp_score_accum_multi_ex). */
#define DCTP_DTYPE_F32   0
#define DCTP_DTYPE_BF16  1        /* the activations of a forward pass under torch.autocast(dtype=torch.bfloat16) */
#define DCTP_DTYPE_F16   2        /* ... under torch.autocast(dtype=torch.float16) */

/* dctp_score_accum for an activation x of element type `dtype` (DCTP_DTYPE_*; anything else: DCTP_E_INVALID).  Every shape, layout
 * and path dctp_score_accum takes is taken, with the same results for the values x holds: the energies are those of the maps widened
 * to fp32 (exactly), and the non-finite rules above hold unchanged.  accum, energy_out and coeff_out are fp64 / fp32 as there.
 * dctp_score_accum(...) is dctp_score_accum_ex(x, DCTP_DTYPE_F32, ...).
 * 16-bit maps that DCTP_PATH_KRON or DCTP_PATH_STACK take (AUTO's choice or forced) are read by those kernels directly: 2 bytes per
 * element.  Every other 16-bit call widens its scored window into a dense fp32 copy, allocated and freed on `stream`
 * (stream-ordered, graph-capturable: call dctp_prepare first, as for fp32), and scores that copy as dctp_score_accum would with the
 * same path: one extra launch, and 2 + 4 + 4 bytes of traffic per element. */
int dctp_score_accum_ex(const void* x, int dtype, int B, int H, int W,
                        long long stride_b, long long stride_c, long long stride_h,
                        int c_begin, int c_count,
                        double* accum, float* energy_out, float* coeff_out,
                        int path, void* stream);

/* Several hook sites in ONE launch.  The forward pass of the CIFAR nets and of U^2-Netp's small stages fires tens of hooks on
 * activations of a few MB; scored one by one they are bound by the host's launch rate (~12 us per hook), not by the GPU.  The host
 * side may therefore hold on to a run of activations of the same map size and hand them over together
 * (dct_pruning_b200.hooks.ScoreSession does: the deferred form of get_feature_hook, utils/common.py:262-277, one call per run of
 * same-sized sites instead of one per site).  Every site is DENSE: x points at its first scored map (the channel window already
 * applied) and B * c_count maps of H x W floats follow back to back; accum as in dctp_score_accum.  Map sizes the multi-site
 * kernels take (square; side <= 8, even side 10..64 - above 32 a multiple of 4 -, or side 80..320 a multiple of 16) are scored 16 sites per launch;
 * any other shape falls back to one launch per site.  Results are identical to n_sites dctp_score_accum calls. */
typedef struct dctp_site {
    const void* x;                /* first scored element, of the call's dtype (fp32 for dctp_score_accum_multi) */
    double* accum;
    int B;
    int c_count;
} dctp_site;
int dctp_score_accum_multi(const dctp_site* sites, int n_sites, int H, int W, void* stream);
/* The same for sites of element type `dtype` (DCTP_DTYPE_*).  16-bit sites of the shapes the Kronecker and stacked-basis kernels take
 * are scored 16 per launch as above; 16-bit sites of any other shape go through dctp_score_accum_ex one by one. */
int dctp_score_accum_multi_ex(const dctp_site* sites, int n_sites, int H, int W, int dtype, void* stream);

/* Alternative per-slice scoring ops behind the same accumulate / finalise / top-k plumbing: the two lines the reference keeps
 * commented out beside the DCT in get_feature_hook and compares against in chart*.py.
 *   DCTP_OP_DCT2     utils/common.py:267  dct_2d energy per (image, channel)             == dctp_score_accum(..., DCTP_PATH_AUTO)
 *   DCTP_OP_RANK     utils/common.py:268  torch.matrix_rank(output[i,j,:,:]) (HRank): accum[j] += sum_b rank(x[b, c_begin + j]),
 *                    rank = #{sigma > sigma_max * max(H, W) * eps_fp32} of the fp32 map (one-sided Jacobi SVD on the GPU)
 *   DCTP_OP_RANK_SQ  the same line left in front of the unchanged cnt_score (:249-255, :271), which squares every entry:
 *                    accum[j] += sum_b rank^2
 *   DCTP_OP_DCT3     utils/common.py:269  dct_3d(output[i,:,:,:]) -> cnt_score: ONE value per image, accum[0] += sum_b energy of the
 *                    3-D coefficient cube over channels [c_begin, c_begin + c_count) (accum has ONE entry for this op)
 * values_out  optional fp32: per-(image, channel) value [B * c_count] for DCT2 / RANK / RANK_SQ, per-image energy [B] for DCT3.
 * RANK / RANK_SQ hold a map in shared memory: longer side m <= 256 and (n * (m | 1) + n + 1) * 4 bytes <= 200 KiB, n the shorter
 * side, which is side <= 225 for square maps and shorter side <= 198 at a longer side of 256 (DCTP_E_UNSUPPORTED beyond).
 * Every call may run on its own stream: DCT3 allocates its scratch on the caller's stream (stream-ordered, graph-capturable). */
#define DCTP_OP_DCT2     0
#define DCTP_OP_RANK     1
#define DCTP_OP_RANK_SQ  2
#define DCTP_OP_DCT3     3
int dctp_score_op(int op, const float* x, int B, int H, int W,
                  long long stride_b, long long stride_c, long long stride_h,
                  int c_begin, int c_count, double* accum, float* values_out, void* stream);

/* out[i] = (float)(accum[i] / n_images).  Replaces the running mean over images
 * (utils/common.py:275-277) and the fp32 vector np.save writes (:394). */
int dctp_finalize(const double* accum, double n_images, float* out, int n, void* stream);

/* Segmented top-k: for segment s, scores[seg_offsets[s] .. seg_offsets[s+1]) are one layer's channel
 * scores; writes the seg_k[s] kept channel ids (relative to the segment, ascending, int64) at
 * out_idx[out_offsets[s] ...].  Replaces `np.argsort(imp)[C-k:]` + `.sort()`
 * (utils/load_models.py:39-41, :102-104, :265-267, :313-315, :352-354, :407-409, :469-471, :521-523,
 * :629-631 ... :746-748) with the stable tie rule (ties at the cut keep the highest channel ids).
 * All four index arrays are device pointers; seg_offsets / out_offsets have n_seg + 1 entries. */
int dctp_topk_segmented(const float* scores, const int* seg_offsets, const int* seg_k, int n_seg,
                        long long* out_idx, const int* out_offsets, void* stream);

/* Pruned-weight gather (the step downstream of top-k):
 *   out[i][j][r] = w[sel_out ? sel_out[i] : i][sel_in ? sel_in[j] : j][r],  i < k_out, j < k_in, r < inner
 * w is [c_out][c_in][inner] fp32 contiguous (inner = kH*kW; 1 with c_in = 1 for BatchNorm / bias vectors), out is
 * [k_out][k_in][inner]; sel_out / sel_in are device int64 arrays or NULL for "all, in order" (then k == c).
 * Replaces the element-wise Python copy loops of utils/load_models.py:43-51, :106-114, :482-500, :526-542,
 * :633-639 ...  An index outside [0, c) sets the device status word (reported by dctp_check). */
int dctp_gather_weight(const float* w, int c_out, int c_in, int inner, const long long* sel_out, int k_out,
                       const long long* sel_in, int k_in, float* out, void* stream);

/* Synchronise `stream` and report the device status word (DCTP_OK or DCTP_E_DEVICE); clears it. */
int dctp_check(void* stream);

/* Host-buffer convenience: score one activation that lives in HOST memory.  Copies x_host
 * (contiguous [B, C, H, W] fp32) to the device, scores channels [c_begin, c_begin + c_count),
 * divides by B and writes fp32 scores_host[c_count].  Synchronous.  This is the whole of
 * get_feature_hook for one batch behind one call, for callers without a device tensor. */
int dctp_score_host(const float* x_host, int B, int C, int H, int W, int c_begin, int c_count,
                    float* scores_host, int path);

/* Introspection for tests and benchmarks: which kernel path AUTO picks for a shape (DCTP_PATH_*),
 * the number of kernel launches issued by this library since dctp_init(), SM count of the device. */
int dctp_path_for(int H, int W, long long stride_h);
/* resident CTAs per SM of the tensor-core kernel instantiation (kp in {64,128}; load mode 0..5: dense
 * 8/4/2-byte scatter, generic 128/64/32-bit loads) at a typical table size.  DCTP_E_UNSUPPORTED for kp 128
 * with mode 2: no side that kernel serves has 2-byte scatter entries, so that instantiation is not built. */
int dctp_occupancy(int kp, int mode);
long long dctp_launch_count(void);
/* Name of the kernel instantiation the most recent dctp_score_accum call launched (AUTO's choice made visible: bench.py labels
 * its per-kernel table with it instead of re-deriving the dispatch; 16-bit instantiations carry ",IN=bf16" / ",IN=f16").  Static
 * storage, valid until the next score call. */
const char* dctp_last_kernel(void);
int dctp_sm_count(void);

#ifdef __cplusplus
}
#endif
#endif /* DCTP_H */
