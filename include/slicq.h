/* libslicq -- B200-native sliced constant-Q transform (sliCQT) analysis / synthesis.
 *
 * C ABI of the drop-in boundary.  The reference (sevagh/xumx-sliCQ V2) is pure Python/torch and
 * has no FFI of its own; these entry points are what a maintainer would bind (ctypes stub in
 * INTEGRATION.md) in place of the torch internals of
 *     xumx_slicq_v2/nsgt/slicq.py:182-196   NSGT_sliced.forward   -> slicq_forward
 *     xumx_slicq_v2/nsgt/slicq.py:198-230   NSGT_sliced.backward  -> slicq_inverse
 *     xumx_slicq_v2/nsgt/slicq.py:70-151    NSGT_sliced.__init__  -> slicq_plan_create
 * as called by the wrappers xumx_slicq_v2/transforms.py:106-131 (NSGT_SL.forward) and
 * transforms.py:154-178 (INSGT_SL.forward).
 *
 * Conventions
 *   - plain pointers and sizes only; all data pointers are DEVICE pointers owned by the caller
 *     (PyTorch); the library never allocates, frees or synchronises caller memory.
 *   - every call is asynchronous on the cudaStream_t passed in (as void*).
 *   - return value 0 = success, negative = SLICQ_E_* ; slicq_last_error() gives a thread-local
 *     human readable message.  No C++ exception crosses the boundary.
 *   - a plan is immutable after creation; calls on one plan are re-entrant across threads as
 *     long as they use distinct scratch buffers (large calls fork onto the plan's internal side
 *     streams: that enqueue sequence is serialised by a per-plan mutex, the GPU work is not).
 *   - a plan belongs to the device that was current in slicq_plan_create; one process may hold
 *     plans on several devices (kernel attributes are set per device).
 *   - "row"  = one flattened (batch x channel) signal,  "slice" = one 50 %-overlapping window of
 *     sl_len samples advancing by hop = sl_len/2,  "bin" = one frequency channel j with M_j
 *     coefficients per slice, "bucket" = maximal run of consecutive bins with equal M_j.
 */
#ifndef SLICQ_H
#define SLICQ_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SLICQ_ABI_VERSION 1

enum {
    SLICQ_OK = 0,
    SLICQ_E_INVALID = -1,      /* bad argument / shape                         */
    SLICQ_E_UNSUPPORTED = -2,  /* plan parameters no kernel was compiled for   */
    SLICQ_E_CUDA = -3,         /* CUDA runtime / launch failure                */
    SLICQ_E_SCRATCH = -4       /* scratch buffer too small                     */
};

/* Host-side filter-bank tables (what NSGT_sliced.__init__ derives: nsgt/nsgfwin_sl.py:8-111,
 * nsgt/util.py:72-116, nsgt/slicing.py:7-18).  All arrays are HOST pointers, copied at create. */
typedef struct slicq_tables {
    int32_t sl_len;        /* slice length L (multiple of 4)                              */
    int32_t n_bins;        /* J: bins 0..J-1 = DC, the scale's bins, Nyquist              */
    const int32_t* bin_M;  /* [J] coefficients per slice (multiple of 4)                  */
    const int32_t* bin_pos;/* [J] even centre position rfbas_j in FFT bins of the slice   */
    const float* win_fwd;  /* [sum M] analysis windows g_j[m] (peak at m = 0)             */
    const float* win_inv;  /* [sum M] dual windows gd_j[m]                                */
    const float* tukey;    /* [L] slicing window                                          */
    int32_t flags;         /* SLICQ_PLAN_* bits                                           */
} slicq_tables;

/* Plan flag: the ANALYSIS entry of this plan computes the adjoint (transpose) of the SYNTHESIS of the
 * normal plan -- used for autograd through INSGT_SL (the reference gets it from torch autograd on
 * nsgt/nsigtf.py + nsgt/unslicing.py).  The slice spectrum is scaled by 2/L (1/L at DC / Nyquist) and
 * bins reaching outside [0, L/2] read zeros instead of the Hermitian mirror; for bins that reach below DC the
 * analysis also adds the adjoint of the synthesis' mirrored-bin pass (nsgt/nsigtf.py:63-80).  The caller passes
 * tukey = 1 and win_fwd = gd * M^2. */
#define SLICQ_PLAN_ADJOINT_OF_SYNTHESIS 1
/* Plan flag: the SYNTHESIS entry of this plan computes the adjoint (transpose) of the ANALYSIS of the normal plan --
 * autograd through NSGT_SL (the reference gets it from torch autograd on nsgt/slicing.py + nsgt/nsgtf.py,
 * training.py:77-95).  Bin spectra that reach below DC / above Nyquist are folded back (conjugated) instead of
 * dropped, DC / Nyquist count twice, and the slice is multiplied by the slicing window before the overlap-add; the
 * caller passes win_inv = g * L / (2 M^2) and the normal tukey. */
#define SLICQ_PLAN_ADJOINT_OF_ANALYSIS 2

typedef struct slicq_plan slicq_plan; /* opaque */

/* One bucket of the ragged coefficient list as the caller's tensor lays it out.
 * Element (row, bin f in bucket, slice k, m) is ptr[row*s_row + f*s_bin + k*s_slice + m]
 * in complex64 units (interleaved re, im); the M axis must be contiguous. */
typedef struct slicq_bucket_view {
    void* ptr;
    int64_t s_row, s_bin, s_slice;
} slicq_bucket_view;

int slicq_abi_version(void);
/* 0 = CUDA build (the product), 1 = host emulation of the kernels (test infrastructure, tests/emu) */
int slicq_build_kind(void);
const char* slicq_last_error(void);

int slicq_plan_create(const slicq_tables* tables, slicq_plan** out);
void slicq_plan_destroy(slicq_plan* plan);

/* plan queries */
int slicq_plan_n_buckets(const slicq_plan* plan);
int slicq_plan_bucket_info(const slicq_plan* plan, int b, int32_t* first_bin, int32_t* n_bins, int32_t* M);
int64_t slicq_plan_num_slices(const slicq_plan* plan, int64_t n_samples);

/* Scratch (device) bytes needed by a forward / inverse call over n_rows x n_slices units.
 * Scratch holds the intermediate spectra of one chunk of units (analysis: padded half spectra, 73.6 KB per unit;
 * synthesis: two planes of windowed bin spectra, 147 KB per unit); SLICQ_CHUNK_MB bounds a chunk (default 2 GiB:
 * one chunk per call -- measured faster than L2-sized chunks, DESIGN.md section 8).  The scratch pointer must be 16-byte
 * aligned (its rows are moved with 16-byte vector and bulk copies); a misaligned one is refused with SLICQ_E_SCRATCH. */
size_t slicq_scratch_bytes(const slicq_plan* plan, int64_t n_rows, int64_t n_slices, int inverse);

/* Analysis.  x: [n_rows] rows of float32, row r at x + r*x_row_stride, n_samples valid samples
 * whose first one is global sample t0 (0 when x holds the whole signal).  Computes local slices
 * 0..n_slices-1 = global slices k0..k0+n_slices-1 (slice k covers global samples
 * [(k-1)*hop, (k+1)*hop); samples outside [t0, t0+n_samples) read as zero) and writes
 * buckets[b] for all plan buckets. */
int slicq_forward(const slicq_plan* plan, const float* x, int64_t n_rows, int64_t x_row_stride,
                  int64_t n_samples, int64_t t0, int64_t k0, int64_t n_slices,
                  const slicq_bucket_view* buckets, void* scratch, size_t scratch_bytes, void* stream);

/* Same as slicq_forward for the canonical packed layout: `coefs` is ONE allocation of
 * n_rows * n_slices * sum(M_j) complex64 in which bucket b is the contiguous block
 * [n_rows][F_b][n_slices][M_b], buckets in order (what the Python wrappers allocate). */
int slicq_forward_packed(const slicq_plan* plan, const float* x, int64_t n_rows, int64_t x_row_stride,
                         int64_t n_samples, int64_t t0, int64_t k0, int64_t n_slices, void* coefs,
                         void* scratch, size_t scratch_bytes, void* stream);

/* Analysis fused with the magnitude the model consumes (replaces the separate ComplexNorm pass,
 * xumx_slicq_v2/transforms.py:181-208 called at separator.py:338,346 and training.py; abs_of_real_complex
 * phase.py:116-118): besides the coefficients, norms[b] (fp32, logical shape [n_rows][F_b][S][M_b],
 * strides in floats, M contiguous) receives |c| = sqrt(re^2 + im^2) from the epilogue of the per-bin
 * transforms, so |X| costs 4 extra bytes per coefficient instead of an 8-byte read + 4-byte write pass. */
int slicq_forward_norm(const slicq_plan* plan, const float* x, int64_t n_rows, int64_t x_row_stride,
                       int64_t n_samples, int64_t t0, int64_t k0, int64_t n_slices,
                       const slicq_bucket_view* buckets, const slicq_bucket_view* norms, void* scratch,
                       size_t scratch_bytes, void* stream);
/* packed variant: `norms` is ONE allocation of n_rows * n_slices * sum(M_j) floats, same bucket order */
int slicq_forward_packed_norm(const slicq_plan* plan, const float* x, int64_t n_rows, int64_t x_row_stride,
                              int64_t n_samples, int64_t t0, int64_t k0, int64_t n_slices, void* coefs,
                              void* norms, void* scratch, size_t scratch_bytes, void* stream);

/* Synthesis.  y: [n_rows] rows, row r at y + r*y_row_stride, receives `length` samples whose
 * first one is global sample t0.  halo_out (optional, [n_rows][hop] float32) receives the part of
 * local slice 0 that belongs to the hop before this shard (only when k0 > 0). */
int slicq_inverse(const slicq_plan* plan, const slicq_bucket_view* buckets, int64_t n_rows,
                  int64_t n_slices, int64_t k0, float* y, int64_t y_row_stride, int64_t length,
                  int64_t t0, float* halo_out, void* scratch, size_t scratch_bytes, void* stream);

/* Synthesis fused with the realtime model's mask * mixture recombination (reference: Y_t =
 * mask_t * |X| * (cos, sin)(angle X) == mask_t * X, phase.py:96-113 called from model.py:258-265):
 * mix[b] holds the MIXTURE coefficients (n_rows rows), masks[b] an fp32 tensor with the logical shape
 * [n_targets * n_rows][F_b][S][M_b] (element strides in floats, M contiguous).  Output row
 * t * n_rows + r = synthesis of masks[t * n_rows + r] * mix[r]; y has n_targets * n_rows rows.
 * The four target coefficient sets are never materialised (24 instead of 32 bytes per coefficient). */
int slicq_inverse_masked(const slicq_plan* plan, const slicq_bucket_view* mix, const slicq_bucket_view* masks,
                         int64_t n_targets, int64_t n_rows, int64_t n_slices, int64_t k0, float* y,
                         int64_t y_row_stride, int64_t length, int64_t t0, float* halo_out, void* scratch,
                         size_t scratch_bytes, void* stream);

/* Gradient of slicq_inverse_masked with respect to its masks, for autograd through the fused synthesis.  Only valid on
 * a plan created with SLICQ_PLAN_ADJOINT_OF_SYNTHESIS (SLICQ_E_INVALID otherwise).  g: n_targets * n_rows rows of
 * float32 (row r at g + r*g_row_stride, n_samples valid samples from global sample t0), the gradient with respect to
 * slicq_inverse_masked's output in the same row order; mix: the n_rows MIXTURE rows that call read (read only).
 * grad_masks[b] (fp32, logical shape [n_targets * n_rows][F_b][S][M_b], strides in floats, M contiguous) receives
 *     grad[t * n_rows + r] = Re(conj(mix[r]) * (S^T g)[t * n_rows + r]),
 * S^T g the adjoint of the synthesis that this plan's analysis computes.  The product with the mixture is taken in the
 * epilogue of the per-bin transforms (and of the mirrored-bin adjoint for bins that reach below DC), so S^T g is never
 * written: 8 bytes read and 4 written per coefficient and target.  Scratch: slicq_scratch_bytes(plan,
 * n_targets * n_rows, n_slices, 0). */
int slicq_forward_mask_grad(const slicq_plan* plan, const float* g, int64_t n_targets, int64_t n_rows,
                            int64_t g_row_stride, int64_t n_samples, int64_t t0, int64_t k0, int64_t n_slices,
                            const slicq_bucket_view* mix, const slicq_bucket_view* grad_masks,
                            void* scratch, size_t scratch_bytes, void* stream);

/* number of kernel launches issued by this library since load (bench bookkeeping) */
int64_t slicq_launch_count(void);

/* Optional per-kernel timing with CUDA events on the launching stream (bench roofline accounting).
 * slicq_profile_read synchronises the recorded events, adds their durations (milliseconds) per
 * kernel id {0 slice_fft_fwd, 1 bins_fwd, 2 bins_inv, 3 slice_fft_inv (incl. overlap-add)} and resets. */
int slicq_profile_enable(int on);
int slicq_profile_read(double* ms /*[4]*/, int64_t* launches /*[4]*/);

#ifdef __cplusplus
}
#endif
#endif /* SLICQ_H */
