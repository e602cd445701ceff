// C-ABI of libslicq (include/slicq.h): plan construction and the chunked launch sequences.
//
// forward  : per chunk of (row,slice) units   slice_fft_fwd_kernel -> bins_fwd_kernel [-> mirror_adj_kernel]
//            (slicq_forward_mask_grad: the same sequence, bins_fwd_kernel / mirror_adj_kernel in their mask-gradient mode)
// inverse  : per chunk                         bins_inv_kernel [-> mirror_fix_kernel] -> slice_fft_inv_kernel (even slices,
//                                              then odd slices)
//            (bins_inv_ovr_kernel in place of bins_inv_kernel for plans whose overflow spans several transform runs)
// (the bracketed kernels only for bins that reach below DC; mirror_adj_kernel only in the adjoint-of-synthesis plan)
// A chunk's intermediate spectra (analysis: padded half spectra H; synthesis: the two bin planes T) live in the
// caller-provided scratch buffer; SLICQ_CHUNK_MB bounds the chunk (default: one chunk per call).
#include "slicq_common.cuh"
#include "../../include/slicq.h"

#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <vector>
#include <algorithm>
#include <atomic>
#include <memory>
#include <mutex>

#ifdef SLICQ_EMU
#include <condition_variable>
#include <mutex>
#include <thread>
thread_local dim3 threadIdx;
dim3 blockIdx, blockDim, gridDim;
static unsigned char slicq_emu_smem_buf[256 * 1024] __attribute__((aligned(16)));
unsigned char* slicq_emu_smem = slicq_emu_smem_buf;
namespace {
struct EmuBarrier {
    std::mutex m; std::condition_variable cv; int count = 0, gen = 0, n = 1;
    void wait() {
        std::unique_lock<std::mutex> lk(m);
        const int g = gen;
        if (++count == n) { count = 0; ++gen; cv.notify_all(); }
        else cv.wait(lk, [&] { return gen != g; });
    }
} g_emu_bar;
}  // namespace
void slicq_emu_sync() { g_emu_bar.wait(); }
void slicq_emu_launch(dim3 grid, dim3 block, const std::function<void()>& body) {
    gridDim = grid; blockDim = block; g_emu_bar.n = (int)block.x;
    std::vector<std::thread> th(block.x);
    for (unsigned bz = 0; bz < grid.z; ++bz)
        for (unsigned by = 0; by < grid.y; ++by)
            for (unsigned bx = 0; bx < grid.x; ++bx) {
                blockIdx = dim3(bx, by, bz);
                for (unsigned t = 0; t < block.x; ++t)
                    th[t] = std::thread([t, &body]() { threadIdx = dim3(t, 0, 0); body(); });
                for (unsigned t = 0; t < block.x; ++t) th[t].join();
            }
}
#endif

extern "C" int slicq_launch_bins(const SlicqBinsParams* p, int n_tiles, int smem_bytes, SlicqBinsKernel k, cudaStream_t s);
extern "C" int slicq_launch_slice_fwd(const SlicqSliceParams* p, cudaStream_t s);
extern "C" int slicq_launch_slice_inv(const SlicqSliceParams* p, cudaStream_t s);
extern "C" int slicq_slice_smem_bytes(int L);
extern "C" int slicq_launch_mirror_fix(const SlicqBinsParams* p, cudaStream_t s);
extern "C" int slicq_launch_mirror_adj(const SlicqBinsParams* p, cudaStream_t s);

namespace {

const int kTunedSliceLen = 18060;      // slice length of the tuned prime-factor slice kernels (k_slice.cu, 2 * Pfa9030::N)

thread_local std::string g_err;
std::atomic<long long> g_launches{0};

// ---- optional per-kernel CUDA-event timing (bench.py roofline accounting) -----------------
enum { K_SLICE_FWD = 0, K_BINS_FWD, K_BINS_INV, K_SLICE_INV, K_COUNT };
std::atomic<bool> g_prof{false};
#ifndef SLICQ_EMU
struct ProfRec { int kid; cudaEvent_t a, b; };
std::vector<ProfRec> g_prof_recs;
std::mutex g_prof_mutex;
#endif
struct ProfScope {
#ifndef SLICQ_EMU
    int kid; cudaStream_t s; cudaEvent_t a, b; bool on;
    ProfScope(int k, cudaStream_t st) : kid(k), s(st), on(g_prof) {
        if (on) { cudaEventCreate(&a); cudaEventCreate(&b); cudaEventRecord(a, s); }
    }
    ~ProfScope() {
        if (on) { cudaEventRecord(b, s); ProfRec r; r.kid = kid; r.a = a; r.b = b; std::lock_guard<std::mutex> lk(g_prof_mutex); g_prof_recs.push_back(r); }
    }
#else
    ProfScope(int, cudaStream_t) {}
#endif
};

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}

struct FftPlan { int M, kind, A, B, cost; };
const FftPlan kFftPlans[] = {
#define SLICQ_FFT_SIZE(M_, K_, A_, B_, C_) {M_, K_, A_, B_, C_},
#include "fft_sizes.inc"
#undef SLICQ_FFT_SIZE
};

const FftPlan* find_fft_plan(int M) {
    for (size_t i = 0; i < sizeof(kFftPlans) / sizeof(kFftPlans[0]); ++i)
        if (kFftPlans[i].M == M) return &kFftPlans[i];
    return nullptr;
}

// shared-memory bytes one transform of this plan needs (max over analysis / synthesis)
int fft_smem_per_transform(const FftPlan& f) {
    if (f.kind == 1) return (f.M + 1) * 8;
    if (f.kind == 2) {
        const int bp = (f.B % 2 == 0) ? f.B + 1 : f.B;
        const int ap = (f.A % 2 == 0) ? f.A + 1 : f.A;
        const int a = f.A * bp, b = f.B * ap;
        return (a > b ? a : b) * 8;
    }
    return (f.M + f.A) * 8;  // kind 3: [R][P] (synthesis) / [P][R + 1] (analysis) complex
}

// threads one transform occupies in the pass whose per-thread state is hoisted out of the unit loop
int fft_threads_per_transform(const FftPlan& f) {
    if (f.kind == 1) return 1;
    if (f.kind == 2) return f.B;
    return f.B * (f.A <= 41 ? 2 : (f.A <= 61 ? 3 : 4));  // kind 3: (part, n2): the DFT-P is split by outputs over 2-4 threads
}

struct Bucket {
    int M, first_bin, n_bins, gt, tw_off, kind, A, B, smem_per_fft;
    int gap_first, gap_n;   // entries of the gap list (zero-filled positions of T) this bucket owns
    double cost;     // relative work per unit (for the job split)
};

template <class T> int upload(const std::vector<T>& h, const T** d, std::vector<void*>& owned) {
    void* p = nullptr;
    if (cudaMalloc(&p, h.size() * sizeof(T)) != cudaSuccess) return -1;
    if (cudaMemcpy(p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice) != cudaSuccess) return -1;
    owned.push_back(p);
    *d = reinterpret_cast<const T*>(p);
    return 0;
}

}  // namespace

struct slicq_plan {
    int L, N2, hop, J;
    std::vector<int> bin_M, bin_pos, bin_coff;
    std::vector<Bucket> buckets;
    SlicqDeviceTables dev;
    std::vector<void*> owned;
    int bins_smem;        // dynamic shared memory of the bins kernels
    bool ov_multi_run;    // a two-pass / prime bin diverts more than its first run of outputs: synthesis by bins_inv_ovr_kernel
    long long spec_stride_fwd;
    long long t_stride;   // complex elements per unit of the synthesis intermediate T
    long long chunk_bytes;
    // Large calls are split by rows into two halves that run on two internal streams (forked from and
    // joined back into the caller's stream): the memory-latency-bound and the issue-bound kernels of
    // the two halves overlap on the SMs.  Rows are independent, so the results do not change.
    long long split_units;          // split when the call has at least this many units (0 = never)
    mutable cudaStream_t side[2];
    mutable cudaEvent_t ev_fork, ev_join[2];
    mutable bool side_ready;
    // calls that split share the side streams and the fork / join events: their enqueue sequence (record, waits, launches,
    // joins) runs under this mutex, so that one thread's waits always see its own records.  Un-split calls take no lock.
    mutable std::mutex split_mutex;
};

extern "C" int slicq_abi_version(void) { return SLICQ_ABI_VERSION; }
#ifdef SLICQ_EMU
extern "C" int slicq_build_kind(void) { return 1; }
#else
extern "C" int slicq_build_kind(void) { return 0; }
#endif
extern "C" const char* slicq_last_error(void) { return g_err.c_str(); }
extern "C" int64_t slicq_launch_count(void) { return g_launches.load(); }

extern "C" int slicq_profile_enable(int on) { g_prof = on != 0; return SLICQ_OK; }

extern "C" int slicq_profile_read(double* ms, int64_t* launches) {
    for (int i = 0; i < K_COUNT; ++i) { if (ms) ms[i] = 0.0; if (launches) launches[i] = 0; }
#ifndef SLICQ_EMU
    std::lock_guard<std::mutex> lk(g_prof_mutex);
    for (ProfRec& r : g_prof_recs) {
        float t = 0.f;
        if (cudaEventSynchronize(r.b) == cudaSuccess && cudaEventElapsedTime(&t, r.a, r.b) == cudaSuccess) {
            if (ms) ms[r.kid] += t;
            if (launches) launches[r.kid] += 1;
        }
        cudaEventDestroy(r.a); cudaEventDestroy(r.b);
    }
    g_prof_recs.clear();
#endif
    return SLICQ_OK;
}

extern "C" void slicq_plan_destroy(slicq_plan* p) {
    if (!p) return;
    if (p->side_ready) {
        for (int h = 0; h < 2; ++h) { cudaStreamDestroy(p->side[h]); cudaEventDestroy(p->ev_join[h]); }
        cudaEventDestroy(p->ev_fork);
    }
    for (void* q : p->owned) cudaFree(q);
    delete p;
}

// ---- plan construction: slicq_plan_create runs the steps below in order.  Each step fills its part of the plan (scalars
// straight into the device tables) and of the host tables, or returns the error of the first check that fails.
namespace {

// the host copies of the arrays of SlicqDeviceTables, and the bucket of each bin
struct PlanTables {
    std::vector<int> bin_bucket;
    std::vector<float> tukey, wf, wi;
    std::vector<float2> post_tw, tw, wN;
    std::vector<double2> wP;
    std::vector<int> toff, ov, ovoff;
    std::vector<int4> ex;
    std::vector<int2> gaps;
    std::vector<SlicqMirrorEntry> mir;
    std::vector<SlicqMirrorBin> mir_bins;
};

// bin lengths and positions; bin j's coefficients start at bin_coff[j] of a packed [sum_M] row
int check_bins(const slicq_tables& t, slicq_plan& p) {
    p.bin_M.assign(t.bin_M, t.bin_M + p.J);
    p.bin_pos.assign(t.bin_pos, t.bin_pos + p.J);
    p.bin_coff.resize(p.J);
    int off = 0;
    for (int j = 0; j < p.J; ++j) {
        const int M = p.bin_M[j], pos = p.bin_pos[j];
        if (M < 4 || M % 4 != 0 || M > SLICQ_MAX_M || !find_fft_plan(M))
            return fail(SLICQ_E_UNSUPPORTED, "bin length M must be a multiple of 4 in [16, 292]");
        // the lowest bins of Bark / mel filterbanks with few bins or a low fmin can share a position
        if (pos % 2 != 0 || pos < 0 || pos > p.N2 || (j > 0 && pos < p.bin_pos[j - 1]))
            return fail(SLICQ_E_UNSUPPORTED, "bin positions must be even, non-decreasing and within [0, L/2]");
        p.bin_coff[j] = off;
        off += M;
    }
    p.dev.sum_M = off;
    // The reference also accumulates a mirrored copy of bins 1..J-2 at L - pos_j (nsigtf.py:63-80).  It reaches the kept
    // half spectrum [0, L/2] only from a bin that extends past Nyquist (unsupported) or below DC (handled by
    // mirror_fix_kernel, entries built by build_mirror_entries).
    for (int j = 1; j < p.J - 1; ++j)
        if (p.bin_pos[j] + p.bin_M[j] / 2 > p.N2)
            return fail(SLICQ_E_UNSUPPORTED, "a bin below Nyquist reaches beyond it: the mirrored-bin pass above Nyquist is not implemented");
    return SLICQ_OK;
}

// buckets = maximal runs of equal M (nsgtf.py:66-78), their units per CTA iteration, shared memory, cost and twiddles
int build_buckets(slicq_plan& p, PlanTables& h) {
    h.bin_bucket.resize(p.J);
    int tw_off = 0;
    for (int j = 0; j < p.J; ++j) {
        if (p.buckets.empty() || p.buckets.back().M != p.bin_M[j]) {
            const FftPlan* f = find_fft_plan(p.bin_M[j]);
            Bucket b;
            b.M = p.bin_M[j]; b.first_bin = j; b.n_bins = 0; b.tw_off = tw_off;
            b.kind = f->kind; b.A = f->A; b.B = f->B; b.smem_per_fft = fft_smem_per_transform(*f);
            b.gt = 1; b.cost = 0.0; b.gap_first = 0; b.gap_n = 0;
            tw_off += b.M;
            p.buckets.push_back(b);
        }
        p.buckets.back().n_bins++;
        h.bin_bucket[j] = (int)p.buckets.size() - 1;
    }
    if ((int)p.buckets.size() > SLICQ_MAX_BUCKETS) return fail(SLICQ_E_UNSUPPORTED, "too many buckets");
    p.dev.n_buckets = (int)p.buckets.size();
    // units per CTA iteration: fill the 256 threads of the hoisted pass, shared memory <= 48 KB
    p.bins_smem = 0;
    for (Bucket& b : p.buckets) {
        const FftPlan* f = find_fft_plan(b.M);
        int gt = kBinsThreads / (b.n_bins * fft_threads_per_transform(*f));
        if (gt < 1) gt = 1;
        while (gt > 1 && b.n_bins * gt * b.smem_per_fft > 48 * 1024) --gt;
        if (b.n_bins * fft_threads_per_transform(*f) > kBinsThreads)
            return fail(SLICQ_E_UNSUPPORTED, "bucket has too many bins for one CTA");
        b.gt = gt;
        // + SLICQ_SLOT_BYTES; single-thread transforms keep the bucket's windows behind the stage
        // two-pass and prime transforms keep the job's twiddles (M complex) and dual windows (F * M floats) there too
        const int sm = b.n_bins * gt * b.smem_per_fft + 4096 + (f->kind == 1 ? b.n_bins * b.M * 4 + b.n_bins * 12 + 32 : 0) + (f->kind == 3 ? b.n_bins * 12 + 16 : 0) +
                       (f->kind >= 2 ? b.M * 8 + b.n_bins * b.M * 4 + b.n_bins * 4 + 16 : 0);
        if (sm > p.bins_smem) p.bins_smem = sm;
        // work model: flops ~ M log2 M per transform plus a per-coefficient load/store term
        b.cost = (double)b.n_bins * f->cost;   // instructions per transform (fft_sizes.inc)
    }
    h.tw.resize(tw_off);
    for (const Bucket& b : p.buckets)
        for (int j = 0; j < b.M; ++j) {
            const double a = -2.0 * M_PI * (double)j / (double)b.M;
            h.tw[b.tw_off + j] = make_float2((float)cos(a), (float)sin(a));
        }
    return SLICQ_OK;
}

// the windows in centred order, the margins of the spectra below DC and above Nyquist, and the support of the slicing
// window
int build_windows(const slicq_tables& t, slicq_plan& p, PlanTables& h) {
    SlicqDeviceTables& d = p.dev;
    h.wf.resize(d.sum_M); h.wi.resize(d.sum_M);
    int pad_l = 0, pad_r = 0;
    for (int j = 0; j < p.J; ++j) {
        const int M = p.bin_M[j], o = p.bin_coff[j];
        const double sgn = ((p.bin_pos[j] / 2) % 2) ? -1.0 : 1.0;
        for (int mc = 0; mc < M; ++mc) {            // centred order m' = m~ + M/2
            const int m = (mc + M / 2) % M;         // reference order (peak at m = 0)
            h.wf[o + mc] = (float)((double)t.win_fwd[o + m] * sgn / (double)M);
            h.wi[o + mc] = (float)((double)t.win_inv[o + m] * sgn * (double)M / (double)p.L);   // 1/L of the slice IFFT folded in
        }
        pad_l = std::max(pad_l, M / 2 - p.bin_pos[j]);
        pad_r = std::max(pad_r, p.bin_pos[j] + M / 2 - 1 - p.N2);
    }
    pad_l = (pad_l + 1) & ~1;
    pad_r = (pad_r + 1) & ~1;
    if (pad_l > p.N2 / 2 || pad_r > p.N2 / 2) return fail(SLICQ_E_UNSUPPORTED, "bins reach too far beyond DC / Nyquist");
    d.pad_l = pad_l; d.pad_r = pad_r;
    h.tukey.assign(t.tukey, t.tukey + p.L);
    d.tw_lo = 0; d.tw_hi = p.L;
    while (d.tw_lo < p.L && h.tukey[d.tw_lo] == 0.f) ++d.tw_lo;
    while (d.tw_hi > d.tw_lo && h.tukey[d.tw_hi - 1] == 0.f) --d.tw_hi;
    return SLICQ_OK;
}

// synthesis intermediate T (see SlicqDeviceTables): two planes + overflow, and the overflow entries in rounds
int build_synthesis_layout(const slicq_tables& t, slicq_plan& p, PlanTables& h) {
    SlicqDeviceTables& d = p.dev;
    const int N2 = p.N2, J = p.J;
    d.pl_off = d.pad_l;                                                          // even
    d.pl_len = (d.pl_off + N2 + 2 + std::max(d.pad_r, 2) + 1) & ~1;              // positions -pl_off .. N2 + 1 + pad_r, even
    // Bin j writes positions [lo_j + ov_j, lo_j + M_j) of its plane.  Its leading ov_j positions, those that an earlier bin
    // of the plane already reaches (the furthest end of all of them, clamped to the bin), go to its overflow slot: every
    // plane position has at most one writer.  ov_j is even (positions and half lengths are), and may be all of M_j.
    h.toff.assign(J, 0); h.ov.assign(J, 0); h.ovoff.assign(J, 0);
    int n_ovf = 0;
    int plane_end[2] = {-2 * N2 - 2, -2 * N2 - 2};
    for (int j = 0; j < J; ++j) {
        const int lo = p.bin_pos[j] - p.bin_M[j] / 2;
        h.toff[j] = (j & 1) * d.pl_len + d.pl_off + lo;
        h.ov[j] = std::min(p.bin_M[j], std::max(0, plane_end[j & 1] - lo));
        plane_end[j & 1] = std::max(plane_end[j & 1], lo + p.bin_M[j]);
        h.ovoff[j] = 2 * d.pl_len + n_ovf;
        n_ovf += h.ov[j];
    }
    // two-pass / prime transforms divert only their first run of outputs (A, resp. R = B) to the overflow slot, through one
    // select; a plan with a longer overflow runs the synthesis variant that checks every output (bins_inv_ovr_kernel)
    p.ov_multi_run = false;
    for (int j = 0; j < J; ++j) {
        const Bucket& b = p.buckets[h.bin_bucket[j]];
        if ((b.kind == 2 && h.ov[j] > b.A) || (b.kind == 3 && h.ov[j] > b.B)) p.ov_multi_run = true;
    }
    p.t_stride = (2LL * d.pl_len + n_ovf + 1) & ~1LL;
    d.t_stride = (int)p.t_stride;
    // overflow entries {f, off0, off1 or -1, fold | round << 1}: position f also receives T[off0] (+ T[off1]).  The synthesis
    // drops the parts outside [0, N2]; the adjoint of the analysis folds them back conjugated (the analysis reads the
    // Hermitian mirror there), as separate entries after the direct ones: their targets may coincide with direct targets,
    // so the slice kernel adds them in a later pass.  The slots of one position, in bin order, pair up into entries; the
    // r-th entry of every position belongs to round r, so the targets of a round are distinct and the slice kernel adds
    // the rounds one after the other (a barrier in between, no atomics).  Entries are ordered by (fold, round, f).
    const bool fold = (t.flags & SLICQ_PLAN_ADJOINT_OF_ANALYSIS) != 0;
    std::vector<std::vector<int> > slots[2] = {std::vector<std::vector<int> >(N2 + 1), std::vector<std::vector<int> >(N2 + 1)};
    for (int j = 0; j < J; ++j)
        for (int m = 0; m < h.ov[j]; ++m) {
            int f = p.bin_pos[j] - p.bin_M[j] / 2 + m;
            const bool out = f < 0 || f > N2;
            if (out && !fold) continue;
            if (f < 0) f = -f;
            if (f > N2) f = 2 * N2 - f;
            slots[out][f].push_back(h.ovoff[j] + m);
        }
    d.ex_rounds = 0;
    for (int w = 0; w < 2; ++w) {
        size_t most = 0;
        for (const std::vector<int>& s : slots[w]) most = std::max(most, s.size());
        const int rounds = (int)((most + 1) / 2);
        d.ex_rounds = std::max(d.ex_rounds, rounds);
        for (int r = 0; r < rounds; ++r)
            for (int f = 0; f <= N2; ++f) {
                const std::vector<int>& s = slots[w][f];
                if ((int)s.size() > 2 * r) h.ex.push_back(int4{f, s[2 * r], (int)s.size() > 2 * r + 1 ? s[2 * r + 1] : -1, w | (r << 1)});
            }
    }
    // the tuned slice kernels (k_slice.cu) have no folded pass and add the entries in one round
    if (p.L == kTunedSliceLen && h.ex.size() > 0 && h.ex.back().w)
        return fail(SLICQ_E_UNSUPPORTED, "adjoint of the analysis: overflow below DC / above Nyquist is not implemented in "
                                         "the tuned slice kernels (slice length 18060)");
    if (p.L == kTunedSliceLen && d.ex_rounds > 1)
        return fail(SLICQ_E_UNSUPPORTED, "more than two overflow entries at one spectrum position are not implemented in "
                                         "the tuned slice kernels (slice length 18060)");
    d.n_ex = (int)h.ex.size();
    if (h.ex.empty()) h.ex.push_back(int4{0, 0, -1, 0});
    return SLICQ_OK;
}

// gaps: positions of a plane row (-pl_off .. pl_len - pl_off - 1, margins included: the adjoint-of-analysis mode folds
// them back) that none of its bins writes (a position a bin diverts to its overflow slot is written only if another bin
// of the plane writes it); owner = the bin covering the next written position (or the plane's last bin)
int build_gap_lists(slicq_plan& p, PlanTables& h) {
    const int pl_off = p.dev.pl_off, pl_len = p.dev.pl_len;
    std::vector<std::vector<int2> > per_bucket(p.buckets.size());
    for (int q = 0; q < 2; ++q) {
        std::vector<int> owner(pl_len, -1);    // covering bin or -1, index = pl_off + f
        std::vector<char> written(pl_len, 0);
        int last = -1;
        for (int j = q; j < p.J; j += 2) {
            const int lo = std::max(0, pl_off + p.bin_pos[j] - p.bin_M[j] / 2), hi = std::min(pl_len, pl_off + p.bin_pos[j] + p.bin_M[j] / 2);
            for (int f = lo; f < hi; ++f) owner[f] = j;
            for (int f = std::max(lo, pl_off + p.bin_pos[j] - p.bin_M[j] / 2 + h.ov[j]); f < hi; ++f) written[f] = 1;
            last = j;
        }
        if (last < 0) return fail(SLICQ_E_UNSUPPORTED, "a bin plane is empty");
        for (int f = 0; f < pl_len;) {
            if (written[f]) { ++f; continue; }
            int g = f;
            while (g < pl_len && !written[g]) ++g;
            const int next = g < pl_len ? owner[g] : last;
            per_bucket[h.bin_bucket[next]].push_back(int2{q * pl_len + f, g - f});
            f = g;
        }
    }
    for (size_t i = 0; i < p.buckets.size(); ++i) {
        p.buckets[i].gap_first = (int)h.gaps.size();
        p.buckets[i].gap_n = (int)per_bucket[i].size();
        h.gaps.insert(h.gaps.end(), per_bucket[i].begin(), per_bucket[i].end());
    }
    if (h.gaps.empty()) h.gaps.push_back(int2{0, 0});
    return SLICQ_OK;
}

// mirrored-bin entries (see mirror_fix_kernel): bin j >= 1 with pos_j < M_j / 2; reference-order index m in [pos_j, M_j/2)
// lands at spectrum position f = m - pos_j (< pad_l <= N2 / 2)
int build_mirror_entries(const slicq_tables& t, slicq_plan& p, PlanTables& h) {
    SlicqDeviceTables& d = p.dev;
    for (int j = 1; j < p.J - 1; ++j) {
        const int M = p.bin_M[j], pos = p.bin_pos[j], bi = h.bin_bucket[j];
        if (pos >= M / 2) continue;
        h.mir_bins.push_back(SlicqMirrorBin{bi, j - p.buckets[bi].first_bin, (int)h.mir.size(), M / 2 - pos});
        d.mir_nf = std::max(d.mir_nf, M / 2 - pos);
        d.mir_nc += M;
        for (int m = pos; m < M / 2; ++m) {
            SlicqMirrorEntry e;
            e.m_src = m + 1;
            const double gdm = (double)t.win_inv[p.bin_coff[j] + (M - m) % M];      // dual window of the mirrored bin at m
            const double sgn = (((pos / 2) + m) % 2) ? -1.0 : 1.0;                     // (-1)^(pos/2) (-1)^m
            e.weight = (float)(sgn * gdm * (double)M / (double)p.L);
            h.mir.push_back(e);
        }
    }
    // (the adjoint-of-analysis plan has no such pass: the analysis reads the exact Hermitian mirror; the adjoint-of-synthesis
    // plan runs the pass's transpose, mirror_adj_kernel, after its analysis bins)
    d.n_mir = (t.flags & SLICQ_PLAN_ADJOINT_OF_ANALYSIS) ? 0 : (int)h.mir.size();
    if (h.mir.empty()) h.mir.push_back(SlicqMirrorEntry{0, 0.f});
    d.n_mir_bins = (int)h.mir_bins.size();
    if (h.mir_bins.empty()) h.mir_bins.push_back(SlicqMirrorBin{0, 0, 0, 0});
    return SLICQ_OK;
}

// twiddles of the slice transforms: exp(-2 pi i k / L) of the real-FFT post-processing, and for the generic slice kernels
// the prime factors of N2 (largest first) and exp(-2 pi i k / N2)
int build_slice_tables(slicq_plan& p, PlanTables& h) {
    const int N2 = p.N2;
    h.post_tw.resize(N2 / 2 + 1);
    for (int k = 0; k <= N2 / 2; ++k) {
        const double a = -2.0 * M_PI * (double)k / (double)p.L;
        h.post_tw[k] = make_float2((float)cos(a), (float)sin(a));
    }
    std::vector<int> fac;
    { int n = N2; for (int d = 2; d * d <= n; ++d) while (n % d == 0) { fac.push_back(d); n /= d; } if (n > 1) fac.push_back(n); }
    std::sort(fac.begin(), fac.end(), [](int x, int y) { return x > y; });
    if (fac.size() > 20) return fail(SLICQ_E_UNSUPPORTED, "too many prime factors in the slice length");
    p.dev.n_fac = (int)fac.size();
    for (size_t i = 0; i < fac.size(); ++i) p.dev.fac[i] = fac[i];
    h.wP.resize(fac[0] > 32 ? fac[0] : 1);
    for (size_t kk = 0; kk < h.wP.size(); ++kk) {
        const double ang = -2.0 * M_PI * (double)kk / (double)h.wP.size();
        h.wP[kk].x = cos(ang); h.wP[kk].y = sin(ang);
    }
    h.wN.resize(N2);
    for (int kk = 0; kk < N2; ++kk) {
        const double ang = -2.0 * M_PI * (double)kk / (double)N2;
        h.wN[kk] = make_float2((float)cos(ang), (float)sin(ang));
    }
    return SLICQ_OK;
}

int upload_tables(slicq_plan& p, const PlanTables& h) {
    SlicqDeviceTables& d = p.dev;
    int rc = 0;
    rc |= upload(h.tukey, &d.tukey, p.owned);
    rc |= upload(h.wf, &d.wf, p.owned);
    rc |= upload(h.wi, &d.wi, p.owned);
    rc |= upload(p.bin_pos, &d.bin_pos, p.owned);
    rc |= upload(p.bin_M, &d.bin_M, p.owned);
    rc |= upload(p.bin_coff, &d.bin_coff, p.owned);
    rc |= upload(h.post_tw, &d.post_tw, p.owned);
    rc |= upload(h.tw, &d.tw, p.owned);
    rc |= upload(h.toff, &d.bin_toff, p.owned);
    rc |= upload(h.ov, &d.bin_ov, p.owned);
    rc |= upload(h.ovoff, &d.bin_ovoff, p.owned);
    rc |= upload(h.ex, &d.ex, p.owned);
    rc |= upload(h.gaps, &d.gaps, p.owned);
    rc |= upload(h.mir, &d.mir, p.owned);
    rc |= upload(h.mir_bins, &d.mir_bins, p.owned);
    rc |= upload(h.wN, &d.wN, p.owned);
    rc |= upload(h.wP, &d.wP, p.owned);
    return rc ? fail(SLICQ_E_CUDA, "device table upload failed") : SLICQ_OK;
}

}  // namespace

extern "C" int slicq_plan_create(const slicq_tables* t, slicq_plan** out) {
    if (!t || !out) return fail(SLICQ_E_INVALID, "null argument");
    *out = nullptr;
    const int L = t->sl_len, J = t->n_bins;
    if (L <= 0 || L % 4 != 0) return fail(SLICQ_E_INVALID, "sl_len must be a positive multiple of 4");
    if (J < 2 || !t->bin_M || !t->bin_pos || !t->win_fwd || !t->win_inv || !t->tukey)
        return fail(SLICQ_E_INVALID, "missing tables");
    if (slicq_slice_smem_bytes(L) < 0) {
        char buf[160];
        snprintf(buf, sizeof buf, "slice length %d does not fit the slice kernels' shared memory (two buffers of sl_len/2 complex numbers)", L);
        return fail(SLICQ_E_UNSUPPORTED, buf);
    }
    std::unique_ptr<slicq_plan, decltype(&slicq_plan_destroy)> p(new slicq_plan(), slicq_plan_destroy);
    p->L = L; p->N2 = L / 2; p->hop = L / 2; p->J = J;
    p->side_ready = false;
    SlicqDeviceTables& d = p->dev;
    memset(&d, 0, sizeof d);
    d.L = L; d.N2 = p->N2; d.hop = p->hop; d.n_bins = J;
    d.adjoint = t->flags & (SLICQ_PLAN_ADJOINT_OF_SYNTHESIS | SLICQ_PLAN_ADJOINT_OF_ANALYSIS);
    d.spec_scale = (d.adjoint & 1) ? (float)(2.0 / L) : 1.f;
    d.ends_scale = (d.adjoint & 1) ? (float)(1.0 / L) : 1.f;
    PlanTables h;
    if (int rc = check_bins(*t, *p)) return rc;
    if (int rc = build_buckets(*p, h)) return rc;
    if (int rc = build_windows(*t, *p, h)) return rc;
    if (int rc = build_synthesis_layout(*t, *p, h)) return rc;
    if (int rc = build_gap_lists(*p, h)) return rc;
    if (int rc = build_mirror_entries(*t, *p, h)) return rc;
    if (int rc = build_slice_tables(*p, h)) return rc;
    if (int rc = upload_tables(*p, h)) return rc;
    p->spec_stride_fwd = (d.pad_l + p->N2 + 1 + d.pad_r + 1) & ~1LL;  // even: 16-byte aligned rows
    const char* env = getenv("SLICQ_CHUNK_MB");
    long long mb = env ? atoll(env) : 2048;
    if (mb < 1) mb = 1;
    p->chunk_bytes = mb << 20;
    const char* envs = getenv("SLICQ_SPLIT_UNITS");
    p->split_units = envs ? atoll(envs) : 1184;
    *out = p.release();
    return SLICQ_OK;
}

#ifdef SLICQ_EMU
// emulation build only (tests/emu): the synthesis layout the plan derived, for tests of the plan rules.  The emulated
// device tables are host memory.
extern "C" int slicq_emu_plan_layout(const slicq_plan* p, const int** ov, const int4** ex, int* n_ex, int* ex_rounds,
                                     int* ov_multi_run) {
    if (!p) return SLICQ_E_INVALID;
    *ov = p->dev.bin_ov; *ex = p->dev.ex; *n_ex = p->dev.n_ex; *ex_rounds = p->dev.ex_rounds;
    *ov_multi_run = p->ov_multi_run ? 1 : 0;
    return SLICQ_OK;
}
#endif

extern "C" int slicq_plan_n_buckets(const slicq_plan* p) { return p ? (int)p->buckets.size() : SLICQ_E_INVALID; }

extern "C" int slicq_plan_bucket_info(const slicq_plan* p, int b, int32_t* first_bin, int32_t* n_bins, int32_t* M) {
    if (!p || b < 0 || b >= (int)p->buckets.size()) return fail(SLICQ_E_INVALID, "bad bucket index");
    if (first_bin) *first_bin = p->buckets[b].first_bin;
    if (n_bins) *n_bins = p->buckets[b].n_bins;
    if (M) *M = p->buckets[b].M;
    return SLICQ_OK;
}

extern "C" int64_t slicq_plan_num_slices(const slicq_plan* p, int64_t T) {
    if (!p || T < 0) return SLICQ_E_INVALID;
    const int64_t hh = p->L / 4;
    const int64_t nblk = (T + hh - 1) / hh;  // quarter-hop blocks (slicing.py:34-42)
    return (nblk + 1) / 2 + 1;               // slicing.py:49,61-72
}

namespace {
long long bytes_per_unit(const slicq_plan* p, int inverse) {
    if (!inverse) return p->spec_stride_fwd * 8;
    return p->t_stride * 8;
}
long long chunk_units(const slicq_plan* p, int inverse) {
    long long c = p->chunk_bytes / bytes_per_unit(p, inverse);
    if (c >= 296) c -= c % 296;   // whole waves of the slice kernels (148 SMs x 2 CTAs)
    return c < 1 ? 1 : c;
}
bool use_split(const slicq_plan* p, int64_t n_rows, int64_t n_slices) {
    return p->split_units > 0 && n_rows >= 2 && n_rows * n_slices >= p->split_units;
}
// a split call deals its rows to two groups of (almost) equal size; group h = rows [part_row0(h), part_row0(h + 1))
int64_t part_row0(int64_t n_rows, int h) { return n_rows * h / 2; }
size_t half_scratch(const slicq_plan* p, int64_t rows, int64_t n_slices, int inverse) {
    long long units = rows * n_slices;
    const long long c = chunk_units(p, inverse);
    if (units > c) units = c;
    return ((size_t)(units * bytes_per_unit(p, inverse)) + 511) & ~(size_t)255;
}
int ensure_side_streams(const slicq_plan* p) {
    if (p->side_ready) return 0;
    if (cudaEventCreateWithFlags(&p->ev_fork, cudaEventDisableTiming)) return -1;
    for (int h = 0; h < 2; ++h)
        if (cudaStreamCreateWithFlags(&p->side[h], cudaStreamNonBlocking) || cudaEventCreateWithFlags(&p->ev_join[h], cudaEventDisableTiming))
            return -1;
    p->side_ready = true;
    return 0;
}
}  // namespace

extern "C" size_t slicq_scratch_bytes(const slicq_plan* p, int64_t n_rows, int64_t n_slices, int inverse) {
    if (!p || n_rows <= 0 || n_slices <= 0) return 0;
    if (use_split(p, n_rows, n_slices)) {
        size_t total = 256;
        for (int h = 0; h < 2; ++h)
            total += half_scratch(p, part_row0(n_rows, h + 1) - part_row0(n_rows, h), n_slices, inverse);
        return total;
    }
    return half_scratch(p, n_rows, n_slices, inverse) + 256;
}

namespace {
// One call of the C ABI, as the seven slicq_forward* / slicq_inverse* entries describe it to run_call.
struct Call {
    bool inverse;
    const float* x;                    // signal rows: the analysed signal, or the synthesis output (that one may be null if
                                       // n_samples == 0)
    int64_t n_rows;                    // output rows (analysis: rows of x)
    int64_t x_row_stride, n_samples, t0, k0, n_slices;
    const slicq_bucket_view* coefs;    // complex64: the analysis output or the synthesis input, or the mixture
    const slicq_bucket_view* aux;      // fp32, optional: |c| or the mask gradient (analysis), the masks (synthesis)
    int64_t mix_rows;                  // 0: coefs follow the output rows; > 0: coefs hold a mixture of mix_rows rows, read
                                       // as row r % mix_rows by output row r and shared by all row groups
    float* halo_out;                   // synthesis: [rows][hop] or null
};

SlicqBinsKernel bins_kernel(const slicq_plan* p, const Call& c) {
    if (c.inverse) return p->ov_multi_run ? bins_inv_ovr : bins_inv;
    return c.mix_rows ? bins_fwd_mask_grad : bins_fwd;
}

// the parameters every chunk of a row group shares; a chunk's intermediate spectra start at the first 256-byte boundary
// of the scratch
void init_params(const slicq_plan* p, const Call& c, void* scratch, SlicqSliceParams& sp, SlicqBinsParams& bp) {
    float2* spec = reinterpret_cast<float2*>((reinterpret_cast<uintptr_t>(scratch) + 255) & ~(uintptr_t)255);
    const long long spec_stride = c.inverse ? p->t_stride : p->spec_stride_fwd;
    memset(&sp, 0, sizeof sp);
    sp.t = p->dev; sp.x = const_cast<float*>(c.x); sp.x_row_stride = c.x_row_stride; sp.T = c.n_samples; sp.t0 = c.t0;
    sp.k0 = c.k0; sp.spec = spec; sp.spec_stride = spec_stride; sp.S = (int)c.n_slices; sp.halo_out = c.halo_out;
    bp.t = p->dev; bp.spec = spec; bp.spec_stride = spec_stride; bp.S = (int)c.n_slices; bp.k0 = (int)c.k0;
    bp.x_rows = (int)c.mix_rows; bp.mask_grad = bins_kernel(p, c) == bins_fwd_mask_grad;
}

// the caller's views and the job split of one bins launch over units [rs0, rs0 + n_rs) of the row group
int fill_bins_params(const slicq_plan* p, const Call& c, SlicqBinsParams& bp, int n_rs, int rs0) {
    int jobs = 0;
    bp.n_rs = n_rs; bp.rs0 = rs0;
    bp.n_buckets = (int)p->buckets.size();
    double total = 0.0;
    for (const Bucket& b : p->buckets) total += b.cost;
    // jobs per bins launch: 148 SMs x 3 resident CTAs x 10 waves for large launches (short jobs even out the tail;
    // swept 666 ... 8880 at batch 8 in both rounds), 1184 for small ones (a job keeps enough iterations to amortise its
    // set-up)
    const int target = std::min(4440, std::max(1184, 4 * n_rs));
    for (size_t i = 0; i < p->buckets.size(); ++i) {
        const Bucket& b = p->buckets[i];
        SlicqBucketArg& a = bp.b[i];
        a.ptr = reinterpret_cast<float2*>(c.coefs[i].ptr);
        a.s_row = c.coefs[i].s_row; a.s_bin = c.coefs[i].s_bin; a.s_slice = c.coefs[i].s_slice;
        a.M = b.M; a.first_bin = b.first_bin; a.n_bins = b.n_bins; a.gt = b.gt; a.tw_off = b.tw_off;
        a.gap_first = b.gap_first; a.gap_n = b.gap_n;
        a.mptr = c.aux && c.inverse ? reinterpret_cast<const float*>(c.aux[i].ptr) : nullptr;
        a.nptr = c.aux && !c.inverse ? reinterpret_cast<float*>(c.aux[i].ptr) : nullptr;
        a.ms_row = c.aux ? c.aux[i].s_row : 0; a.ms_bin = c.aux ? c.aux[i].s_bin : 0; a.ms_slice = c.aux ? c.aux[i].s_slice : 0;
        const int groups = (n_rs + b.gt - 1) / b.gt;                 // iterations available in this chunk
        int nj = (int)(target * b.cost / total + 0.5);
        if (nj > groups) nj = groups;
        if (nj < 1) nj = 1;
        const int gpj = (groups + nj - 1) / nj;                      // iterations per job
        a.units_per_job = gpj * b.gt;
        a.n_jobs = (n_rs + a.units_per_job - 1) / a.units_per_job;
        a.job_start = jobs;
        jobs += a.n_jobs;
    }
    return jobs;
}

int launch_result(int rc) {
    if (!rc) return SLICQ_OK;
    char buf[128];
    snprintf(buf, sizeof buf, "kernel launch failed: %s", rc > 0 ? cudaGetErrorString((cudaError_t)rc) : "unsupported");
    return fail(SLICQ_E_CUDA, buf);
}

// analysis of one row group, per chunk of units: slice_fft_fwd -> bins_fwd [-> mirror_adj]
int forward_one(const slicq_plan* p, const Call& c, void* scratch, cudaStream_t s) {
    const long long units = c.n_rows * c.n_slices, cu = chunk_units(p, 0);
    SlicqSliceParams sp;
    SlicqBinsParams* bp = new SlicqBinsParams();
    init_params(p, c, scratch, sp, *bp);
    int rc = 0;
    for (long long u0 = 0; u0 < units && rc == 0; u0 += cu) {
        const int n = (int)((units - u0 < cu) ? (units - u0) : cu);
        sp.n_rs = n; sp.rs0 = (int)u0;
        { ProfScope ps(K_SLICE_FWD, s); rc = slicq_launch_slice_fwd(&sp, s); }
        ++g_launches;
        if (rc) break;
        const int jobs = fill_bins_params(p, c, *bp, n, (int)u0);
        { ProfScope ps(K_BINS_FWD, s); rc = slicq_launch_bins(bp, jobs, p->bins_smem, bins_kernel(p, c), s); }
        ++g_launches;
        if (rc) break;
        if ((p->dev.adjoint & 1) && p->dev.n_mir > 0) {      // transpose of the mirrored-bin pass, reads this chunk's H
            rc = slicq_launch_mirror_adj(bp, s);
            ++g_launches;
        }
    }
    delete bp;
    return launch_result(rc);
}

// synthesis of one row group, per chunk of units: bins_inv [-> mirror_fix] -> slice_fft_inv (even slices, then odd slices)
int inverse_one(const slicq_plan* p, const Call& c, void* scratch, cudaStream_t s) {
    const long long units = c.n_rows * c.n_slices, cu = chunk_units(p, 1);
    SlicqSliceParams sp;
    SlicqBinsParams* bp = new SlicqBinsParams();
    init_params(p, c, scratch, sp, *bp);
    int rc = 0;
    for (long long u0 = 0; u0 < units && rc == 0;) {
        long long n = (units - u0 < cu) ? (units - u0) : cu;
        // a chunk must not start on an even slice k > 0: the odd slice before it accumulates into
        // hops that the even slice has to have stored first (see slice_fft_inv_kernel)
        while (n > 1 && u0 + n < units && ((u0 + n) % c.n_slices) != 0 && (((u0 + n) % c.n_slices) & 1) == 0) --n;
        const int jobs = fill_bins_params(p, c, *bp, (int)n, (int)u0);
        { ProfScope ps(K_BINS_INV, s); rc = slicq_launch_bins(bp, jobs, p->bins_smem, bins_kernel(p, c), s); }
        ++g_launches;
        if (rc) break;
        if (p->dev.n_mir > 0) {          // mirrored-bin pass of configurations whose first bins reach below DC
            rc = slicq_launch_mirror_fix(bp, s);
            ++g_launches;
            if (rc) break;
        }
        sp.n_rs = (int)n; sp.rs0 = (int)u0;
        {
            ProfScope ps(K_SLICE_INV, s);
            sp.parity = 0; rc = slicq_launch_slice_inv(&sp, s);
            if (!rc) { sp.parity = 1; rc = slicq_launch_slice_inv(&sp, s); }
        }
        g_launches += 2;
        u0 += n;
    }
    delete bp;
    return launch_result(rc);
}

int run_rows(const slicq_plan* p, const Call& c, void* scratch, cudaStream_t s) {
    return c.inverse ? inverse_one(p, c, scratch, s) : forward_one(p, c, scratch, s);
}

// checks a call, and runs it whole or, when it is large enough, as two row groups on the plan's side streams
int run_call(const slicq_plan* p, const Call& c, void* scratch, size_t scratch_bytes, void* stream) {
    // the synthesis output may be null when length == 0 (a shard that owns no output samples still produces its halo)
    if (!p || (!c.x && (!c.inverse || c.n_samples > 0)) || !c.coefs) return fail(SLICQ_E_INVALID, "null argument");
    if (c.n_rows <= 0 || c.n_slices <= 0 || c.n_samples < 0) return fail(SLICQ_E_INVALID, "bad shape");
    if (c.n_rows * c.n_slices > 0x7fffffffLL) return fail(SLICQ_E_INVALID, "too many (row,slice) units");
    if (scratch_bytes < slicq_scratch_bytes(p, c.n_rows, c.n_slices, c.inverse) || !scratch)
        return fail(SLICQ_E_SCRATCH, "scratch buffer too small (see slicq_scratch_bytes)");
    if (reinterpret_cast<uintptr_t>(scratch) & 15) return fail(SLICQ_E_SCRATCH, "scratch buffer must be 16-byte aligned");
    for (size_t i = 0; i < p->buckets.size(); ++i)
        if (!c.coefs[i].ptr || (c.aux && !c.aux[i].ptr)) return fail(SLICQ_E_INVALID, "null bucket pointer");
    cudaStream_t s0 = reinterpret_cast<cudaStream_t>(stream);
    // output row r reads mixture row r % mix_rows, so a row group must start on a multiple of mix_rows
    if (!use_split(p, c.n_rows, c.n_slices) || (c.mix_rows && part_row0(c.n_rows, 1) % c.mix_rows != 0))
        return run_rows(p, c, scratch, s0);
    std::lock_guard<std::mutex> lock(p->split_mutex);
    if (ensure_side_streams(p)) return fail(SLICQ_E_CUDA, "cannot create internal streams");
    unsigned char* base = reinterpret_cast<unsigned char*>(scratch);
    slicq_bucket_view coefs[SLICQ_MAX_BUCKETS], aux[SLICQ_MAX_BUCKETS];
    cudaEventRecord(p->ev_fork, s0);
    int rc = 0;
    for (int h = 0; h < 2 && rc == 0; ++h) {
        // row group h: the signal, the fp32 views and the halo move by r0 rows, the coefficients too unless the mixture
        // is shared
        const int64_t r0 = part_row0(c.n_rows, h), rows = part_row0(c.n_rows, h + 1) - r0;
        Call g = c;
        g.n_rows = rows;
        g.x = c.x + r0 * c.x_row_stride;
        g.halo_out = c.halo_out ? c.halo_out + r0 * p->hop : nullptr;
        for (size_t i = 0; i < p->buckets.size(); ++i) {
            coefs[i] = c.coefs[i];
            if (!c.mix_rows) coefs[i].ptr = reinterpret_cast<float2*>(c.coefs[i].ptr) + r0 * c.coefs[i].s_row;
            if (c.aux) { aux[i] = c.aux[i]; aux[i].ptr = reinterpret_cast<float*>(c.aux[i].ptr) + r0 * c.aux[i].s_row; }
        }
        g.coefs = coefs;
        g.aux = c.aux ? aux : nullptr;
        cudaStreamWaitEvent(p->side[h], p->ev_fork, 0);
        rc = run_rows(p, g, base, p->side[h]);
        base += half_scratch(p, rows, c.n_slices, c.inverse);
        cudaEventRecord(p->ev_join[h], p->side[h]);
        cudaStreamWaitEvent(s0, p->ev_join[h], 0);
    }
    return rc;
}

// canonical packed layout: bucket b = contiguous [n_rows][F_b][S][M_b] elements of `elem` bytes, buckets in order
std::vector<slicq_bucket_view> packed_views(const slicq_plan* p, void* base_, int64_t n_rows, int64_t n_slices, size_t elem) {
    std::vector<slicq_bucket_view> v(p->buckets.size());
    unsigned char* base = reinterpret_cast<unsigned char*>(base_);
    for (size_t i = 0; i < p->buckets.size(); ++i) {
        const Bucket& b = p->buckets[i];
        v[i].ptr = base;
        v[i].s_slice = b.M;
        v[i].s_bin = (int64_t)n_slices * b.M;
        v[i].s_row = (int64_t)b.n_bins * n_slices * b.M;
        base += (size_t)n_rows * b.n_bins * n_slices * b.M * elem;
    }
    return v;
}
}  // namespace

extern "C" int slicq_forward(const slicq_plan* p, const float* x, int64_t n_rows, int64_t x_row_stride,
                             int64_t n_samples, int64_t t0, int64_t k0, int64_t n_slices,
                             const slicq_bucket_view* buckets, void* scratch, size_t scratch_bytes, void* stream) {
    const Call c = {false, x, n_rows, x_row_stride, n_samples, t0, k0, n_slices, buckets, nullptr, 0, nullptr};
    return run_call(p, c, scratch, scratch_bytes, stream);
}

extern "C" int slicq_forward_norm(const slicq_plan* p, const float* x, int64_t n_rows, int64_t x_row_stride,
                                  int64_t n_samples, int64_t t0, int64_t k0, int64_t n_slices,
                                  const slicq_bucket_view* buckets, const slicq_bucket_view* norms, void* scratch,
                                  size_t scratch_bytes, void* stream) {
    if (!norms) return fail(SLICQ_E_INVALID, "norms missing");
    const Call c = {false, x, n_rows, x_row_stride, n_samples, t0, k0, n_slices, buckets, norms, 0, nullptr};
    return run_call(p, c, scratch, scratch_bytes, stream);
}

// Canonical packed layout: all buckets in one allocation, bucket b = contiguous [n_rows][F_b][S][M_b].
extern "C" int slicq_forward_packed(const slicq_plan* p, const float* x, int64_t n_rows, int64_t x_row_stride,
                                    int64_t n_samples, int64_t t0, int64_t k0, int64_t n_slices, void* coefs,
                                    void* scratch, size_t scratch_bytes, void* stream) {
    if (!p || !coefs) return fail(SLICQ_E_INVALID, "null argument");
    std::vector<slicq_bucket_view> v = packed_views(p, coefs, n_rows, n_slices, 8);
    const Call c = {false, x, n_rows, x_row_stride, n_samples, t0, k0, n_slices, v.data(), nullptr, 0, nullptr};
    return run_call(p, c, scratch, scratch_bytes, stream);
}

extern "C" int slicq_forward_packed_norm(const slicq_plan* p, const float* x, int64_t n_rows, int64_t x_row_stride,
                                         int64_t n_samples, int64_t t0, int64_t k0, int64_t n_slices, void* coefs,
                                         void* norms, void* scratch, size_t scratch_bytes, void* stream) {
    if (!p || !coefs || !norms) return fail(SLICQ_E_INVALID, "null argument");
    std::vector<slicq_bucket_view> v = packed_views(p, coefs, n_rows, n_slices, 8);
    std::vector<slicq_bucket_view> nv = packed_views(p, norms, n_rows, n_slices, 4);
    const Call c = {false, x, n_rows, x_row_stride, n_samples, t0, k0, n_slices, v.data(), nv.data(), 0, nullptr};
    return run_call(p, c, scratch, scratch_bytes, stream);
}

// the analysis of the adjoint-of-synthesis plan with the mask-gradient epilogue: `mix` holds the mixture (n_rows rows,
// read only) and `grad_masks` receive the mask gradient of the n_targets * n_rows rows of g
extern "C" int slicq_forward_mask_grad(const slicq_plan* p, const float* g, int64_t n_targets, int64_t n_rows,
                                       int64_t g_row_stride, int64_t n_samples, int64_t t0, int64_t k0, int64_t n_slices,
                                       const slicq_bucket_view* mix, const slicq_bucket_view* grad_masks,
                                       void* scratch, size_t scratch_bytes, void* stream) {
    if (!p || !grad_masks || n_targets <= 0 || n_rows <= 0) return fail(SLICQ_E_INVALID, "null argument or bad shape");
    if (!(p->dev.adjoint & SLICQ_PLAN_ADJOINT_OF_SYNTHESIS))
        return fail(SLICQ_E_INVALID, "the mask gradient needs a plan created with SLICQ_PLAN_ADJOINT_OF_SYNTHESIS");
    const Call c = {false, g, n_targets * n_rows, g_row_stride, n_samples, t0, k0, n_slices, mix, grad_masks, n_rows, nullptr};
    return run_call(p, c, scratch, scratch_bytes, stream);
}

extern "C" int slicq_inverse(const slicq_plan* p, const slicq_bucket_view* buckets, int64_t n_rows,
                             int64_t n_slices, int64_t k0, float* y, int64_t y_row_stride, int64_t length,
                             int64_t t0, float* halo_out, void* scratch, size_t scratch_bytes, void* stream) {
    const Call c = {true, y, n_rows, y_row_stride, length, t0, k0, n_slices, buckets, nullptr, 0, halo_out};
    return run_call(p, c, scratch, scratch_bytes, stream);
}

// the synthesis of n_targets * n_rows output rows from the mixture `mix` (n_rows rows) times the per-output-row fp32 masks
extern "C" int slicq_inverse_masked(const slicq_plan* p, const slicq_bucket_view* mix, const slicq_bucket_view* masks,
                                    int64_t n_targets, int64_t n_rows, int64_t n_slices, int64_t k0, float* y,
                                    int64_t y_row_stride, int64_t length, int64_t t0, float* halo_out, void* scratch,
                                    size_t scratch_bytes, void* stream) {
    if (!masks || n_targets <= 0) return fail(SLICQ_E_INVALID, "masks / n_targets missing");
    if (p) for (size_t i = 0; i < p->buckets.size(); ++i)
        if (!masks[i].ptr) return fail(SLICQ_E_INVALID, "null mask pointer");
    const Call c = {true, y, n_targets * n_rows, y_row_stride, length, t0, k0, n_slices, mix, masks, n_rows, halo_out};
    return run_call(p, c, scratch, scratch_bytes, stream);
}
