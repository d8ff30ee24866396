// step_inst.cu - one translation unit per collocation size: compiled once for every M in 2..9 with
// -DSDCGYM_M=<M> (sdc_gym_b200/build.py) so the eight heavy instantiation sets build in parallel.
// Exposes sdcgym_launch_reset_m<M> / sdcgym_launch_step_m<M>, dispatched from sdcgym_abi.cu.
#include <atomic>
#include <cstdlib>
#include <type_traits>

#include "step_params.cuh"
#include "team_kernels.cuh"
#include "fast_kernels.cuh"
#include "stream_kernels.cuh"

#ifndef SDCGYM_M
#error "compile with -DSDCGYM_M=<2..9>"
#endif

#ifndef SDCGYM_STREAM_MINB
#define SDCGYM_STREAM_MINB 2  // blocks (of 256 threads) per SM of the streaming sdc-v1 kernel
#endif

#define SDCGYM_CAT_(a, b) a##b
#define SDCGYM_CAT(a, b) SDCGYM_CAT_(a, b)

namespace sdcgym {

constexpr int kM = SDCGYM_M;
constexpr int kHoldDiag = HoldPolicy<kM>::diag;
constexpr int kHoldDense = HoldPolicy<kM>::dense;


// opt-in to > 48 KB of dynamic shared memory: a per-DEVICE function attribute, remembered per (instantiation, device)
template <typename K>
static cudaError_t opt_in_smem(K kernel, size_t smem, std::atomic<uint64_t>& configured) {
    if (smem <= 48 * 1024) return cudaSuccess;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    const uint64_t bit = (dev >= 0 && dev < 64) ? (uint64_t(1) << dev) : 0;
    if (!(configured.load(std::memory_order_relaxed) & bit)) {
        e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        configured.fetch_or(bit, std::memory_order_relaxed);
    }
    return cudaSuccess;
}


// Hand-over rules of the phased dense solve (step_one PHASE), one per pass but the last (which runs every env to its
// end): a warp of pass k hands its stragglers over once they all have done stop[k] sweeps and fewer than lanes[k] of
// its lanes are still iterating.  Defaults measured on B200 against the single launch (profiles/README.md).
// Experiments: SDCGYM_PHASE_STOPS="a,b,..." (ascending sweep counts; alone: hand over at exactly these counts whatever
// the occupancy), SDCGYM_PHASE_LANES="a,b,..." (occupancy thresholds; alone: from the first sweep on).  An empty
// SDCGYM_PHASE_STOPS or SDCGYM_PHASE_LANES switches the phased solve off.  At most 6 hand-overs.
#ifndef SDCGYM_INVERSE_MINB
#define SDCGYM_INVERSE_MINB 4  // blocks of 128 threads per SM of inverse_kernel at M = 4, 5: 128 registers (5 blocks = 96
                               // registers spill 300 bytes at M = 5: 2.65 instead of 2.47 ms per 2^22-env strictly_lower_tri step)
#endif
struct PhasePlan {
    // first pass as two launches (inverse_kernel, then the first sweeps with the inverse reloaded): measured faster than
    // the fused first pass wherever the phased solve pays at all (2^22 envs, strictly_lower_tri, M = 3 ... 7: 0.87 /
    // 1.36 / 2.47 / 3.70 / 5.85 ms against 0.97 / 1.49 / 2.72 / 4.10 / 8.44 ms); SDCGYM_PHASE_SPLIT=0: fused first pass
    bool split = getenv("SDCGYM_PHASE_SPLIT") ? atoi(getenv("SDCGYM_PHASE_SPLIT")) != 0 : true;
    // one hand-over: every further pass ends with a tail of a few warps that run up to 45 dependent sweeps (>= 60 us);
    // 2^22 envs, M = 3 / 5 / 7: strictly_lower_tri 1.41 / 1.54 / 1.51 x, lower_tri 0.92 / 0.95 / 0.97 x the single launch
    int n = 1;
    int stop[6] = {5, 0, 0, 0, 0, 0};
    int lanes[6] = {8, 0, 0, 0, 0, 0};
    static int parse(const char* e, int* out, bool ascending) {
        int n = 0, prev = 0;
        while (*e && n < 6) {
            char* end = nullptr;
            const long v = strtol(e, &end, 10);
            if (end == e) break;
            if (v > 0 && v < (1 << 20) && (!ascending || v > prev)) out[n++] = prev = (int)v;
            e = (*end == ',') ? end + 1 : end;
        }
        return n;
    }
    PhasePlan() {
        const char* es = getenv("SDCGYM_PHASE_STOPS");
        const char* el = getenv("SDCGYM_PHASE_LANES");
        if (!es && !el) return;
        int st[6] = {0, 0, 0, 0, 0, 0}, ln[6] = {0, 0, 0, 0, 0, 0};
        const int ns = es ? parse(es, st, true) : 0, nl = el ? parse(el, ln, false) : 0;
        n = es ? (el ? (ns < nl ? ns : nl) : ns) : nl;
        for (int k = 0; k < 6; k++) {
            stop[k] = (k < n && es) ? st[k] : 0;    // no sweep count given: from the first sweep on
            lanes[k] = (k < n) ? (el ? ln[k] : 33) : 0;  // no threshold given: whatever the occupancy
        }
    }
};

// sdc-v0, dense Q_delta, one env per thread: inverse + sweeps for every env until its warp hands over, then one pass
// per further hand-over rule over the compacted list of the envs that are still iterating
template <int V>
static cudaError_t launch_phased_dense(const StepParams<kM>& p0, const PhasePlan& plan, cudaStream_t s) {
    constexpr int hold = kHoldDense, minb = HoldPolicy<kM>::dense_minb, block = HoldPolicy<kM>::dense_block;
    constexpr size_t smem = step_kernel_smem_bytes<kM, hold, block>();
    auto first = step_phase_kernel<kM, V, hold, minb, block, 1>;
    auto later = step_phase_kernel<kM, V, hold, minb, block, 2>;
    static std::atomic<uint64_t> conf1{0}, conf2{0};
    cudaError_t e = opt_in_smem(first, smem, conf1);
    if (e != cudaSuccess) return e;
    e = opt_in_smem(later, smem, conf2);
    if (e != cudaSuccess) return e;
    int32_t* const lists = p0.cont_list;
    int32_t* const counts = p0.cont_count;
    e = cudaMemsetAsync(counts, 0, sizeof(int32_t) * SDCGYM_PHASE_COUNTERS, s);
    if (e != cudaSuccess) return e;
    StepParams<kM> p = p0;
    p.it_stop = plan.stop[0];
    p.min_lanes = plan.lanes[0];
    p.cont_list = lists;
    p.cont_count = counts;
    const unsigned blocks = (unsigned)((p.N + block - 1) / block);
    if (plan.split) {
        // first pass in two launches: every inverse into the work planes (few registers, many warps), then the
        // first sweeps with the inverse reloaded
        constexpr int iminb = (kM <= 3) ? 8 : ((kM <= 5) ? SDCGYM_INVERSE_MINB : 2);
        inverse_kernel<kM, V, iminb><<<(unsigned)((p.N + kBlock - 1) / kBlock), kBlock, 0, s>>>(p);
        e = cudaGetLastError();
        if (e != cudaSuccess) return e;
        auto sweeps = step_phase_kernel<kM, V, hold, minb, block, 4>;
        static std::atomic<uint64_t> conf4{0};
        e = opt_in_smem(sweeps, smem, conf4);
        if (e != cudaSuccess) return e;
        sweeps<<<blocks, block, smem, s>>>(p, nullptr, nullptr);
    } else {
        first<<<blocks, block, smem, s>>>(p, nullptr, nullptr);
    }
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    // the list lengths live on the device: every later pass is launched with one block per `block` envs of the whole
    // batch, and the blocks past the end of the list return at once (a short fixed grid striding over the list
    // measured 20-25 % slower: two to four list rounds per block, the last one mostly empty)
    for (int j = 1; j <= plan.n; j++) {
        if (plan.stop[j - 1] >= p0.max_iters) break;  // nobody was suspended
        p.it_stop = (j < plan.n) ? plan.stop[j] : 0x7fffffff;
        p.min_lanes = (j < plan.n) ? plan.lanes[j] : 0;
        p.cont_list = lists + (int64_t)(j & 1) * p.N;
        p.cont_count = counts + j;
        later<<<blocks, block, smem, s>>>(p, lists + (int64_t)((j - 1) & 1) * p.N, counts + j - 1);
        e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

#ifndef SDCGYM_TMEM_MINB_SMALL
#define SDCGYM_TMEM_MINB_SMALL 5  // CTAs per SM of step_tmem_kernel at M <= 3 (96 registers; M = 4: 5 CTAs 0.563, 4 CTAs 0.550 ms)
#endif
template <int KIND, int V, bool DENSE>
static cudaError_t launch_step(const StepParams<kM>& p, cudaStream_t s) {
    if constexpr (DENSE && KIND == SDCGYM_ENV_FULL && kM < kTeamMinM) {
        static const PhasePlan plan;
        if (plan.n > 0 && p.cont_list && p.cont_count && p.pinv_scratch && p.old_states == nullptr &&
            p.N <= 0x7fffffff && p.max_iters > plan.stop[0])  // (the caller decides by passing the work buffers: the host
            // layer does so from 16 384 envs on - below that the second launch costs more than it saves)
            return launch_phased_dense<V>(p, plan, s);
    }
    if constexpr (DENSE && kM >= kTeamMinM) {
        // large dense Q_delta: one env per team of M lanes (team_kernels.cuh); collect_states keeps the per-thread kernel
        static const bool no_team = getenv("SDCGYM_NO_TEAM") != nullptr;  // A/B switch for tools/bench_dense.py
        if (p.old_states == nullptr && !no_team) {
            constexpr int envs_per_block = (kTeamBlock / 32) * (32 / kM);
            team_step_kernel<kM, KIND, V><<<(unsigned)((p.N + envs_per_block - 1) / envs_per_block), kTeamBlock, 0, s>>>(p);
            return cudaGetLastError();
        }
    }
    constexpr bool kStep = (KIND == SDCGYM_ENV_STEP);
    if constexpr (kStep && !DENSE && HoldPolicy<kM>::step == 0 && kM <= 7) {
        // sdc-v1, diagonal Q_delta, large batch: persistent blocks with the next tile's inputs in flight as bulk
        // asynchronous copies (stream_kernels.cuh); the tail that does not fill a tile takes the plain kernel below
        static const bool no_stream = getenv("SDCGYM_NO_STREAM") != nullptr;  // A/B switches for experiments
        static const bool stream_all = getenv("SDCGYM_STREAM_ALL") != nullptr;
        const int w = p.is_complex ? 2 : 1;
        const bool has_act = p.prec_type != SDCGYM_PREC_FIXED;
        const bool rows_ok = !has_act || (p.a_cs == w && p.a_es == (int64_t)kM * w &&
                                          (reinterpret_cast<uintptr_t>(p.action) & 15u) == 0);
        const bool aligned = ((reinterpret_cast<uintptr_t>(p.lam) | reinterpret_cast<uintptr_t>(p.S) |
                               reinterpret_cast<uintptr_t>(p.resnorm) | reinterpret_cast<uintptr_t>(p.niter) |
                               reinterpret_cast<uintptr_t>(p.episodes) | reinterpret_cast<uintptr_t>(p.rng_ctr) |
                               reinterpret_cast<uintptr_t>(p.norm_init)) & 15u) == 0 &&
                             (p.ld % 2) == 0;
        const int64_t tiles = p.N / kStreamTile;
        if (!no_stream && p.old_states == nullptr && rows_ok && aligned && tiles >= 148 * 2 &&
            (p.strategy == SDCGYM_REW_ITERATION_ONLY || (p.strategy == SDCGYM_REW_RESIDUAL_CHANGE && p.norm_init) ||
             stream_all)) {  // (measured faster for these two; the others are FP64-latency bound, see stream_kernels.cuh)
            constexpr int sminb = SDCGYM_STREAM_MINB > 0 ? SDCGYM_STREAM_MINB : HoldPolicy<kM>::step_minb;
            constexpr size_t smem = StreamStage<kM>::bytes;
            auto kern = step_stream_kernel<kM, V, sminb>;
            static std::atomic<uint64_t> configured{0};
            cudaError_t e = opt_in_smem(kern, smem, configured);
            if (e != cudaSuccess) return e;
            const int64_t want = (int64_t)148 * sminb;  // persistent: every SM at its resident block count
            const unsigned grid = (unsigned)(tiles < want ? tiles : want);
            kern<<<grid, kStreamTile, smem, s>>>(p, tiles, has_act ? kM * w * 8 : 0);
            e = cudaGetLastError();
            if (e != cudaSuccess) return e;
            const int64_t done = tiles * kStreamTile;
            if (done == p.N) return cudaSuccess;
            // tail: the same envs through the plain kernel, addressed by offset pointers
            StepParams<kM> q = p;
            q.N = p.N - done;
            q.lam += done; q.S += done; q.resnorm += done; q.niter += done; q.episodes += done; q.rng_ctr += done;
            if (q.norm_init) q.norm_init += done;
            if (q.action) q.action += done * p.a_es;
            if (q.reward) q.reward += done;
            if (q.flags) q.flags += done;
            if (q.info_res) q.info_res += done;
            if (q.info_niter) q.info_niter += done;
            if (q.info_lam) q.info_lam += 2 * done;
            if (q.term) q.term += done;
            q.env_offset += done;
            return launch_step<KIND, V, DENSE>(q, s);
        }
    }
    if constexpr (!DENSE && !kStep && kM <= 5) {
        // C of every env in tensor memory (step_tmem_kernel) instead of registers (M <= 4) / shared memory (M = 5).
        // Measured per 2^20-env step (tools/bench_headline.py): M = 2 0.255 -> 0.255, M = 3 0.368 -> 0.350, M = 4
        // 0.597 -> 0.550, M = 5 0.745 -> 0.755 ms: the default for M = 3, 4.  SDCGYM_TMEM=0 / 1: never / whenever it fits.
        static const int tmem_env = getenv("SDCGYM_TMEM") ? atoi(getenv("SDCGYM_TMEM")) : -1;
        const bool use_tmem = tmem_env < 0 ? (kM == 3 || kM == 4) : tmem_env != 0;
        if (use_tmem && p.old_states == nullptr) {
            step_tmem_kernel<kM, V, (kM <= 3) ? SDCGYM_TMEM_MINB_SMALL : 4><<<(unsigned)((p.N + 127) / 128), 128, 0, s>>>(p);
            return cudaGetLastError();
        }
    }
    constexpr int hold = DENSE ? kHoldDense : (kStep ? HoldPolicy<kM>::step : kHoldDiag);
    constexpr int minb = DENSE ? HoldPolicy<kM>::dense_minb : (kStep ? HoldPolicy<kM>::step_minb : HoldPolicy<kM>::diag_minb);
    constexpr int block = DENSE ? HoldPolicy<kM>::dense_block : ((!kStep) ? HoldPolicy<kM>::diag_block : kBlock);
    static_assert(!(DENSE && kStep && hold >= 3) || true, "");
    constexpr size_t smem = step_kernel_smem_bytes<kM, hold, block>();
    auto kernel = step_kernel<kM, KIND, V, DENSE, hold, minb, block>;
    if (smem > 48 * 1024) {
        // the opt-in is a per-DEVICE function attribute: remember it per (instantiation, device ordinal), so a process
        // that drives several GPUs configures each of them (devices beyond the table are configured on every launch)
        static std::atomic<uint64_t> configured{0};
        int dev = 0;
        cudaError_t e = cudaGetDevice(&dev);
        if (e != cudaSuccess) return e;
        const uint64_t bit = (dev >= 0 && dev < 64) ? (uint64_t(1) << dev) : 0;
        if (!(configured.load(std::memory_order_relaxed) & bit)) {
            e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
            configured.fetch_or(bit, std::memory_order_relaxed);
        }
    }
    kernel<<<(unsigned)((p.N + block - 1) / block), block, smem, s>>>(p);
    return cudaGetLastError();
}

#ifndef SDCGYM_FAST_MINB
#define SDCGYM_FAST_MINB 4  // blocks per SM of the substitution-sweep kernel at M <= 5 (experiments: 5 -> 96 registers)
#endif

// SDCGYM_SWEEP_CERTIFIED, diagonal Q_delta, sdc-v0: certificate -> substitution sweeps -> exact kernel over the
// fallback list (fast_kernels.cuh).  Three launches on the caller's stream.
template <int V>
static cudaError_t launch_certified_diag(const StepParams<kM>& p, const FastWork& fw, cudaStream_t s) {
    cert_kernel<kM, V><<<(unsigned)((p.N + kCertBlock - 1) / kCertBlock), kCertBlock, 0, s>>>(p, fw);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    constexpr int fminb = (kM <= 5) ? SDCGYM_FAST_MINB : ((kM <= 7) ? 3 : 2);
    fast_step_kernel<kM, V, fminb><<<(unsigned)((p.N + kFastBlock - 1) / kFastBlock), kFastBlock, 0, s>>>(p, fw);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    constexpr int hold = kHoldDiag, minb = HoldPolicy<kM>::diag_minb, block = HoldPolicy<kM>::diag_block;
    constexpr size_t smem = step_kernel_smem_bytes<kM, hold, block>();
    auto kernel = step_list_kernel<kM, V, hold, minb, block>;
    static std::atomic<uint64_t> configured{0};
    e = opt_in_smem(kernel, smem, configured);
    if (e != cudaSuccess) return e;
    // a fixed grid (the list is short and its length lives on the device): grid-stride over the list
    const int64_t want = (p.N / 16 + block - 1) / block;
    const unsigned grid = (unsigned)(want < 1 ? 1 : (want > 148 * 4 ? 148 * 4 : want));
    kernel<<<grid, block, smem, s>>>(p, fw);
    return cudaGetLastError();
}

// sdcgym_full_solve_counts: the per-thread kernel of launch_step at HoldPolicy's residency for every M (the team kernel
// and the phased solve give the same bits and are not used), plus the histogram behind the side store.  With
// PopulationEval, `rows` rows of the population (gridDim.y), hist [rows][max_iters + 3].
template <int V, bool DENSE, class Src>
static cudaError_t launch_full_solve_counts(const StepParams<kM>& p, const Src& src, int64_t* hist, cudaStream_t s,
                                            unsigned rows = 1) {
    constexpr int hold = DENSE ? kHoldDense : kHoldDiag;
    constexpr int minb = DENSE ? HoldPolicy<kM>::dense_minb : HoldPolicy<kM>::diag_minb;
    constexpr int block = DENSE ? HoldPolicy<kM>::dense_block : HoldPolicy<kM>::diag_block;
    constexpr bool kPop = std::is_same<Src, PopulationEval>::value;
    const size_t smem = step_kernel_smem_bytes<kM, hold, block>() + (hist ? (size_t)(p.max_iters + 3) * sizeof(int) : 0);
    auto kernel = [] {
        if constexpr (kPop) return full_solve_counts_population_kernel<kM, V, DENSE, hold, minb, block>;
        else return full_solve_counts_kernel<kM, V, DENSE, hold, minb, block>;
    }();
    if (smem > 48 * 1024) {
        // per-device opt-in, raised when a call needs more than the largest size granted so far
        static std::atomic<size_t> granted[64];
        int dev = 0;
        cudaError_t e = cudaGetDevice(&dev);
        if (e != cudaSuccess) return e;
        if (dev < 0 || dev >= 64 || granted[dev].load(std::memory_order_relaxed) < smem) {
            e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
            if (dev >= 0 && dev < 64) granted[dev].store(smem, std::memory_order_relaxed);
        }
    }
    kernel<<<dim3((unsigned)((p.N + block - 1) / block), rows), block, smem, s>>>(
        p, src, reinterpret_cast<unsigned long long*>(hist));
    return cudaGetLastError();
}

}  // namespace sdcgym

using namespace sdcgym;

namespace sdcgym {

// StepParams and the lambda source of sdcgym_full_solve_counts(_population): no env state, every plane NULL
static void fill_counts(StepParams<kM>& p, ResetEval& src, const sdcgym_env_desc* d, const sdcgym_lambda_grid* g,
                        int64_t N, const double* lam, const double* action, int64_t a_es, int64_t a_cs) {
    sdcgym_state st{};
    st.N = st.ld = N;
    fill_params<kM>(p, d, &st);
    p.action = action;
    p.a_es = a_es;
    p.a_cs = a_cs;
    p.autoreset = 0;
    p.strategy = SDCGYM_REW_ITERATION_ONLY;
    src.lam = g ? nullptr : lam;
    if (g) {
        src.grid_re = g->n_re;
        src.grid_im = g->n_im;
        src.grid_first = g->first;
        src.re_lo = g->re_lo;
        src.re_hi = g->re_hi;
        src.im_lo = g->im_lo;
        src.im_hi = g->im_hi;
    }
}

template <class Src>
static cudaError_t dispatch_full_solve_counts(const sdcgym_env_desc* d, const StepParams<kM>& p, const Src& src,
                                              int64_t* hist, cudaStream_t s, unsigned rows = 1) {
    bool dense = d->prec_type != SDCGYM_PREC_DIAG;
    if (d->prec_type == SDCGYM_PREC_FIXED) {  // a fixed diagonal matrix takes the diagonal kernel, as in sdcgym_step
        bool diagonal = true;
        for (int r = 0; r < kM; r++)
            for (int c = 0; c < kM; c++)
                if (r != c && d->Qd_fixed[r * kM + c] != 0.0) diagonal = false;
        dense = !diagonal;
    }
    if (d->blas_variant == SDCGYM_BLAS_SKYLAKEX)
        return dense ? launch_full_solve_counts<0, true>(p, src, hist, s, rows)
                     : launch_full_solve_counts<0, false>(p, src, hist, s, rows);
    return dense ? launch_full_solve_counts<1, true>(p, src, hist, s, rows)
                 : launch_full_solve_counts<1, false>(p, src, hist, s, rows);
}

}  // namespace sdcgym

extern "C" int SDCGYM_CAT(sdcgym_launch_full_solve_counts_m, SDCGYM_M)(
    const sdcgym_env_desc* d, const sdcgym_lambda_grid* g, int64_t N, const double* lam, const double* action,
    int64_t a_es, int64_t a_cs, int32_t* niter_out, double* residual_out, uint8_t* flags_out, double* lam_out,
    int64_t* hist, void* stream) {
    StepParams<kM> p;
    ResetEval src{};
    fill_counts(p, src, d, g, N, lam, action, a_es, a_cs);
    p.info_niter = niter_out;
    p.info_res = residual_out;
    p.flags = flags_out;
    p.info_lam = lam_out;
    return (int)dispatch_full_solve_counts(d, p, src, hist, (cudaStream_t)stream);
}

// P rows in launches of at most 65535 (gridDim.y), each row's histogram at hist + row * (max_iters + 3)
extern "C" int SDCGYM_CAT(sdcgym_launch_full_solve_counts_population_m, SDCGYM_M)(
    const sdcgym_env_desc* d, const sdcgym_lambda_grid* g, int64_t N, const double* lam, int64_t P,
    const double* action, int64_t a_rs, int64_t a_cs, int64_t* hist, void* stream) {
    constexpr int64_t kMaxRows = 65535;
    StepParams<kM> p;
    PopulationEval src{};
    fill_counts(p, src, d, g, N, lam, action, 0, a_cs);
    src.a_rs = a_rs;
    for (int64_t r0 = 0; r0 < P; r0 += kMaxRows) {
        const int64_t rows = P - r0 < kMaxRows ? P - r0 : kMaxRows;
        p.action = action + r0 * a_rs;
        const cudaError_t e = dispatch_full_solve_counts(d, p, src, hist + r0 * (int64_t)(d->max_iters + 3),
                                                         (cudaStream_t)stream, (unsigned)rows);
        if (e != cudaSuccess) return (int)e;
    }
    return 0;
}

extern "C" int SDCGYM_CAT(sdcgym_launch_reset_m, SDCGYM_M)(const sdcgym_env_desc* d, const sdcgym_state* st,
                                                          const double* lam_in, const uint8_t* mask, double* old_states,
                                                          void* stream) {
    StepParams<kM> p;
    fill_params<kM>(p, d, st);
    p.lam_in = lam_in;
    p.mask = mask;
    p.old_states = old_states;
    if (p.N <= 0) return 0;
    const unsigned grid = (unsigned)((p.N + kBlock - 1) / kBlock);
    cudaStream_t s = (cudaStream_t)stream;
    if (d->blas_variant == SDCGYM_BLAS_SKYLAKEX) reset_kernel<kM, 0><<<grid, kBlock, 0, s>>>(p);
    else reset_kernel<kM, 1><<<grid, kBlock, 0, s>>>(p);
    return (int)cudaGetLastError();
}

extern "C" int SDCGYM_CAT(sdcgym_launch_step_m, SDCGYM_M)(const sdcgym_env_desc* d, const sdcgym_state* st,
                                                         const sdcgym_step_io* io, void* stream) {
    StepParams<kM> p;
    fill_params<kM>(p, d, st);
    fill_step_io<kM>(p, io);
    if (p.N <= 0) return 0;
    cudaStream_t s = (cudaStream_t)stream;
    bool dense = d->prec_type != SDCGYM_PREC_DIAG;
    if (d->prec_type == SDCGYM_PREC_FIXED) {  // a fixed diagonal matrix takes the diagonal fast path
        bool diagonal = true;
        for (int r = 0; r < kM; r++)
            for (int c = 0; c < kM; c++)
                if (r != c && d->Qd_fixed[r * kM + c] != 0.0) diagonal = false;
        dense = !diagonal;
    }
    const bool full = d->env_kind == SDCGYM_ENV_FULL;
    const bool skx = d->blas_variant == SDCGYM_BLAS_SKYLAKEX;
    cudaError_t e;
    if (d->sweep_mode == SDCGYM_SWEEP_CERTIFIED && full && !dense && io->old_states == nullptr) {
        FastWork fw{st->cert, st->fallback_list, st->fallback_count};
        e = skx ? launch_certified_diag<0>(p, fw, s) : launch_certified_diag<1>(p, fw, s);
        return (int)e;
    }
#define SDCGYM_DISPATCH(KIND, V, DENSE) e = launch_step<KIND, V, DENSE>(p, s)
    if (full) {
        if (skx) { if (dense) SDCGYM_DISPATCH(SDCGYM_ENV_FULL, 0, true); else SDCGYM_DISPATCH(SDCGYM_ENV_FULL, 0, false); }
        else     { if (dense) SDCGYM_DISPATCH(SDCGYM_ENV_FULL, 1, true); else SDCGYM_DISPATCH(SDCGYM_ENV_FULL, 1, false); }
    } else {
        if (skx) { if (dense) SDCGYM_DISPATCH(SDCGYM_ENV_STEP, 0, true); else SDCGYM_DISPATCH(SDCGYM_ENV_STEP, 0, false); }
        else     { if (dense) SDCGYM_DISPATCH(SDCGYM_ENV_STEP, 1, true); else SDCGYM_DISPATCH(SDCGYM_ENV_STEP, 1, false); }
    }
#undef SDCGYM_DISPATCH
    return (int)e;
}
