// C ABI, device part (include/heyoka_b200.h section C): device-resident batch state, kernel selection and
// launches. The kernels themselves are in kernels.cuh.
#include <heyoka_b200.h>

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <memory>
#include <new>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include <cuda_runtime.h>

#include "capi_common.hpp"
#include "coop_variants.hpp"
#include "device_program.cuh"
#include "kernels.cuh"
#include "nb_kernel.cuh"
#include "nb_plan.hpp"
#include "nb_variants.hpp"
#include "nn_kernel.cuh"
#include "nn_plan.hpp"
#include "nn_variants.hpp"
#include "small_kernels.cuh"
#include "ev_kernels.cuh"
#include "program.hpp"
#include "smem_plan.hpp"

namespace hy = heyoka_b200;
namespace dev = heyoka_b200::dev;
using hy::detail::cuda_error;
using hy::detail::translate_exception;

#define HY_CUDA_CHECK(expr)                                                                                            \
    do {                                                                                                               \
        const cudaError_t err_ = (expr);                                                                               \
        if (err_ != cudaSuccess) {                                                                                     \
            throw cuda_error(std::string("CUDA error in " #expr ": ") + cudaGetErrorString(err_));                     \
        }                                                                                                              \
    } while (0)

// ------------------------------------------------------------------------------------------------
// Cooperative-kernel dispatch over (lanes per CTA, lanes per thread).
// ------------------------------------------------------------------------------------------------
namespace
{

using hy::detail::coop_variant;

// maxt: upper bound on the threads per CTA the variant was compiled for (256: up to 255 registers per thread).
// mode: 1 = the plan contains elementary ops, 0 = superinstructions only, 2 / 3 = idem with tensor memory,
// 4 = any plan, tape and tables in global memory, 5 = idem with the whole CTA working on one chunk of lanes.
const coop_variant *find_variant(int L, int N, int maxt, int mode)
{
    const hy::detail::coop_family fams[] = {
        hy::detail::coop_family_n1_512_m1(),
        hy::detail::coop_family_n1_512_m0(),
        hy::detail::coop_family_n1_256_m1(),
        hy::detail::coop_family_n1_256_m0(),
        hy::detail::coop_family_n2_512_m1(),
        hy::detail::coop_family_n2_512_m0(),
        hy::detail::coop_family_n2_256_m1(),
        hy::detail::coop_family_n2_256_m0(),
        hy::detail::coop_family_n4_512_m1(),
        hy::detail::coop_family_n4_512_m0(),
        hy::detail::coop_family_n4_256_m1(),
        hy::detail::coop_family_n4_256_m0(),
        hy::detail::coop_family_n1_512_m2(),
        hy::detail::coop_family_n1_512_m3(),
        hy::detail::coop_family_n1_384_m2(),
        hy::detail::coop_family_n1_384_m3(),
        hy::detail::coop_family_n1_256_m2(),
        hy::detail::coop_family_n1_256_m3(),
        hy::detail::coop_family_n2_512_m2(),
        hy::detail::coop_family_n2_512_m3(),
        hy::detail::coop_family_n2_384_m2(),
        hy::detail::coop_family_n2_384_m3(),
        hy::detail::coop_family_n2_256_m2(),
        hy::detail::coop_family_n2_256_m3(),
        hy::detail::coop_family_n1_512_m4(),
        hy::detail::coop_family_n2_512_m4(),
        hy::detail::coop_family_n1_512_m5(),
        hy::detail::coop_family_n2_512_m5()};
    for (const auto &f : fams) {
        for (std::size_t i = 0; i < f.n; ++i) {
            if (f.v[i].L == L && f.v[i].N == N && f.v[i].maxt == maxt && f.v[i].mode == mode) {
                return f.v + i;
            }
        }
    }
    return nullptr;
}

// The N-body kernel's instantiations (nb_variants.hpp).
const hy::detail::nb_variant *find_nb_variant(int LT, bool cta, bool tmem, int maxt, bool lane = false)
{
    const hy::detail::nb_family fams[] = {hy::detail::nb_family_lt1_cta0(),  hy::detail::nb_family_lt2_cta0(),
                                          hy::detail::nb_family_lt4_cta0(),  hy::detail::nb_family_lt8_cta0(),
                                          hy::detail::nb_family_lt16_cta0(), hy::detail::nb_family_lt32_cta0(),
                                          hy::detail::nb_family_lt1_cta1(),  hy::detail::nb_family_lane()};
    for (const auto &f : fams) {
        for (std::size_t i = 0; i < f.n; ++i) {
            if (f.v[i].LT == LT && f.v[i].cta == cta && f.v[i].tmem == tmem && f.v[i].maxt == maxt
                && f.v[i].lane == lane) {
                return f.v + i;
            }
        }
    }
    return nullptr;
}

// The program tables of the cooperative kernels as one blob of 32-bit words (copied to shared memory by every
// CTA): header (dev::coop_header), ops (8 words per item: opcode, a, b, c, destination row, 3 spare), level
// offsets, n-ary argument table, superinstruction operand tables, constants (doubles), state-variable table
// ({row, right-hand-side reference} per state variable).
std::vector<std::uint32_t> make_plan_blob(const hy::detail::smem_plan &pl, const hy_program &p)
{
    std::vector<std::uint32_t> b(sizeof(dev::coop_header) / 4u, 0u);
    const auto align = [&](std::size_t words) {
        while (b.size() % words != 0u) {
            b.push_back(0u);
        }
    };
    dev::coop_header h{};
    h.n_items = static_cast<std::uint32_t>(pl.ops.size());
    h.n_segments = pl.n_segments;
    h.n_eq = p.n_eq;
    h.n_slots = pl.n_slots;
    h.n_gslots = pl.n_gslots;
    h.tmem = pl.tmem;
    align(4);
    h.off_ops = static_cast<std::uint32_t>(b.size());
    for (std::size_t i = 0; i < pl.ops.size(); ++i) {
        const auto &op = pl.ops[i];
        b.insert(b.end(), {op.opcode, op.a, op.b, op.c, pl.dst[i], pl.svo[i], 0u, 0u});
    }
    h.off_seg = static_cast<std::uint32_t>(b.size());
    b.insert(b.end(), pl.seg_offsets.begin(), pl.seg_offsets.end());
    h.off_args = static_cast<std::uint32_t>(b.size());
    b.insert(b.end(), pl.args.begin(), pl.args.end());
    h.off_aux = static_cast<std::uint32_t>(b.size());
    b.insert(b.end(), pl.aux.begin(), pl.aux.end());
    align(2);
    h.off_consts = static_cast<std::uint32_t>(b.size());
    const auto push_double = [&](double c) {
        std::uint32_t w[2];
        std::memcpy(w, &c, sizeof(double));
        b.push_back(w[0]);
        b.push_back(w[1]);
    };
    for (const double c : p.consts) {
        push_double(c);
    }
    for (const double c : pl.extra_consts) {
        push_double(c);
    }
    align(2);
    // Reciprocals 1 / k (IEEE division on the host) for the exact small-integer divisions.
    h.off_rcp = static_cast<std::uint32_t>(b.size());
    for (std::uint32_t k = 0; k <= p.order + 2u; ++k) {
        const double r = k == 0u ? 0. : 1. / static_cast<double>(k);
        std::uint32_t w[2];
        std::memcpy(w, &r, sizeof(double));
        b.push_back(w[0]);
        b.push_back(w[1]);
    }
    align(4);
    h.off_sv = static_cast<std::uint32_t>(b.size());
    for (std::uint32_t i = 0; i < p.n_eq; ++i) {
        b.insert(b.end(), {pl.sv_rows[i], pl.sv_defs[i], pl.sv_cover[i], pl.sv_parent[i]});
    }
    h.off_svout = static_cast<std::uint32_t>(b.size());
    b.insert(b.end(), pl.svout.begin(), pl.svout.end());
    h.off_svphase = static_cast<std::uint32_t>(b.size());
    h.n_svphase = static_cast<std::uint32_t>(pl.sv_phase.size());
    b.insert(b.end(), pl.sv_phase.begin(), pl.sv_phase.end());
    align(4);
    h.n_words = static_cast<std::uint32_t>(b.size());
    std::memcpy(b.data(), &h, sizeof(h));
    return b;
}

// Shared memory of one warp owning L lanes (must match dev::coop_smem<L>::warp_doubles()).
std::size_t coop_warp_bytes(std::uint32_t n_slots, int L)
{
    const std::size_t l = static_cast<std::size_t>(L);
    return (static_cast<std::size_t>(n_slots) * l + 2u * l + (l + 1u) / 2u + 1u) / 2u * 2u * sizeof(double);
}

} // namespace

// ------------------------------------------------------------------------------------------------
// Host objects. A batch (hy_batch) is a front over one or more shards: a shard is one device and a contiguous block of
// the batch's lanes, with the device arrays, plans, kernel selection, event state and stream of those lanes.
// ------------------------------------------------------------------------------------------------
struct shard {
    int device = 0;
    cudaStream_t stream = nullptr;
    std::uint32_t n = 0;
    std::uint32_t n_eq = 0, n_pars = 0, order = 0, n_uvars = 0;
    bool high_accuracy = false;

    // Device copies of the program arrays ("hbm" encoding) ...
    uint4 *d_ops = nullptr;
    std::uint32_t *d_args = nullptr, *d_sv_defs = nullptr;
    double *d_consts = nullptr;
    dev::program prog{};
    // ... and of the cooperative plan.
    hy::detail::smem_plan plan;
    std::uint32_t *d_blob = nullptr;
    std::size_t blob_bytes = 0; // rounded up to 16 bytes
    double *d_gscratch = nullptr; // overflow tape of the cooperative kernels (spilled private rows)
    double *d_cscratch = nullptr; // private per-warp coefficient store of the cooperative kernels (see dev::coef_view)
    std::shared_ptr<const hy_program> prog_host; // kept for re-planning
    bool opt_fuse = true, opt_fuse_sv = true;
    int opt_spill = -1; // -1 automatic, 0 never, 1 always
    bool opt_tmem = true, allow_tmem = true;
    std::uint32_t opt_tmem_rows = 0; // 0: automatic, 2 / 3: forced (HEYOKA_B200_TMEM_ROWS)
    void replan(bool spill, std::uint32_t tmem_max_pairs = 0, std::uint32_t tmem_rows = 2);
    void ensure_tc();
    void setup_coop_global(int L, int N, std::uint32_t threads, int cta = -1);
    bool c_cta = false; // ... and the whole CTA working on one chunk of lanes (kernel mode 5)
    bool c_global = false; // cooperative kernel with the tape in global memory (kernel mode 4)
    // The dedicated N-body kernel (nb_kernel.cuh): plan, device copies of its tables, selected instantiation.
    hy::detail::nb_plan nbp;
    hy::detail::nb_pair_desc *d_nb_pairs = nullptr;
    hy::detail::nb_role *d_nb_roles = nullptr;
    std::uint32_t opt_nb_threads = 0; // HEYOKA_B200_NB_THREADS: preferred CTA size of the N-body kernel
    double *d_nb_consts = nullptr, *d_nb_fac = nullptr;
    dev::nb_dev_plan nbd{};
    const hy::detail::nb_variant *nbv = nullptr;
    coop_variant nb_cv{}; // (L, N, maxt, mode 6) of the selected N-body instantiation, for the code that reads cv->L
    bool nb_on = false;
    int opt_nb = -1; // -1 automatic, 0 never (HEYOKA_B200_NB=0), 1 preferred
    bool setup_nb(int LT, std::uint32_t threads, int want_tmem, int want_cta, int want_lane = 0);
    int opt_nb_lane = -1; // one thread per lane for single-pair systems: -1 automatic, 0 never (HEYOKA_B200_NB_LANE=0)
    bool nb_lane = false;
    // The dense-network kernel (nn_kernel.cuh): plan, padded weight image, device plan.
    hy::detail::nn_plan nnp;
    double *d_nn_wimg = nullptr;
    std::uint32_t *d_nn_out = nullptr;
    dev::nn_dev_plan nnd{};
    bool nn_on = false;
    int opt_nn = -1; // 0: never (HEYOKA_B200_NN=0)
    bool setup_nn();

    // Event detection (section E of the C ABI; ev_kernels.cuh). n_ev > 0: the program carries event equations, every
    // step is an event step (jet without propagation + detection + propagation cut at the first terminal event).
    std::uint32_t n_ev = 0;
    dev::ev_args eva{};
    std::vector<void *> ev_allocs;
    std::vector<hy_event_rec> ev_host; // the events of the last step in this shard's lanes, in callback order
    void ev_setup(std::uint32_t n_te, const std::int32_t *dirs, const double *cooldowns, double tol);
    void ev_step(const double *max_delta_t, int backward);

    // Resident arrays.
    double *d_state = nullptr, *d_pars = nullptr, *d_t_hi = nullptr, *d_t_lo = nullptr, *d_last_h = nullptr,
           *d_tc = nullptr, *d_d_out = nullptr;
    long long *d_step_outcome = nullptr, *d_prop_outcome = nullptr;
    double *d_prop_min_h = nullptr, *d_prop_max_h = nullptr;
    unsigned long long *d_prop_n_steps = nullptr, *d_prop_iters = nullptr;
    unsigned char *d_skip = nullptr; // per-lane mask of the masked zero-length step (propagate_finish())

    // Scratch.
    double *d_scratch = nullptr; // per-warp tape slabs ("hbm" strategy only, allocated on demand)
    std::size_t slab_doubles = 0;
    double *d_tmp = nullptr;      // 3 * n doubles: staged per-lane inputs (t_final hi/lo, max_delta_t)
    double *d_snapshot = nullptr; // state + time snapshot for the global-exit replay
    unsigned int *d_counter = nullptr;
    dev::run_flags *d_flags = nullptr;

    // Kernel selection / launch geometry.
    std::uint32_t n_sms = 0;
    std::size_t smem_per_block_max = 0, smem_per_sm = 0;
    int mode = 0;           // 1 = hbm, 2 = coop (resolved)
    const coop_variant *cv = nullptr;
    std::uint32_t c_threads = 0, c_grid = 0, c_ctas_per_sm = 0;
    std::size_t c_smem = 0;
    std::uint32_t h_threads = 256, h_blocks_per_sm = 0, h_grid = 0;
    std::uint64_t n_launches = 0;

    ~shard();
    void free_all() noexcept;
    dev::batch view() const;
    template <typename T>
    T *dalloc(std::size_t count);
    template <typename T>
    T *dupload(const std::vector<T> &v);
    void configure(int want_mode, int L, int N, std::uint32_t threads, std::uint32_t blocks_per_sm);
    void setup_hbm(std::uint32_t threads, std::uint32_t blocks_per_sm);
    bool setup_coop(int L, int N, std::uint32_t threads, std::uint32_t ctas_per_sm);
    void launch(bool prop, const dev::run_args &R);
};

struct hy_batch {
    std::uint32_t n = 0;
    // Shard i holds the lanes [shard_off[i], shard_off[i + 1]). sharded: made by hy_batch_create_multi(), which
    // refuses the single-device-only entry points even with one shard.
    std::vector<std::unique_ptr<shard>> shards;
    std::vector<std::uint32_t> shard_off;
    bool sharded = false;

    std::uint32_t n_ev = 0, n_te = 0;
    bool ev_set = false;
    std::vector<hy_event_rec> ev_host; // the events of the last step, in the order the callbacks must run
};

template <typename T>
T *shard::dalloc(std::size_t count)
{
    void *p = nullptr;
    HY_CUDA_CHECK(cudaMalloc(&p, std::max<std::size_t>(count, 1u) * sizeof(T)));
    return static_cast<T *>(p);
}

template <typename T>
T *shard::dupload(const std::vector<T> &v)
{
    T *p = dalloc<T>(v.size());
    if (!v.empty()) {
        HY_CUDA_CHECK(cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    }
    return p;
}

void shard::free_all() noexcept
{
    for (void *p :
         {static_cast<void *>(d_ops), static_cast<void *>(d_args), static_cast<void *>(d_sv_defs),
          static_cast<void *>(d_consts), static_cast<void *>(d_blob), static_cast<void *>(d_gscratch),
          static_cast<void *>(d_cscratch),
          static_cast<void *>(d_state),
          static_cast<void *>(d_pars),
          static_cast<void *>(d_t_hi), static_cast<void *>(d_t_lo), static_cast<void *>(d_last_h),
          static_cast<void *>(d_tc), static_cast<void *>(d_d_out), static_cast<void *>(d_step_outcome),
          static_cast<void *>(d_prop_outcome), static_cast<void *>(d_prop_min_h), static_cast<void *>(d_prop_max_h),
          static_cast<void *>(d_prop_n_steps), static_cast<void *>(d_prop_iters), static_cast<void *>(d_skip),
          static_cast<void *>(d_scratch), static_cast<void *>(d_tmp),
          static_cast<void *>(d_snapshot), static_cast<void *>(d_counter), static_cast<void *>(d_flags),
          static_cast<void *>(d_nb_pairs), static_cast<void *>(d_nb_roles), static_cast<void *>(d_nb_consts),
          static_cast<void *>(d_nb_fac), static_cast<void *>(d_nn_wimg), static_cast<void *>(d_nn_out)}) {
        if (p != nullptr) {
            cudaFree(p);
        }
    }
    for (void *p : ev_allocs) {
        cudaFree(p);
    }
    ev_allocs.clear();
}

shard::~shard()
{
    int cur = 0;
    if (cudaGetDevice(&cur) == cudaSuccess) {
        cudaSetDevice(device);
        free_all();
        cudaSetDevice(cur);
    }
}

dev::batch shard::view() const
{
    dev::batch b{};
    b.n = n;
    b.state = d_state;
    b.t_hi = d_t_hi;
    b.t_lo = d_t_lo;
    b.last_h = d_last_h;
    b.tc = d_tc;
    b.pars = d_pars;
    b.step_outcome = d_step_outcome;
    b.prop_outcome = d_prop_outcome;
    b.prop_min_h = d_prop_min_h;
    b.prop_max_h = d_prop_max_h;
    b.prop_n_steps = d_prop_n_steps;
    b.prop_iters = d_prop_iters;
    return b;
}

void shard::setup_hbm(std::uint32_t threads, std::uint32_t blocks_per_sm)
{
    if (threads != 0u) {
        if (threads % 32u != 0u || threads > 256u) {
            throw std::invalid_argument("block_threads must be a multiple of 32 not larger than 256");
        }
        h_threads = threads;
    }
    if (blocks_per_sm == 0u) {
        int occ = 0;
        HY_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, dev::k_hbm<true>,
                                                                    static_cast<int>(h_threads), 0));
        blocks_per_sm = static_cast<std::uint32_t>(std::max(occ, 1));
    }
    h_blocks_per_sm = blocks_per_sm;

    // One slab per resident warp; never more warps than chunks of 32 lanes.
    const std::uint32_t warps_per_block = h_threads / 32u;
    const std::uint32_t n_chunks = (n + 31u) / 32u;
    const std::uint32_t needed_blocks = (n_chunks + warps_per_block - 1u) / warps_per_block;
    h_grid = std::max(1u, std::min(n_sms * h_blocks_per_sm, needed_blocks));

    if (d_scratch != nullptr) {
        HY_CUDA_CHECK(cudaFree(d_scratch));
        d_scratch = nullptr;
    }
    slab_doubles = static_cast<std::size_t>(n_uvars) * (order + 1u) * 32u;
    // The slabs of the resident warps must fit in (half of the free) device memory: large systems (model::ffnn
    // 3 x 64: 43 MB per warp) run with fewer resident blocks rather than failing to allocate.
    {
        std::size_t free_b = 0, total_b = 0;
        HY_CUDA_CHECK(cudaMemGetInfo(&free_b, &total_b));
        const std::size_t per_block = static_cast<std::size_t>(warps_per_block) * slab_doubles * sizeof(double);
        const std::size_t max_blocks = std::max<std::size_t>(free_b / 2u / std::max<std::size_t>(per_block, 1u), 1u);
        h_grid = static_cast<std::uint32_t>(std::min<std::size_t>(h_grid, max_blocks));
    }
    d_scratch = dalloc<double>(static_cast<std::size_t>(h_grid) * warps_per_block * slab_doubles);
    mode = 1;
}

void shard::replan(bool spill, std::uint32_t tmem_max_pairs, std::uint32_t tmem_rows)
{
    plan = hy::detail::make_smem_plan(*prog_host, opt_fuse, opt_fuse_sv, spill, tmem_max_pairs, tmem_rows);
    const auto blob = make_plan_blob(plan, *prog_host);
    if (d_blob != nullptr) {
        HY_CUDA_CHECK(cudaFree(d_blob));
        d_blob = nullptr;
    }
    d_blob = dupload(blob);
    blob_bytes = (blob.size() + 3u) / 4u * 16u;
}

// Returns false if the requested / any configuration does not fit in shared memory.
// L = lanes per warp, N = lanes per thread, threads = 32 x warps per block.
bool shard::setup_coop(int L, int N, std::uint32_t threads, std::uint32_t ctas_per_sm)
{
    const std::size_t reserve = 1024u; // per-block reservation of the driver
    const bool auto_shape = N == 0 && L == 0;
    if (N == 0) {
        // Two lanes per thread: the interpreter's per-item overhead is shared and the recurrences get ILP 2.
        N = (L == 0 || L >= 2) ? 2 : 1;
    }
    // Optional overflow tape (HEYOKA_B200_SPILL=1): the superinstructions' private history rows move from shared
    // memory to global memory / L2, which lets 12 instead of 8 warps of the 6-body system reside on an SM.
    // Measured slower (1.89e7 vs 2.47e7 lane-steps/s: the L2 latency lands on the serial pow recurrence), hence
    // off by default; kept because it is what a system slightly too large for shared memory needs.
    {
        const bool have_spill = plan.n_gslots != 0u;
        const bool want_spill = opt_spill > 0;
        if (want_spill != have_spill || plan.tmem) {
            replan(want_spill); // (the tensor-memory decision is taken again below for this L, N)
        }
    }
    if (L == 0) {
        // Lanes per warp: enough of them that an average dependency segment gives work to most of the
        // 32 threads (one work item = one u variable x N lanes), as long as at least 4 warps fit on an SM.
        const double avg_width = static_cast<double>(plan.ops.size()) / std::max(1u, plan.n_segments);
        for (const int cand : {1, 2, 4, 8, 16, 32}) {
            if (cand < N) {
                continue;
            }
            const auto bytes = coop_warp_bytes(plan.n_slots, cand);
            if (blob_bytes + bytes + reserve > smem_per_block_max || (smem_per_sm - blob_bytes) / bytes < 4u) {
                break;
            }
            L = cand;
            if (avg_width * cand / N >= 12.) {
                break;
            }
        }
        if (L == 0) {
            // Not even 4 warps of the smallest shape fit: take whatever fits at all.
            if (blob_bytes + coop_warp_bytes(plan.n_slots, N) + reserve > smem_per_block_max) {
                return false;
            }
            L = N;
        }
    }
    // Warps per CTA that fit next to one copy of the tables (at most 16).
    const auto fit_warps = [&](std::uint32_t n_slots, int lanes) -> std::size_t {
        const auto wb = coop_warp_bytes(n_slots, lanes);
        if (blob_bytes + wb + reserve > smem_per_block_max) {
            return 0u;
        }
        return std::min<std::size_t>((smem_per_block_max - reserve - blob_bytes) / wb, 16u);
    };
    // Tensor memory (HEYOKA_B200_TMEM=0 disables): if the program consists of superinstructions only, with at
    // most one pair interaction per thread of a warp, the history rows that only their own thread touches (r^2,
    // r^alpha, optionally one of the coordinate differences) can live in TMEM (one TMEM lane per thread, 512
    // columns shared by the warps of a quadrant) instead of shared memory. Taken when it lets more warps reside
    // on an SM. 6-body system, order 20: 8 warps of 2 lanes without TMEM; 12 with two rows of 2 lanes per thread
    // in TMEM; 16 with three rows of 1 lane per thread (2 lanes per warp, 30 busy threads in the pair level).
    const auto tm_warps_of = [&](int lanes_per_thread, std::uint32_t rows) -> std::size_t {
        const std::uint32_t cols = rows * (order + 1u) * 2u * static_cast<std::uint32_t>(lanes_per_thread);
        return cols <= 512u ? 4u * (512u / cols) : 0u;
    };
    struct tm_choice {
        std::uint32_t rows = 0;
        std::size_t warps = 0;
    };
    const auto best_tmem = [&](int lanes, int lanes_per_thread) {
        tm_choice best;
        const std::uint32_t G = static_cast<std::uint32_t>(lanes / lanes_per_thread);
        if (!(opt_tmem && allow_tmem && lanes_per_thread <= 2 && G != 0u && G <= 32u && opt_spill <= 0)) {
            return best;
        }
        for (const std::uint32_t rows : {2u, 3u}) {
            if ((opt_tmem_rows != 0u && rows != opt_tmem_rows)
                || find_variant(lanes, lanes_per_thread, 512, static_cast<int>(rows)) == nullptr) {
                continue;
            }
            const auto cand = hy::detail::make_smem_plan(*prog_host, opt_fuse, opt_fuse_sv, false, 32u / G, rows);
            if (cand.tmem != rows) {
                continue;
            }
            const auto w = std::min(fit_warps(cand.n_slots, lanes), tm_warps_of(lanes_per_thread, rows));
            if (w > best.warps) {
                best = tm_choice{rows, w};
            }
        }
        return best;
    };
    {
        tm_choice pick = best_tmem(L, N);
        if (auto_shape && plan.n_fused != 0u && plan.n_fused <= 32u) {
            // The tensor-memory shape of choice: 1 lane per thread and as many lanes per warp as give every thread
            // one pair interaction (15 pairs: 2 lanes, 30 busy threads; 1 pair: 32 lanes). Taken when it puts
            // more lanes in flight on an SM.
            int alt_l = 1;
            while (static_cast<std::uint32_t>(2 * alt_l) * plan.n_fused <= 32u) {
                alt_l *= 2;
            }
            const auto alt = best_tmem(alt_l, 1);
            if (alt.warps * static_cast<std::size_t>(alt_l)
                > std::max(pick.warps, fit_warps(plan.n_slots, L)) * static_cast<std::size_t>(L)) {
                pick = alt;
                L = alt_l;
                N = 1;
            }
        }
        if (pick.rows != 0u && pick.warps > fit_warps(plan.n_slots, L)) {
            replan(false, 32u / static_cast<std::uint32_t>(L / N), pick.rows);
            // Level 0 must be exactly the pair interactions, at most one per thread.
            const auto b0 = plan.seg_offsets[0], e0 = plan.seg_offsets[1];
            bool ok = plan.tmem == pick.rows && (e0 - b0) * static_cast<std::uint32_t>(L / N) <= 32u;
            for (std::size_t i = 0; i < plan.ops.size(); ++i) {
                ok = ok && ((plan.ops[i].opcode == hy::detail::HY_FOP_NBODY_PAIR) == (i >= b0 && i < e0));
            }
            if (!ok) {
                throw std::logic_error("Inconsistent tensor-memory plan");
            }
        }
    }
    const auto warp_bytes = coop_warp_bytes(plan.n_slots, L);
    if (blob_bytes > 24u * 1024u || blob_bytes + warp_bytes + reserve > smem_per_block_max) {
        return false;
    }
    const std::size_t tm_warp_limit = plan.tmem != 0u ? tm_warps_of(N, plan.tmem) : 16u;
    if (threads == 0u) {
        // One CTA per SM holding as many warps as fit (shared memory, tensor-memory columns).
        const std::size_t W = std::min(fit_warps(plan.n_slots, L), tm_warp_limit);
        threads = static_cast<std::uint32_t>(32u * std::max<std::size_t>(W, 1u));
    }
    if (threads % 32u != 0u || threads == 0u || threads > 512u || threads / 32u > tm_warp_limit) {
        throw std::invalid_argument("Invalid number of threads for the cooperative kernel");
    }
    // Registers: 65536 / 512 threads = 128 per thread, 170 with at most 384 threads, 255 with at most 256.
    int kmode = static_cast<int>(plan.tmem); // 0, 2 or 3
    for (const auto &op : plan.ops) {
        kmode = op.opcode < hy::detail::HY_FOP_FIRST ? 1 : kmode;
    }
    // (Not every shape is compiled for every CTA size: fall back to the next larger bound.)
    const int pref_maxt = threads <= 256u ? 256 : (threads <= 384u && kmode >= 2 ? 384 : 512);
    const coop_variant *v = nullptr;
    for (const int m : {256, 384, 512}) {
        if (m >= pref_maxt && v == nullptr) {
            v = find_variant(L, N, m, kmode);
        }
    }
    if (v == nullptr) {
        throw std::invalid_argument("Unsupported cooperative kernel configuration: " + std::to_string(L)
                                    + " lanes per warp, " + std::to_string(N) + " lanes per thread");
    }
    const std::size_t bytes = blob_bytes + static_cast<std::size_t>(threads / 32u) * warp_bytes;
    if (bytes + reserve > smem_per_block_max) {
        return false;
    }
    for (auto fn : {v->step, v->prop}) {
        HY_CUDA_CHECK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bytes)));
    }
    if (ctas_per_sm == 0u) {
        int occ = 0;
        HY_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, v->prop, static_cast<int>(threads), bytes));
        ctas_per_sm = static_cast<std::uint32_t>(std::max(occ, 1));
    }
    if (d_gscratch != nullptr) {
        HY_CUDA_CHECK(cudaFree(d_gscratch));
        d_gscratch = nullptr;
    }
    if (d_cscratch != nullptr) {
        HY_CUDA_CHECK(cudaFree(d_cscratch));
        d_cscratch = nullptr;
    }
    cv = v;
    c_threads = threads;
    c_smem = bytes;
    c_ctas_per_sm = ctas_per_sm;
    const std::uint32_t lanes_per_block = static_cast<std::uint32_t>(L) * (threads / 32u);
    const std::uint32_t n_blocks_needed = (n + lanes_per_block - 1u) / lanes_per_block;
    c_grid = std::max(1u, std::min(n_sms * ctas_per_sm, n_blocks_needed));
    if (plan.n_gslots != 0u) {
        d_gscratch = dalloc<double>(static_cast<std::size_t>(c_grid) * (threads / 32u) * plan.n_gslots
                                    * static_cast<std::size_t>(L));
    }
    d_cscratch = dalloc<double>(static_cast<std::size_t>(c_grid) * (threads / 32u) * (order + 1u) * n_eq
                                * static_cast<std::size_t>(L));
    mode = 2;
    return true;
}

// The cooperative kernel for systems whose compact tape does not fit in shared memory (model::nbody with 32
// bodies: 56k doubles per lane): same program, same planner, but every warp's tape is a slab of global memory and
// the tables are read in place. Unlike the one-thread-per-lane HBM-tape kernel it fills the GPU with a few
// thousand lanes (a warp works on L lanes, its threads on different u variables).
void shard::setup_coop_global(int L, int N, std::uint32_t threads, int cta)
{
    if (plan.tmem != 0u || plan.n_gslots != 0u) {
        replan(false);
    }
    if (N == 0) {
        N = (L == 0 || L >= 2) ? 2 : 1;
    }
    if (threads == 0u) {
        threads = 512u;
    }
    if (threads % 32u != 0u || threads > 512u) {
        throw std::invalid_argument("Invalid number of threads for the cooperative kernel");
    }
    const std::uint32_t warps = threads / 32u;
    if (cta < 0) {
        // Whole CTAs per chunk of lanes (mode 5) when the levels are wide enough to give work to hundreds of
        // threads and there are too few lanes to keep every warp of the GPU busy for long: the lane-step latency
        // drops by the number of warps (a slow lane no longer holds the launch), and the tapes in flight
        // (n_sms x L lanes) nearly fit in L2. Otherwise one warp per chunk (mode 4).
        const double avg_width = static_cast<double>(plan.ops.size()) / std::max(1u, plan.n_segments);
        const std::uint64_t warp_chunks = (n + static_cast<std::uint32_t>(N) - 1u) / static_cast<std::uint32_t>(N);
        cta = (avg_width >= 128. && warp_chunks < 8ull * n_sms * warps) ? 1 : 0;
    }
    if (L == 0) {
        L = N;
        if (cta == 0) {
            // As many lanes per warp as still leave a chunk of lanes for every resident warp.
            while (2 * L <= 8 && n / static_cast<std::uint32_t>(2 * L) >= n_sms * 16u) {
                L *= 2;
            }
        }
    }
    const auto *v = find_variant(L, N, 512, cta != 0 ? 5 : 4);
    if (v == nullptr) {
        throw std::invalid_argument("Unsupported cooperative kernel configuration (global tape): "
                                    + std::to_string(L) + " lanes per warp, " + std::to_string(N)
                                    + " lanes per thread");
    }
    for (double **ptr : {&d_gscratch, &d_cscratch}) {
        if (*ptr != nullptr) {
            HY_CUDA_CHECK(cudaFree(*ptr));
            *ptr = nullptr;
        }
    }
    // Teams (warps, or whole CTAs) per block, each with its own slab and private coefficient store.
    const std::uint32_t teams = cta != 0 ? 1u : warps;
    const std::size_t team_bytes = coop_warp_bytes(plan.n_slots, L);
    const std::uint32_t lanes_per_block = static_cast<std::uint32_t>(L) * teams;
    const std::uint32_t n_blocks_needed = (n + lanes_per_block - 1u) / lanes_per_block;
    std::size_t free_b = 0, total_b = 0;
    HY_CUDA_CHECK(cudaMemGetInfo(&free_b, &total_b));
    const std::size_t max_blocks = std::max<std::size_t>(free_b / 2u / (team_bytes * teams), 1u);
    cv = v;
    c_threads = threads;
    c_smem = 0;
    c_ctas_per_sm = 1;
    c_grid = static_cast<std::uint32_t>(
        std::max<std::size_t>(1u, std::min<std::size_t>({n_sms, n_blocks_needed, max_blocks})));
    d_gscratch = dalloc<double>(static_cast<std::size_t>(c_grid) * teams * (team_bytes / sizeof(double)));
    d_cscratch = dalloc<double>(static_cast<std::size_t>(c_grid) * teams * (order + 1u) * n_eq
                                * static_cast<std::size_t>(L));
    mode = 2;
    c_global = true;
    c_cta = cta != 0;
}

// The table of the one-thread-per-lane N-body kernel (nb1_kernel.cuh) for a plan with ONE pair interaction whose six
// positions each belong to a velocity driven by a single pair output of the same coordinate, or by a number. Returns
// false for anything else (such plans run on k_nb with 32 lanes per warp).
static bool make_nb1_tab(const hy::detail::nb_plan &pl, std::uint32_t n_eq, std::uint32_t order, dev::nb1_tab &tab)
{
    if (!pl.ok || pl.pairs.size() != 1u || pl.sums.size() != 6u || pl.level_offsets.size() != 2u || n_eq != 12u
        || order < 4u) {
        return false;
    }
    const auto &pr = pl.pairs[0];
    bool seen[12] = {};
    std::uint32_t kinds[6];
    for (std::uint32_t s = 0; s < 6u; ++s) {
        const std::uint32_t k = s % 3u, ps = s < 3u ? pr.pa[k] : pr.pb[k];
        const hy::detail::nb_sum_desc *sd = nullptr;
        for (const auto &cand : pl.sums) {
            if (cand.kind != 0u && cand.pos == ps + 1u) {
                if (sd != nullptr) {
                    return false;
                }
                sd = &cand;
            }
        }
        if (sd == nullptr || (sd->out >> 16) == 0u || ps >= pl.pos_sv.size()) {
            return false;
        }
        tab.v_sv[s] = sd->out & 0xffffu;
        tab.x_sv[s] = (sd->out >> 16) - 1u;
        if (tab.x_sv[s] != pl.pos_sv[ps] || tab.v_sv[s] >= 12u || tab.x_sv[s] >= 12u || seen[tab.v_sv[s]]
            || seen[tab.x_sv[s]]) {
            return false;
        }
        seen[tab.v_sv[s]] = seen[tab.x_sv[s]] = true;
        if (tab.v_sv[s] == 0u || tab.x_sv[s] == 0u) {
            tab.sv0_slot = s;
            tab.sv0_is_x = tab.x_sv[s] == 0u ? 1u : 0u;
        }
        if (sd->kind == 2u) {
            // (Only the right-hand side +0: what model::nbody produces for a body that nothing pulls on.)
            if (sd->cidx >= pl.consts.size() || pl.consts[sd->cidx] != 0. || std::signbit(pl.consts[sd->cidx])) {
                return false;
            }
            kinds[s] = 2u;
        } else if (sd->kind == 1u && sd->n_terms == 1u && sd->terms[0] == pr.om[k]) {
            kinds[s] = 0u;
        } else if (sd->kind == 1u && sd->n_terms == 1u && pr.on[k] != 0xffffu && sd->terms[0] == pr.on[k]) {
            kinds[s] = 1u;
        } else {
            return false;
        }
    }
    for (std::uint32_t side = 0; side < 2u; ++side) {
        if (kinds[3u * side] != kinds[3u * side + 1u] || kinds[3u * side] != kinds[3u * side + 2u]) {
            return false;
        }
        tab.kind[side] = kinds[3u * side];
    }
    return true;
}

// The dedicated N-body kernel. LT = lanes per team (0: as many as give every thread of a warp one pair interaction),
// threads = CTA size (0: as many warps as fit; HEYOKA_B200_NB_THREADS caps it), want_tmem / want_cta: -1 automatic.
// Returns false if the program does not qualify or nothing fits.
bool shard::setup_nb(int LT, std::uint32_t threads, int want_tmem, int want_cta, int want_lane)
{
    if (!nbp.ok) {
        return false;
    }
    const std::size_t reserve = 1024u;
    const std::uint32_t n_pairs = static_cast<std::uint32_t>(nbp.pairs.size());
    const std::uint32_t npp = (order + 1u) / 2u;
    const bool cta = want_cta > 0 || (want_cta < 0 && n_pairs > 32u);
    if (!cta && n_pairs > 32u) {
        return false;
    }
    if (LT == 0) {
        LT = 1;
        if (!cta) {
            while (static_cast<std::uint32_t>(2 * LT) * n_pairs <= 32u) {
                LT *= 2;
            }
        }
    }
    if (cta && (LT != 1 || n_pairs > 512u)) {
        return false;
    }
    if (!cta && (LT < 1 || LT > 32 || (LT & (LT - 1)) != 0 || static_cast<std::uint32_t>(LT) * n_pairs > 32u)) {
        return false;
    }
    // One pair interaction, 32 lanes per warp: one thread per lane, nothing exchanged (nb1_kernel.cuh).
    dev::nb1_tab l1{};
    const bool lane = want_lane != 0 && !cta && LT == 32 && make_nb1_tab(nbp, n_eq, order, l1);
    if (want_lane > 0 && !lane) {
        return false;
    }
    const std::uint32_t TT = cta ? 512u : 32u, NL = LT >= 2 ? 2u : 1u;
    // The role records address the outputs in 16-bit units of 16 bytes.
    if (static_cast<std::uint64_t>(nbp.n_out) * LT >= 0xffffu || static_cast<std::uint64_t>(nbp.n_pos) * LT >= 0xffffu) {
        return false;
    }
    auto roles = hy::detail::make_nb_roles(nbp, TT, static_cast<std::uint32_t>(LT), NL);
    if (roles.n_rounds > 32u) {
        return false;
    }
    if (lane) {
        roles = hy::detail::nb_roles{};
    }
    const auto shared_doubles = [&](bool roles_in_smem) {
        std::size_t d = static_cast<std::size_t>(order + 1u) * nbp.fac_stride + ((order + 5u) & ~1u)
                        + ((nbp.consts.size() + 1u) & ~std::size_t(1));
        if (roles_in_smem) {
            d += roles.table.size() * 4u;
        }
        return d;
    };
    const auto team_slots = [&](bool tmem) {
        // (The one-thread-per-lane kernel keeps positions, pair outputs and norms in registers.)
        const std::size_t d = (lane ? 0u : (static_cast<std::size_t>(nbp.n_pos) + nbp.n_out) * LT * 2u)
                              + static_cast<std::size_t>(tmem ? 2u : 5u) * npp * TT * 2u
                              + (3u * hy::detail::nb_norm_copies(static_cast<std::uint32_t>(LT)) + 16u) * LT; // (+ norms, parked bookkeeping)
        return static_cast<std::uint32_t>((d + LT - 1u) / LT);
    };
    // Teams (warps) per CTA that fit: shared memory, tensor-memory columns (12 per order pair and thread).
    struct choice {
        bool tmem = false, roles_in_smem = false;
        std::uint32_t warps = 0;
    };
    const auto fit = [&](bool tmem) {
        choice c;
        c.tmem = tmem;
        for (const bool ris : {true, false}) {
            const std::size_t sh = shared_doubles(ris) * sizeof(double);
            const std::size_t tb = coop_warp_bytes(team_slots(tmem), LT);
            if (sh + tb + reserve > smem_per_block_max) {
                continue;
            }
            std::uint32_t w = cta ? 16u
                                  : static_cast<std::uint32_t>(
                                        std::min<std::size_t>((smem_per_block_max - reserve - sh) / tb, 16u));
            if (tmem) {
                const std::uint32_t cols = npp * 12u;
                const std::uint32_t per_quadrant = cols == 0u || cols > 512u ? 0u : 512u / cols;
                w = std::min(w, 4u * per_quadrant);
            }
            if (cta && w < 16u) {
                w = 0u;
            }
            if (w > c.warps) {
                c.warps = w;
                c.roles_in_smem = ris;
            }
            if (w != 0u) {
                break;
            }
        }
        return c;
    };
    choice pick;
    if (want_tmem != 0 && opt_tmem) {
        pick = fit(true);
    }
    if (want_tmem <= 0) {
        const auto alt = fit(false);
        if (alt.warps > pick.warps) {
            pick = alt;
        }
    }
    if (pick.warps == 0u) {
        return false;
    }
    if (threads == 0u) {
        // Warp teams: 12 warps by default (168 registers per thread: the pair interaction's working set fits without
        // spilling; measured faster than 16 warps of 128 registers and than 8 of 255).
        threads = 32u * (cta ? pick.warps : std::min(pick.warps, 12u));
        if (!cta && opt_nb_threads != 0u) {
            threads = opt_nb_threads;
        }
    }
    if (!cta) {
        threads = std::min(threads, 32u * pick.warps); // (a tuning knob: clamped to what fits)
    }
    if (threads % 32u != 0u || threads == 0u || threads / 32u > pick.warps || (cta && threads != 512u)) {
        throw std::invalid_argument("Invalid number of threads for the N-body kernel");
    }
    const int pref_maxt = threads <= 256u ? 256 : (threads <= 384u ? 384 : 512);
    const hy::detail::nb_variant *v = nullptr;
    for (const int mt : {256, 384, 512}) {
        if (mt >= pref_maxt && v == nullptr) {
            v = find_nb_variant(LT, cta, pick.tmem, mt, lane);
        }
    }
    if (v == nullptr) {
        return false;
    }
    // Device copies of the tables.
    if (d_nb_pairs == nullptr) {
        d_nb_pairs = dupload(nbp.pairs);
        d_nb_consts = dupload(nbp.consts);
        d_nb_fac = dupload(nbp.fac);
    }
    if (d_nb_roles != nullptr) {
        HY_CUDA_CHECK(cudaFree(d_nb_roles));
        d_nb_roles = nullptr;
    }
    d_nb_roles = dupload(roles.table);
    nbd = dev::nb_dev_plan{};
    nbd.pairs = d_nb_pairs;
    nbd.roles = reinterpret_cast<const uint4 *>(d_nb_roles);
    nbd.consts = d_nb_consts;
    nbd.fac = d_nb_fac;
    nbd.n_pairs = n_pairs;
    nbd.n_pos = nbp.n_pos;
    nbd.n_out = nbp.n_out;
    nbd.n_consts = static_cast<std::uint32_t>(nbp.consts.size());
    nbd.npp = npp;
    nbd.fac_stride = nbp.fac_stride;
    nbd.n_rounds = roles.n_rounds;
    nbd.round_level_end = roles.round_level_end;
    nbd.alpha = nbp.alpha;
    nbd.pow_algo = nbp.pow_algo;
    nbd.roles_in_smem = pick.roles_in_smem ? 1u : 0u;
    nbd.shared_doubles = static_cast<std::uint32_t>(shared_doubles(pick.roles_in_smem));
    nbd.n_slots_equiv = team_slots(pick.tmem);
    nbd.l1 = l1;
    nb_lane = lane;
    const std::size_t team_bytes = coop_warp_bytes(nbd.n_slots_equiv, LT);
    nbd.team_doubles = static_cast<std::uint32_t>(team_bytes / sizeof(double));
    const std::uint32_t teams = cta ? 1u : threads / 32u;
    const std::size_t bytes = static_cast<std::size_t>(nbd.shared_doubles) * sizeof(double) + teams * team_bytes;
    for (auto fn : {v->step, v->prop}) {
        HY_CUDA_CHECK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bytes)));
    }
    for (double **ptr : {&d_gscratch, &d_cscratch}) {
        if (*ptr != nullptr) {
            HY_CUDA_CHECK(cudaFree(*ptr));
            *ptr = nullptr;
        }
    }
    nbv = v;
    nb_cv = coop_variant{LT, LT >= 2 ? 2 : 1, v->maxt, cta ? 7 : 6, nullptr, nullptr};
    cv = &nb_cv;
    c_threads = threads;
    c_smem = bytes;
    c_ctas_per_sm = 1;
    const std::uint32_t lanes_per_block = static_cast<std::uint32_t>(LT) * teams;
    const std::uint32_t n_blocks_needed = (n + lanes_per_block - 1u) / lanes_per_block;
    c_grid = std::max(1u, std::min(n_sms, n_blocks_needed));
    d_cscratch = dalloc<double>(static_cast<std::size_t>(c_grid) * teams * (order + 1u) * n_eq
                                * static_cast<std::size_t>(LT));
    mode = 2;
    nb_on = true;
    c_cta = cta;
    return true;
}

// The dense-network kernel: the padded shared-memory image of the weights is prepared here (row pitch = 4 mod 16
// doubles: the 8 x 4 A fragments of the tensor-core products then read conflict-free), copied once per CTA by the TMA
// unit. Returns false if the program is not a network or does not fit in shared memory.
bool shard::setup_nn()
{
    if (!nnp.ok || nnp.layers.size() > static_cast<std::size_t>(dev::NN_MAX_LAYERS)) {
        return false;
    }
    dev::nn_dev_plan d{};
    std::vector<double> img;
    std::uint32_t hist = 0, max_out = 0, n_hidden = 0;
    d.n_layers = static_cast<std::uint32_t>(nnp.layers.size());
    for (std::uint32_t l = 0; l < d.n_layers; ++l) {
        const auto &L = nnp.layers[l];
        d.n_in[l] = L.n_in;
        d.n_out[l] = L.n_out;
        d.act[l] = static_cast<std::uint32_t>(L.act);
        d.n_in_pad[l] = (L.n_in + 3u) & ~3u;
        d.n_out_pad[l] = (L.n_out + 7u) & ~7u;
        std::uint32_t ldw = d.n_in_pad[l];
        while (ldw % 16u != 4u) {
            ++ldw;
        }
        d.ldw[l] = ldw;
        d.w_off[l] = static_cast<std::uint32_t>(img.size());
        img.resize(img.size() + static_cast<std::size_t>(d.n_out_pad[l]) * ldw, 0.);
        for (std::uint32_t r = 0; r < L.n_out; ++r) {
            for (std::uint32_t c = 0; c < L.n_in; ++c) {
                img[d.w_off[l] + static_cast<std::size_t>(r) * ldw + c] = L.w[static_cast<std::size_t>(r) * L.n_in + c];
            }
        }
        d.b_off[l] = static_cast<std::uint32_t>(img.size());
        img.insert(img.end(), L.bias.begin(), L.bias.end());
        img.resize((img.size() + 1u) & ~std::size_t(1), 0.);
        d.hist_off[l] = hist;
        if (L.act != 0) {
            hist += 2u * order * L.n_out * dev::NN_LB; // z and the activation (its square lives in tensor memory)
            d.tm_slot[l] = n_hidden++;
            d.tm_ipt = std::max(d.tm_ipt, (L.n_out * dev::NN_LB + dev::NN_THREADS - 1u) / dev::NN_THREADS);
        }
        max_out = std::max(max_out, L.n_out);
    }
    // Tensor memory: 48 columns per (neuron, lane) item and hidden layer (16 of padding + 2 per order), 256 columns per
    // thread, orders up to 16 (the history is read back in two windows of eight orders).
    if (n_hidden * d.tm_ipt * 48u > 256u || order > 16u) {
        return false;
    }
    d.wimg_doubles = static_cast<std::uint32_t>(img.size());
    d.hist_doubles = hist;
    d.max_out = max_out;
    const std::size_t doubles = img.size() + hist + static_cast<std::size_t>(order + 1u) * n_eq * dev::NN_LB
                                + static_cast<std::size_t>(max_out) * dev::NN_LB + dev::NN_LB + 4u;
    const std::size_t bytes = doubles * sizeof(double);
    if (bytes + 2048u > smem_per_block_max) {
        return false;
    }
    for (void **ptr : {reinterpret_cast<void **>(&d_nn_wimg), reinterpret_cast<void **>(&d_nn_out)}) {
        if (*ptr != nullptr) {
            HY_CUDA_CHECK(cudaFree(*ptr));
            *ptr = nullptr;
        }
    }
    d_nn_wimg = dupload(img);
    d_nn_out = dupload(nnp.out_of_sv);
    d.wimg = d_nn_wimg;
    d.out_of_sv = d_nn_out;
    nnd = d;
    for (auto fn : {hy::detail::nn_kernel_step(), hy::detail::nn_kernel_prop()}) {
        HY_CUDA_CHECK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bytes)));
    }
    for (double **ptr : {&d_gscratch, &d_cscratch}) {
        if (*ptr != nullptr) {
            HY_CUDA_CHECK(cudaFree(*ptr));
            *ptr = nullptr;
        }
    }
    nb_cv = coop_variant{dev::NN_LB, 1, dev::NN_THREADS, 8, nullptr, nullptr};
    cv = &nb_cv;
    c_threads = dev::NN_THREADS;
    c_smem = bytes;
    c_ctas_per_sm = 1;
    const std::uint32_t n_blocks_needed = (n + dev::NN_LB - 1u) / dev::NN_LB;
    c_grid = std::max(1u, std::min(n_sms, n_blocks_needed));
    mode = 2;
    nn_on = true;
    return true;
}

void shard::configure(int want_mode, int L, int N, std::uint32_t threads, std::uint32_t blocks_per_sm)
{
    c_global = false;
    c_cta = false;
    nb_on = false;
    nb_lane = false;
    nn_on = false;
    // Mode 8: the dense-network kernel (right-hand sides that are feed-forward networks, nn_plan.hpp); the automatic
    // mode takes it whenever the program qualifies.
    if (want_mode == 8 || (want_mode == 0 && opt_nn != 0)) {
        if (setup_nn()) {
            return;
        }
        if (want_mode == 8) {
            throw std::invalid_argument("The dense-network kernel cannot run this program: "
                                        + (nnp.ok ? std::string("it does not fit in shared memory") : nnp.why));
        }
    }
    // Mode 6 / 7: the N-body kernel with warp / CTA teams (N: 0 automatic, 1 tensor memory, 2 shared memory only).
    // Automatic mode takes it whenever the program qualifies (nb_plan.hpp).
    if (want_mode == 6 || want_mode == 7 || want_mode == 9 || (want_mode == 0 && opt_nb != 0)) {
        // Mode 9: one thread per lane (systems with one pair interaction); the automatic mode takes it when it applies,
        // an explicit mode 6 never does (it selects k_nb with the given team shape).
        const int want_lane = want_mode == 9 ? 1 : (want_mode == 0 ? (opt_nb_lane != 0 ? -1 : 0) : 0);
        if (setup_nb(want_mode == 9 ? 32 : L, threads, N == 0 ? -1 : (N == 1 ? 1 : 0),
                     want_mode == 0 ? -1 : (want_mode == 7 ? 1 : 0), want_lane)) {
            return;
        }
        if (want_mode != 0) {
            throw std::invalid_argument("The N-body kernel cannot run this program: "
                                        + (nbp.ok ? std::string("no configuration fits on an SM") : nbp.why));
        }
    }
    if (want_mode == 4 || want_mode == 5) {
        setup_coop_global(L, N, threads, want_mode == 5 ? 1 : 0);
        return;
    }
    if (want_mode == 1) {
        setup_hbm(threads, blocks_per_sm);
        return;
    }
    allow_tmem = want_mode != 3;
    if (want_mode == 3) {
        want_mode = 2;
    }
    if (setup_coop(L, N, threads, blocks_per_sm)) {
        return;
    }
    if (want_mode == 2) {
        throw std::invalid_argument("The derivative tape of this system (" + std::to_string(plan.n_slots)
                                    + " doubles per lane) does not fit in shared memory");
    }
    // Automatic: the cooperative kernel with the tape in global memory.
    setup_coop_global(0, 0, 0);
}

// The public Taylor-coefficient array, [n_eq][order + 1][batch] (src/taylor_00.cpp:574-580), is allocated the first
// time something needs it (write_tc, dense output, hy_batch_get_ptrs()): 6-body, 2^20 lanes: 6.3 GB; the
// cooperative kernels keep the coefficients of the current step in a private per-warp store otherwise.
void shard::ensure_tc()
{
    if (d_tc == nullptr) {
        // (With events, the rows of the event equations follow those of the state variables.)
        const std::size_t sz = static_cast<std::size_t>(n_eq + n_ev) * (order + 1u) * n;
        d_tc = dalloc<double>(sz);
        HY_CUDA_CHECK(cudaMemsetAsync(d_tc, 0, sizeof(double) * sz, stream));
    }
}

// ---- Event detection (ev_kernels.cuh) ----
void shard::ev_setup(std::uint32_t n_te, const std::int32_t *dirs, const double *cooldowns, double tol)
{
    if (n_ev == 0u) {
        throw std::invalid_argument("This batch was built from a program without event equations");
    }
    if (n_te > n_ev) {
        throw std::invalid_argument("The number of terminal events exceeds the number of event equations");
    }
    for (std::uint32_t k = 0; k < n_ev; ++k) {
        if (dirs[k] < -1 || dirs[k] > 1) {
            throw std::invalid_argument("Invalid value selected for the direction of an event");
        }
    }
    for (std::uint32_t k = 0; k < n_te; ++k) {
        if (!std::isfinite(cooldowns[k])) {
            throw std::invalid_argument("Cannot set a non-finite cooldown value for a terminal event");
        }
    }
    for (void *q : ev_allocs) {
        HY_CUDA_CHECK(cudaFree(q));
    }
    ev_allocs.clear();
    const auto keep = [this](auto *q) {
        ev_allocs.push_back(static_cast<void *>(q));
        return q;
    };
    const std::uint32_t p = order, pp1 = p + 1u;
    dev::ev_args E{};
    E.n_ev = n_ev;
    E.n_te = n_te;
    E.tol = tol;
    E.max_svf = *std::max_element(prog_host->ev_defs.begin(), prog_host->ev_defs.end());
    E.ev_defs = keep(dupload(prog_host->ev_defs));
    E.dirs = keep(dupload(std::vector<int>(dirs, dirs + n_ev)));
    E.cooldowns = keep(dupload(std::vector<double>(cooldowns, cooldowns + n_te)));
    // Binomial coefficients, exact in double precision for the orders in use (src/detail/llvm_helpers_ed.cpp:421-455).
    std::vector<double> bc(static_cast<std::size_t>(pp1) * pp1, 0.);
    for (std::uint32_t i = 0; i <= p; ++i) {
        bc[i * pp1] = 1.;
        for (std::uint32_t j = 1; j <= i; ++j) {
            bc[i * pp1 + j] = bc[(i - 1u) * pp1 + j - 1u] + (j < i ? bc[(i - 1u) * pp1 + j] : 0.);
        }
    }
    E.bc = keep(dupload(bc));
    const std::size_t B = n;
    E.h = keep(dalloc<double>(B));
    E.mdt = keep(dalloc<double>(B));
    E.g_eps = keep(dalloc<double>(B));
    E.cd = keep(dalloc<double>(B * 2u * std::max(n_te, 1u)));
    E.cd_on = keep(dalloc<unsigned char>(B * std::max(n_te, 1u)));
    HY_CUDA_CHECK(cudaMemset(E.cd_on, 0, B * std::max(n_te, 1u)));
    // (hy_batch_get_cooldowns() reports every lane, also those that have not been in a cooldown yet.)
    HY_CUDA_CHECK(cudaMemset(E.cd, 0, sizeof(double) * B * 2u * std::max(n_te, 1u)));
    E.cand = keep(dalloc<std::uint32_t>(B * n_ev));
    E.counters = keep(dalloc<unsigned>(4));
    E.rec_cap = static_cast<std::uint32_t>(std::min<std::size_t>(std::max<std::size_t>(B * n_ev, 1024u), 1u << 26));
    E.rec = keep(dalloc<dev::ev_rec>(E.rec_cap));
    E.te_key = keep(dalloc<unsigned long long>(B));
    E.te_sel = keep(dalloc<unsigned long long>(B));
    // One bisection stack per detecting thread: a fraction of the lanes ever needs one at the same time.
    E.arena_threads = 64u * std::min<std::uint32_t>(n_sms, static_cast<std::uint32_t>((B * n_ev + 63u) / 64u));
    E.arena = keep(dalloc<double>(static_cast<std::size_t>(dev::EV_STACK) * (pp1 + 2u) * E.arena_threads));
    eva = E;
    ev_host.clear();
}

void shard::ev_step(const double *d_mdt, int backward)
{
    if (mode != 1 || d_scratch == nullptr) {
        setup_hbm(0, 0);
    }
    ensure_tc();
    const std::uint32_t B = n;
    dev::run_args R{};
    R.max_delta_t = d_mdt;
    R.default_max_delta_t = backward ? -std::numeric_limits<double>::infinity() : std::numeric_limits<double>::infinity();
    R.counter = d_counter;
    R.flags = d_flags;
    HY_CUDA_CHECK(cudaMemsetAsync(d_counter, 0, sizeof(unsigned int), stream));
    dev::k_ev_jet<<<h_grid, h_threads, 0, stream>>>(prog, view(), R, eva, d_scratch, slab_doubles);
    HY_CUDA_CHECK(cudaGetLastError());
    n_launches += 1;
    unsigned counters[4] = {0u, 0u, 0u, 0u};
    for (;;) {
        HY_CUDA_CHECK(cudaMemsetAsync(eva.counters, 0, 4u * sizeof(unsigned), stream));
        const std::size_t n_pairs = static_cast<std::size_t>(n_ev) * B;
        dev::k_ev_fex<<<static_cast<unsigned>((n_pairs + 255u) / 256u), 256, 0, stream>>>(prog, view(), eva);
        dev::k_ev_detect<<<eva.arena_threads / 64u, 64, 0, stream>>>(prog, view(), eva);
        HY_CUDA_CHECK(cudaGetLastError());
        n_launches += 2;
        HY_CUDA_CHECK(cudaMemcpyAsync(counters, eva.counters, sizeof(counters), cudaMemcpyDeviceToHost, stream));
        HY_CUDA_CHECK(cudaStreamSynchronize(stream));
        if (counters[1] <= eva.rec_cap) {
            break;
        }
        // More events than record slots (never seen in practice: one slot per (event, lane) pair): grow and redo the
        // detection, which only reads the jet.
        const std::uint32_t new_cap = counters[1] + counters[1] / 2u;
        dev::ev_rec *nr = dalloc<dev::ev_rec>(new_cap);
        for (auto &q : ev_allocs) {
            if (q == static_cast<void *>(eva.rec)) {
                q = nr;
            }
        }
        HY_CUDA_CHECK(cudaFree(eva.rec));
        eva.rec = nr;
        eva.rec_cap = new_cap;
        HY_CUDA_CHECK(cudaMemsetAsync(eva.te_key, 0xff, sizeof(unsigned long long) * B, stream));
    }
    const unsigned n_rec = counters[1];
    if (n_rec != 0u) {
        dev::k_ev_first<<<(n_rec + 127u) / 128u, 128, 0, stream>>>(view(), eva);
        ++n_launches;
    }
    dev::k_ev_apply<<<(B + 127u) / 128u, 128, 0, stream>>>(prog, view(), eva);
    ++n_launches;
    ev_host.clear();
    if (n_rec != 0u) {
        dev::k_ev_filter<<<(n_rec + 127u) / 128u, 128, 0, stream>>>(view(), eva);
        ++n_launches;
        std::vector<dev::ev_rec> recs(n_rec);
        HY_CUDA_CHECK(cudaMemcpyAsync(recs.data(), eva.rec, sizeof(dev::ev_rec) * n_rec, cudaMemcpyDeviceToHost, stream));
        HY_CUDA_CHECK(cudaStreamSynchronize(stream));
        for (const auto &r : recs) {
            if (r.live != 0u) {
                ev_host.push_back(hy_event_rec{r.lane, r.idx, r.terminal, r.d_sgn, r.t, r.abs_der});
            }
        }
        // Per lane: the non-terminal events in time order (src/taylor_adaptive_batch.cpp:789-790: by |t|; equal times
        // keep the order of the event indices), then the terminal event.
        std::sort(ev_host.begin(), ev_host.end(), [](const hy_event_rec &a, const hy_event_rec &b) {
            if (a.lane != b.lane) {
                return a.lane < b.lane;
            }
            if (a.terminal != b.terminal) {
                return a.terminal < b.terminal;
            }
            if (std::abs(a.t) != std::abs(b.t)) {
                return std::abs(a.t) < std::abs(b.t);
            }
            return a.idx < b.idx;
        });
    }
    HY_CUDA_CHECK(cudaGetLastError());
}

void shard::launch(bool prop, const dev::run_args &R)
{
    if (R.write_tc != 0 || (mode == 2 && d_cscratch == nullptr && !nn_on)) {
        ensure_tc();
    }
    HY_CUDA_CHECK(cudaMemsetAsync(d_counter, 0, sizeof(unsigned int), stream));
    if (nn_on) {
        (prop ? hy::detail::nn_kernel_prop() : hy::detail::nn_kernel_step())<<<c_grid, c_threads, c_smem, stream>>>(
            prog, nnd, view(), R);
    } else if (mode == 2) {
        dev::run_args R2 = R;
        const bool pub = R.write_tc != 0 || d_cscratch == nullptr;
        const auto lanes = static_cast<unsigned long long>(cv->L);
        R2.coef_pub = pub ? 1 : 0;
        R2.coef_base = pub ? d_tc : d_cscratch;
        R2.coef_warp_stride = pub ? 0ull : static_cast<unsigned long long>(order + 1u) * n_eq * lanes;
        R2.coef_stride_sv = pub ? static_cast<unsigned long long>(order + 1u) * n : lanes;
        R2.coef_stride_o = pub ? static_cast<unsigned long long>(n) : static_cast<unsigned long long>(n_eq) * lanes;
        if (nb_on && nb_lane) {
            // k_nb1 always works on its private store ([order][slot][32 lanes], velocities only) and publishes the
            // coefficients to tc on request.
            R2.coef_base = d_cscratch;
            R2.coef_warp_stride = static_cast<unsigned long long>(order + 1u) * n_eq * lanes;
            R2.coef_pub = R.write_tc != 0 ? 1 : 0;
        }
        if (nb_on) {
            (prop ? nbv->prop : nbv->step)<<<c_grid, c_threads, c_smem, stream>>>(prog, nbd, view(), R2);
        } else {
            (prop ? cv->prop : cv->step)<<<c_grid, c_threads, c_smem, stream>>>(prog, d_blob, view(), R2, d_gscratch);
        }
    } else if (prop) {
        dev::k_hbm<true><<<h_grid, h_threads, 0, stream>>>(prog, view(), R, d_scratch, slab_doubles);
    } else {
        dev::k_hbm<false><<<h_grid, h_threads, 0, stream>>>(prog, view(), R, d_scratch, slab_doubles);
    }
    HY_CUDA_CHECK(cudaGetLastError());
    ++n_launches;
}

namespace
{

struct device_guard {
    int prev = 0;
    explicit device_guard(int dev)
    {
        HY_CUDA_CHECK(cudaGetDevice(&prev));
        if (prev != dev) {
            HY_CUDA_CHECK(cudaSetDevice(dev));
        }
    }
    ~device_guard()
    {
        cudaSetDevice(prev);
    }
};

// Stage the shard's lanes [off, off + n) of a host array of doubles into slot `slot` of d_tmp; returns the device
// pointer (null for a null array).
const double *stage(shard &sh, const double *src, std::size_t off, std::uint32_t slot)
{
    if (src == nullptr) {
        return nullptr;
    }
    double *dst = sh.d_tmp + static_cast<std::size_t>(slot) * sh.n;
    HY_CUDA_CHECK(cudaMemcpyAsync(dst, src + off, sizeof(double) * sh.n, cudaMemcpyHostToDevice, sh.stream));
    return dst;
}

// propagate_until() on one shard, in three phases so that a batch of several shards can apply the reference's
// GLOBAL exits across them (propagate()):
//   phase 1  snapshot of (state, time), one launch of the propagate kernel, flags read back (synchronises);
//   replay   if a lane of ANY shard went non-finite: restore the snapshot and re-run with the iteration count capped at
//            the first such iteration (the reference stops EVERY lane there, src/taylor_adaptive_batch.cpp:1462-1467;
//            lanes are independent, so the capped re-run reproduces it exactly);
//   finish   iteration limit -> every lane reports step_limit (:1516-1526); the lanes that were done before the loop's
//            last iteration K took zero-length steps in the reference: last_h = 0 and, with write_tc, Taylor
//            coefficients re-expanded about the final state (one masked zero-length step).
struct prop_ctx {
    dev::run_args R{};
    dev::run_flags fl{};
};

void propagate_phase1(shard &sh, const double *d_tf_hi, const double *d_tf_lo, const double *d_mdt, uint64_t max_steps,
                      int write_tc, prop_ctx &c)
{
    const std::size_t state_doubles = static_cast<std::size_t>(sh.n_eq) * sh.n;
    HY_CUDA_CHECK(cudaMemcpyAsync(sh.d_snapshot, sh.d_state, sizeof(double) * state_doubles, cudaMemcpyDeviceToDevice,
                                  sh.stream));
    HY_CUDA_CHECK(cudaMemcpyAsync(sh.d_snapshot + state_doubles, sh.d_t_hi, sizeof(double) * sh.n,
                                  cudaMemcpyDeviceToDevice, sh.stream));
    HY_CUDA_CHECK(cudaMemcpyAsync(sh.d_snapshot + state_doubles + sh.n, sh.d_t_lo, sizeof(double) * sh.n,
                                  cudaMemcpyDeviceToDevice, sh.stream));
    const dev::run_flags init{0u, 0u, ~0ull, 0ull};
    HY_CUDA_CHECK(cudaMemcpyAsync(sh.d_flags, &init, sizeof(init), cudaMemcpyHostToDevice, sh.stream));
    c.R = dev::run_args{};
    c.R.max_delta_t = d_mdt;
    c.R.tf_hi = d_tf_hi;
    c.R.tf_lo = d_tf_lo;
    c.R.iter_cap = max_steps;
    c.R.replay = 0;
    c.R.write_tc = write_tc;
    c.R.flags = sh.d_flags;
    c.R.counter = sh.d_counter;
    sh.launch(true, c.R);
    HY_CUDA_CHECK(cudaMemcpyAsync(&c.fl, sh.d_flags, sizeof(c.fl), cudaMemcpyDeviceToHost, sh.stream));
    HY_CUDA_CHECK(cudaStreamSynchronize(sh.stream));
}

void propagate_replay(shard &sh, prop_ctx &c, unsigned long long cap)
{
    const std::size_t state_doubles = static_cast<std::size_t>(sh.n_eq) * sh.n;
    HY_CUDA_CHECK(cudaMemcpyAsync(sh.d_state, sh.d_snapshot, sizeof(double) * state_doubles, cudaMemcpyDeviceToDevice,
                                  sh.stream));
    HY_CUDA_CHECK(cudaMemcpyAsync(sh.d_t_hi, sh.d_snapshot + state_doubles, sizeof(double) * sh.n,
                                  cudaMemcpyDeviceToDevice, sh.stream));
    HY_CUDA_CHECK(cudaMemcpyAsync(sh.d_t_lo, sh.d_snapshot + state_doubles + sh.n, sizeof(double) * sh.n,
                                  cudaMemcpyDeviceToDevice, sh.stream));
    const dev::run_flags init{0u, 0u, ~0ull, 0ull};
    HY_CUDA_CHECK(cudaMemcpyAsync(sh.d_flags, &init, sizeof(init), cudaMemcpyHostToDevice, sh.stream));
    c.R.iter_cap = cap;
    c.R.replay = 1;
    sh.launch(true, c.R);
    HY_CUDA_CHECK(cudaMemcpyAsync(&c.fl, sh.d_flags, sizeof(c.fl), cudaMemcpyDeviceToHost, sh.stream));
    HY_CUDA_CHECK(cudaStreamSynchronize(sh.stream));
}

void propagate_finish(shard &sh, bool any_nf, bool any_limit, unsigned long long loop_len, int write_tc)
{
    const std::uint32_t gb = (sh.n + 255u) / 256u;
    if (!any_nf && any_limit) {
        dev::k_fill_outcome<<<gb, 256, 0, sh.stream>>>(sh.d_prop_outcome, sh.n, HY_OUTCOME_STEP_LIMIT);
        HY_CUDA_CHECK(cudaGetLastError());
        ++sh.n_launches;
    }
    // Lanes that were done before the last iteration of the reference's loop.
    unsigned *d_any = reinterpret_cast<unsigned *>(sh.d_flags) + sizeof(dev::run_flags) / sizeof(unsigned);
    HY_CUDA_CHECK(cudaMemsetAsync(d_any, 0, sizeof(unsigned), sh.stream));
    dev::k_prop_early<<<gb, 256, 0, sh.stream>>>(sh.d_prop_iters, loop_len, sh.n, sh.d_last_h, sh.d_skip, sh.d_tmp, d_any);
    HY_CUDA_CHECK(cudaGetLastError());
    ++sh.n_launches;
    if (write_tc != 0) {
        unsigned any = 0;
        HY_CUDA_CHECK(cudaMemcpyAsync(&any, d_any, sizeof(any), cudaMemcpyDeviceToHost, sh.stream));
        HY_CUDA_CHECK(cudaStreamSynchronize(sh.stream));
        if (any != 0u) {
            dev::run_args R{};
            R.max_delta_t = sh.d_tmp; // zeros
            R.write_tc = 1;
            R.flags = sh.d_flags;
            R.counter = sh.d_counter;
            R.skip = sh.d_skip;
            sh.launch(false, R);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// The lanes are independent ODE systems, so a batch shards over the GPUs of a box with no data-path communication
// (src/ensemble_propagate.cpp:192-311 partitions its members over TBB threads the same way). Every entry point is one
// loop over the shards; with several shards each runs on its own host thread. Host arrays are batch-innermost
// ([row][batch]), so a shard's slice of a row is contiguous and the copies of a shard that is not the whole batch are
// pitched 2D copies. The only coupling is the reference's GLOBAL exits of propagate_until() (non-finite state
// anywhere, iteration limit, length of the lock-step loop), applied across the shards between the phases of
// propagate().
// ------------------------------------------------------------------------------------------------

// fn(shard, lane offset, shard index) for every shard in order, on the calling thread.
template <typename F>
void each_shard_in_order(hy_batch *b, F &&fn)
{
    for (std::size_t i = 0; i < b->shards.size(); ++i) {
        device_guard guard(b->shards[i]->device);
        fn(*b->shards[i], static_cast<std::size_t>(b->shard_off[i]), i);
    }
}

// Idem, one host thread per shard when there are several; the error of the first failing shard is rethrown.
template <typename F>
void for_each_shard(hy_batch *b, F &&fn)
{
    const std::size_t ns = b->shards.size();
    if (ns == 1u) {
        each_shard_in_order(b, fn);
        return;
    }
    std::vector<std::exception_ptr> errs(ns);
    std::vector<std::thread> thr;
    thr.reserve(ns);
    for (std::size_t i = 0; i < ns; ++i) {
        thr.emplace_back([&, i] {
            try {
                device_guard guard(b->shards[i]->device);
                fn(*b->shards[i], static_cast<std::size_t>(b->shard_off[i]), i);
            } catch (...) {
                errs[i] = std::current_exception();
            }
        });
    }
    for (auto &t : thr) {
        t.join();
    }
    for (const auto &e : errs) {
        if (e) {
            std::rethrow_exception(e);
        }
    }
}

// rows x (shard lanes) block of a host array with `pitch` elements per row, starting at column `off` (1D if pitch == n).
template <typename T>
void rows_h2d(shard &sh, T *dst, const T *src, std::size_t rows, std::size_t pitch, std::size_t off)
{
    if (src == nullptr || rows == 0u) {
        return;
    }
    if (pitch == sh.n) {
        HY_CUDA_CHECK(cudaMemcpyAsync(dst, src, sizeof(T) * rows * pitch, cudaMemcpyHostToDevice, sh.stream));
    } else {
        HY_CUDA_CHECK(cudaMemcpy2DAsync(dst, sizeof(T) * sh.n, src + off, sizeof(T) * pitch, sizeof(T) * sh.n, rows,
                                        cudaMemcpyHostToDevice, sh.stream));
    }
}
template <typename T>
void rows_d2h(shard &sh, T *dst, const T *src, std::size_t rows, std::size_t pitch, std::size_t off)
{
    if (dst == nullptr || rows == 0u) {
        return;
    }
    if (pitch == sh.n) {
        HY_CUDA_CHECK(cudaMemcpyAsync(dst, src, sizeof(T) * rows * pitch, cudaMemcpyDeviceToHost, sh.stream));
    } else {
        HY_CUDA_CHECK(cudaMemcpy2DAsync(dst + off, sizeof(T) * pitch, src, sizeof(T) * sh.n, sizeof(T) * sh.n, rows,
                                        cudaMemcpyDeviceToHost, sh.stream));
    }
}

// propagate_until() of the whole batch. The final times and step limits are host arrays of the whole batch, or, with
// on_device, device arrays (a batch of one shard). any_flag (optional): 1 = a lane went non-finite, 2 = iteration limit.
int propagate(hy_batch *b, const double *tf_hi, const double *tf_lo, const double *mdt, int on_device,
              uint64_t max_steps, int write_tc, int *any_flag)
{
    std::vector<prop_ctx> ctx(b->shards.size());
    for_each_shard(b, [&](shard &sh, std::size_t off, std::size_t i) {
        const double *d_hi = on_device ? tf_hi : stage(sh, tf_hi, off, 0);
        const double *d_lo = on_device ? tf_lo : stage(sh, tf_lo, off, 1);
        const double *d_mdt = on_device ? mdt : stage(sh, mdt, off, 2);
        propagate_phase1(sh, d_hi, d_lo, d_mdt, max_steps, write_tc, ctx[i]);
    });
    bool any_nf = false;
    unsigned long long cap = ~0ull;
    for (const auto &c : ctx) {
        if (c.fl.any_nf != 0u) {
            any_nf = true;
            cap = std::min(cap, c.fl.min_nf_iter);
        }
    }
    if (any_nf) {
        // Every lane of every shard stops at the first iteration in which any lane went non-finite.
        for_each_shard(b, [&](shard &sh, std::size_t, std::size_t i) { propagate_replay(sh, ctx[i], cap); });
    }
    bool any_limit = false;
    unsigned long long loop_len = 0;
    for (const auto &c : ctx) {
        any_limit = any_limit || c.fl.any_limit != 0u;
        loop_len = std::max(loop_len, c.fl.max_iter);
    }
    for_each_shard(b, [&](shard &sh, std::size_t, std::size_t) {
        propagate_finish(sh, any_nf, any_limit, loop_len, write_tc);
    });
    if (any_flag != nullptr) {
        *any_flag = (any_nf ? 1 : 0) | (any_limit ? 2 : 0);
    }
    return HY_OK;
}

// The set-up of one shard: `lanes` lanes of program p on `device` (-1: the current device).
std::unique_ptr<shard> make_shard(const hy_program *p, std::uint32_t lanes, int device, int n_dev)
{
    if (device < 0) {
        HY_CUDA_CHECK(cudaGetDevice(&device));
    }
    if (device >= n_dev) {
        throw std::invalid_argument("Invalid CUDA device index " + std::to_string(device));
    }

    // Overflow checks on the buffer sizes, like src/taylor_adaptive_batch.cpp:256-264,375-378.
    const std::uint64_t tc_size = static_cast<std::uint64_t>(p->n_eq) * (p->order + 1u) * lanes;
    if (tc_size > (std::numeric_limits<std::uint64_t>::max() >> 4)) {
        throw std::overflow_error("Overflow detected while computing the size of the Taylor coefficients buffer");
    }

    auto sh = std::make_unique<shard>();
    sh->device = device;
    device_guard guard(device);

    sh->n = lanes;
    sh->n_eq = p->n_eq;
    sh->n_pars = p->n_pars;
    sh->order = p->order;
    sh->n_uvars = p->n_uvars;
    sh->high_accuracy = p->high_accuracy;

    cudaDeviceProp prop{};
    HY_CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
    sh->n_sms = static_cast<std::uint32_t>(prop.multiProcessorCount);
    sh->smem_per_block_max = prop.sharedMemPerBlockOptin;
    sh->smem_per_sm = prop.sharedMemPerMultiprocessor;

    // Program arrays, "hbm" encoding.
    static_assert(sizeof(hy_op) == sizeof(uint4), "hy_op must be 16 bytes");
    sh->d_ops = reinterpret_cast<uint4 *>(sh->dupload(p->ops));
    sh->d_args = sh->dupload(p->args);
    sh->d_consts = sh->dupload(p->consts);
    sh->d_sv_defs = sh->dupload(p->sv_defs);

    auto &P = sh->prog;
    P.n_eq = p->n_eq;
    P.n_uvars = p->n_uvars;
    P.n_pars = p->n_pars;
    P.order = p->order;
    P.n_ops = p->n_uvars - p->n_eq;
    P.high_accuracy = p->high_accuracy ? 1 : 0;
    // taylor_determine_h_rhofac(), src/taylor_00.cpp:84-94 (host libm, like the reference's number arithmetic).
    P.rhofac = std::exp((-7. / 10.) / static_cast<double>(p->order - 1u)) / (std::exp(1.) * std::exp(1.));
    P.inv_p = 1. / static_cast<double>(p->order);
    P.inv_pm1 = 1. / static_cast<double>(p->order - 1u);
    P.ops = sh->d_ops;
    P.args = sh->d_args;
    P.consts = sh->d_consts;
    P.sv_defs = sh->d_sv_defs;

    // Cooperative plan.
    // HEYOKA_B200_FUSE=0 disables the superinstructions, HEYOKA_B200_FUSE_SV=0 the fused state-variable
    // propagation, HEYOKA_B200_SPILL=0/1 forces the overflow tape off/on, HEYOKA_B200_TMEM=0 keeps every
    // row in shared memory (diagnostics / tests).
    if (const char *env = std::getenv("HEYOKA_B200_FUSE")) {
        sh->opt_fuse = std::string{env} != "0";
    }
    if (const char *env = std::getenv("HEYOKA_B200_FUSE_SV")) {
        sh->opt_fuse_sv = std::string{env} != "0";
    }
    if (const char *env = std::getenv("HEYOKA_B200_SPILL")) {
        sh->opt_spill = std::string{env} != "0" ? 1 : 0;
    }
    if (const char *env = std::getenv("HEYOKA_B200_TMEM")) {
        sh->opt_tmem = std::string{env} != "0";
    }
    if (const char *env = std::getenv("HEYOKA_B200_TMEM_ROWS")) {
        sh->opt_tmem_rows = std::string{env} == "3" ? 3u : (std::string{env} == "2" ? 2u : 0u);
    }
    if (const char *env = std::getenv("HEYOKA_B200_NB")) {
        sh->opt_nb = std::string{env} != "0" ? 1 : 0;
    }
    if (const char *env = std::getenv("HEYOKA_B200_NB_LANE")) {
        sh->opt_nb_lane = std::string{env} != "0" ? 1 : 0;
    }
    if (const char *env = std::getenv("HEYOKA_B200_NB_THREADS")) {
        sh->opt_nb_threads = static_cast<std::uint32_t>(std::atoi(env));
    }
    sh->prog_host = std::make_shared<const hy_program>(*p);
    sh->replan(false);
    sh->nbp = hy::detail::make_nb_plan(*p);
    if (const char *env = std::getenv("HEYOKA_B200_NN")) {
        sh->opt_nn = std::string{env} != "0" ? 1 : 0;
    }
    sh->nnp = hy::detail::make_nn_plan(*p);

    // Resident arrays.
    const std::size_t n = lanes;
    sh->d_state = sh->dalloc<double>(n * p->n_eq);
    sh->d_pars = sh->dalloc<double>(n * p->n_pars);
    sh->d_t_hi = sh->dalloc<double>(n);
    sh->d_t_lo = sh->dalloc<double>(n);
    sh->d_last_h = sh->dalloc<double>(n);
    sh->d_d_out = sh->dalloc<double>(n * p->n_eq);
    sh->d_step_outcome = sh->dalloc<long long>(n);
    sh->d_prop_outcome = sh->dalloc<long long>(n);
    sh->d_prop_min_h = sh->dalloc<double>(n);
    sh->d_prop_max_h = sh->dalloc<double>(n);
    sh->d_prop_n_steps = sh->dalloc<unsigned long long>(n);
    sh->d_prop_iters = sh->dalloc<unsigned long long>(n);
    sh->d_skip = sh->dalloc<unsigned char>(n);
    sh->d_tmp = sh->dalloc<double>(3u * n);
    sh->d_snapshot = sh->dalloc<double>(n * (p->n_eq + 2u));
    sh->d_counter = sh->dalloc<unsigned int>(1);
    sh->d_flags = sh->dalloc<dev::run_flags>(2); // (+ scratch words behind the flags)

    HY_CUDA_CHECK(cudaMemset(sh->d_state, 0, sizeof(double) * n * p->n_eq));
    HY_CUDA_CHECK(cudaMemset(sh->d_pars, 0, sizeof(double) * std::max<std::size_t>(n * p->n_pars, 1u)));
    HY_CUDA_CHECK(cudaMemset(sh->d_t_hi, 0, sizeof(double) * n));
    HY_CUDA_CHECK(cudaMemset(sh->d_t_lo, 0, sizeof(double) * n));
    HY_CUDA_CHECK(cudaMemset(sh->d_last_h, 0, sizeof(double) * n));

    // Kernel selection: HEYOKA_B200_TAPE = hbm | smem overrides the automatic choice.
    int want = 0;
    if (const char *env = std::getenv("HEYOKA_B200_TAPE")) {
        const std::string s{env};
        want = s == "hbm" ? 1 : (s == "smem" ? 2 : 0);
    }
    sh->n_ev = static_cast<std::uint32_t>(p->ev_defs.size());
    if (sh->n_ev != 0u) {
        // Event detection runs on the thread-per-lane kernel family (ev_kernels.cuh).
        if (p->order + 1u > static_cast<std::uint32_t>(dev::EV_MAXP1)) {
            throw hy::detail::not_implemented_error("Event detection supports Taylor orders up to "
                                                    + std::to_string(dev::EV_MAXP1 - 1));
        }
        want = 1;
    }
    sh->configure(want, 0, 0, 0, 0);
    return sh;
}

// A batch of `batch` lanes split into contiguous blocks, as even as possible, one shard per entry of devs; never more
// shards than lanes.
std::unique_ptr<hy_batch> make_batch(const hy_program *p, std::uint32_t batch, const std::vector<int> &devs, int n_dev)
{
    auto b = std::make_unique<hy_batch>();
    b->n = batch;
    // (Event equations: every shard detects its own lanes' events.)
    b->n_ev = static_cast<std::uint32_t>(p->ev_defs.size());
    const std::uint32_t ns = std::min<std::uint32_t>(static_cast<std::uint32_t>(devs.size()), batch);
    b->shard_off.push_back(0u);
    for (std::uint32_t i = 0; i < ns; ++i) {
        const std::uint32_t lanes = batch / ns + (i < batch % ns ? 1u : 0u);
        b->shards.push_back(make_shard(p, lanes, devs[i], n_dev));
        b->shard_off.push_back(b->shard_off.back() + lanes);
    }
    return b;
}

} // namespace

extern "C" {

int hy_batch_create(const hy_program *p, uint32_t batch, int device, hy_batch **out)
{
    try {
        if (p == nullptr || out == nullptr) {
            throw std::invalid_argument("Null pointer passed to hy_batch_create()");
        }
        if (batch == 0u) {
            throw std::invalid_argument("The batch size in an adaptive Taylor integrator cannot be zero");
        }

        int n_dev = 0;
        if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) {
            throw cuda_error("No usable CUDA device: heyoka_b200 has no CPU fallback");
        }
        *out = make_batch(p, batch, {device}, n_dev).release();
        return HY_OK;
    } catch (...) {
        return translate_exception();
    }
}

int hy_batch_create_multi(const hy_program *p, uint32_t batch, const int *devices, uint32_t n_devices, hy_batch **out)
{
    try {
        if (p == nullptr || out == nullptr) {
            throw std::invalid_argument("Null pointer passed to hy_batch_create_multi()");
        }
        int n_dev = 0;
        if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) {
            throw cuda_error("No usable CUDA device: heyoka_b200 has no CPU fallback");
        }
        std::vector<int> devs;
        if (devices == nullptr || n_devices == 0u) {
            for (int d = 0; d < n_dev; ++d) {
                devs.push_back(d);
            }
        } else {
            devs.assign(devices, devices + n_devices);
        }
        if (batch == 0u) {
            throw std::invalid_argument("The batch size in an adaptive Taylor integrator cannot be zero");
        }
        auto b = make_batch(p, batch, devs, n_dev);
        b->sharded = true;
        *out = b.release();
        return HY_OK;
    } catch (...) {
        return translate_exception();
    }
}

int hy_device_count(void)
{
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess) {
        return 0;
    }
    return n_dev;
}

uint32_t hy_batch_n_shards(const hy_batch *b)
{
    return b == nullptr || !b->sharded ? 0u : static_cast<uint32_t>(b->shards.size());
}

void hy_batch_destroy(hy_batch *b)
{
    delete b;
}

int hy_selftest_div(uint64_t n, uint64_t seed, uint64_t *mismatches)
{
    try {
        if (mismatches == nullptr) {
            throw std::invalid_argument("Null pointer passed to hy_selftest_div()");
        }
        unsigned long long *d = nullptr;
        HY_CUDA_CHECK(cudaMalloc(&d, sizeof(unsigned long long)));
        HY_CUDA_CHECK(cudaMemset(d, 0, sizeof(unsigned long long)));
        dev::k_selftest_div<<<148 * 8, 256>>>(n, seed, d);
        HY_CUDA_CHECK(cudaGetLastError());
        unsigned long long h = 0;
        HY_CUDA_CHECK(cudaMemcpy(&h, d, sizeof(h), cudaMemcpyDeviceToHost));
        HY_CUDA_CHECK(cudaFree(d));
        *mismatches = h;
        return HY_OK;
    } catch (...) {
        return translate_exception();
    }
}

int hy_host_pin(void *ptr, size_t bytes)
{
    if (ptr == nullptr || bytes == 0u) {
        return HY_OK;
    }
    if (cudaHostRegister(ptr, bytes, cudaHostRegisterDefault) != cudaSuccess) {
        cudaGetLastError(); // (not fatal: the copies then go through the driver's staging buffers)
        hy::detail::set_last_error("cudaHostRegister() failed");
        return HY_ERR_CUDA;
    }
    return HY_OK;
}

int hy_host_unpin(void *ptr)
{
    if (ptr != nullptr && cudaHostUnregister(ptr) != cudaSuccess) {
        cudaGetLastError();
        return HY_ERR_CUDA;
    }
    return HY_OK;
}

int hy_batch_set_stream(hy_batch *b, void *cuda_stream)
{
    if (b != nullptr && b->sharded) {
        hy::detail::set_last_error("hy_batch_set_stream() is not available on a multi-device batch");
        return HY_ERR_INVALID_ARG;
    }
    if (b == nullptr) {
        hy::detail::set_last_error("Null batch");
        return HY_ERR_INVALID_ARG;
    }
    b->shards[0]->stream = static_cast<cudaStream_t>(cuda_stream);
    return HY_OK;
}

int hy_batch_sync(hy_batch *b)
{
    try {
        for_each_shard(b, [](shard &sh, std::size_t, std::size_t) { HY_CUDA_CHECK(cudaStreamSynchronize(sh.stream)); });
        return HY_OK;
    } catch (...) {
        return translate_exception();
    }
}

int hy_batch_set_launch_config(hy_batch *b, uint32_t block_threads, uint32_t blocks_per_sm)
{
    try {
        each_shard_in_order(b, [&](shard &sh, std::size_t, std::size_t) {
            HY_CUDA_CHECK(cudaStreamSynchronize(sh.stream));
            const int L = sh.cv != nullptr && sh.mode == 2 ? sh.cv->L : 0;
            const int N = sh.cv != nullptr && sh.mode == 2 ? sh.cv->N : 0;
            if (sh.nn_on) {
                sh.configure(8, 0, 0, 0, 0);
            } else if (sh.nb_on) {
                sh.configure(sh.nb_lane ? 9 : (sh.c_cta ? 7 : 6), L, sh.nbv->tmem ? 1 : 2, block_threads, blocks_per_sm);
            } else {
                sh.configure(sh.mode, L, N, block_threads, blocks_per_sm);
            }
        });
        return HY_OK;
    } catch (...) {
        return translate_exception();
    }
}

int hy_batch_set_kernel(hy_batch *b, int tape_mode, uint32_t lanes_per_warp, uint32_t lanes_per_thread,
                        uint32_t block_threads, uint32_t blocks_per_sm)
{
    try {
        if (b == nullptr) {
            throw std::invalid_argument("Null batch");
        }
        if (tape_mode < 0 || tape_mode > 9) {
            throw std::invalid_argument("Invalid tape mode");
        }
        each_shard_in_order(b, [&](shard &sh, std::size_t, std::size_t) {
            HY_CUDA_CHECK(cudaStreamSynchronize(sh.stream));
            sh.configure(tape_mode, static_cast<int>(lanes_per_warp), static_cast<int>(lanes_per_thread), block_threads,
                         blocks_per_sm);
        });
        return HY_OK;
    } catch (...) {
        return translate_exception();
    }
}

int hy_batch_get_kernel(const hy_batch *b, hy_kernel_info *out)
{
    if (b == nullptr || out == nullptr) {
        hy::detail::set_last_error("Null pointer passed to hy_batch_get_kernel()");
        return HY_ERR_INVALID_ARG;
    }
    const shard &s = *b->shards[0]; // (every shard runs the same kernel shape)
    out->tape_mode = s.nn_on ? 8 : s.nb_on ? (s.nb_lane ? 9 : (s.c_cta ? 7 : 6)) : (s.mode == 2 && s.c_global ? (s.c_cta ? 5 : 4) : s.mode);
    out->lanes_per_warp = s.mode == 2 ? static_cast<uint32_t>(s.cv->L) : 32u;
    out->lanes_per_thread = s.mode == 2 ? static_cast<uint32_t>(s.cv->N) : 1u;
    out->block_threads = s.mode == 2 ? s.c_threads : s.h_threads;
    out->blocks_per_sm = s.mode == 2 ? s.c_ctas_per_sm : s.h_blocks_per_sm;
    out->grid = s.mode == 2 ? s.c_grid : s.h_grid;
    out->smem_bytes = s.mode == 2 ? static_cast<uint64_t>(s.c_smem) : 0u;
    out->tape_slots_per_lane = s.nb_on ? s.nbd.n_slots_equiv : (s.mode == 2 ? s.plan.n_slots : s.n_uvars * (s.order + 1u));
    out->n_segments = s.plan.n_segments;
    out->n_fused = s.plan.n_fused;
    out->n_sms = s.n_sms;
    out->tmem_cols_per_warp
        = s.nb_on ? (s.nbv->tmem ? s.nbd.npp * 12u : 0u)
                  : (s.mode == 2 && s.plan.tmem != 0u
                         ? s.plan.tmem * (s.order + 1u) * 2u * static_cast<uint32_t>(s.cv->N)
                         : 0u);
    out->reserved = 0u;
    return HY_OK;
}

int hy_batch_upload(hy_batch *b, const double *state, const double *pars, const double *t_hi, const double *t_lo)
{
    try {
        for_each_shard(b, [&](shard &sh, std::size_t off, std::size_t) {
            rows_h2d(sh, sh.d_state, state, sh.n_eq, b->n, off);
            rows_h2d(sh, sh.d_pars, pars, sh.n_pars, b->n, off);
            rows_h2d(sh, sh.d_t_hi, t_hi, 1u, b->n, off);
            rows_h2d(sh, sh.d_t_lo, t_lo, 1u, b->n, off);
            HY_CUDA_CHECK(cudaStreamSynchronize(sh.stream));
        });
        return HY_OK;
    } catch (...) {
        return translate_exception();
    }
}

int hy_batch_download(hy_batch *b, double *state, double *t_hi, double *t_lo, double *last_h)
{
    try {
        for_each_shard(b, [&](shard &sh, std::size_t off, std::size_t) {
            rows_d2h(sh, state, sh.d_state, sh.n_eq, b->n, off);
            rows_d2h(sh, t_hi, sh.d_t_hi, 1u, b->n, off);
            rows_d2h(sh, t_lo, sh.d_t_lo, 1u, b->n, off);
            rows_d2h(sh, last_h, sh.d_last_h, 1u, b->n, off);
            HY_CUDA_CHECK(cudaStreamSynchronize(sh.stream));
        });
        return HY_OK;
    } catch (...) {
        return translate_exception();
    }
}

int hy_batch_download_step_res(hy_batch *b, int64_t *outcome, double *h)
{
    try {
        for_each_shard(b, [&](shard &sh, std::size_t off, std::size_t) {
            rows_d2h(sh, reinterpret_cast<long long *>(outcome), sh.d_step_outcome, 1u, b->n, off);
            rows_d2h(sh, h, sh.d_last_h, 1u, b->n, off);
            HY_CUDA_CHECK(cudaStreamSynchronize(sh.stream));
        });
        return HY_OK;
    } catch (...) {
        return translate_exception();
    }
}

int hy_batch_download_prop_res(hy_batch *b, int64_t *outcome, double *min_h, double *max_h, uint64_t *n_steps)
{
    try {
        for_each_shard(b, [&](shard &sh, std::size_t off, std::size_t) {
            rows_d2h(sh, reinterpret_cast<long long *>(outcome), sh.d_prop_outcome, 1u, b->n, off);
            rows_d2h(sh, min_h, sh.d_prop_min_h, 1u, b->n, off);
            rows_d2h(sh, max_h, sh.d_prop_max_h, 1u, b->n, off);
            rows_d2h(sh, reinterpret_cast<unsigned long long *>(n_steps), sh.d_prop_n_steps, 1u, b->n, off);
            HY_CUDA_CHECK(cudaStreamSynchronize(sh.stream));
        });
        return HY_OK;
    } catch (...) {
        return translate_exception();
    }
}

int hy_batch_download_tc(hy_batch *b, double *tc)
{
    try {
        for_each_shard(b, [&](shard &sh, std::size_t off, std::size_t) {
            sh.ensure_tc();
            rows_d2h(sh, tc, sh.d_tc, static_cast<std::size_t>(sh.n_eq) * (sh.order + 1u), b->n, off);
            HY_CUDA_CHECK(cudaStreamSynchronize(sh.stream));
        });
        return HY_OK;
    } catch (...) {
        return translate_exception();
    }
}

int hy_batch_upload_tc(hy_batch *b, const double *tc)
{
    try {
        if (b == nullptr || tc == nullptr) {
            throw std::invalid_argument("Null pointer passed to hy_batch_upload_tc()");
        }
        for_each_shard(b, [&](shard &sh, std::size_t off, std::size_t) {
            sh.ensure_tc();
            rows_h2d(sh, sh.d_tc, tc, static_cast<std::size_t>(sh.n_eq) * (sh.order + 1u), b->n, off);
            HY_CUDA_CHECK(cudaStreamSynchronize(sh.stream));
        });
        return HY_OK;
    } catch (...) {
        return translate_exception();
    }
}

int hy_batch_get_ptrs(hy_batch *b, hy_batch_ptrs *out)
{
    if (b != nullptr && b->sharded) {
        hy::detail::set_last_error("hy_batch_get_ptrs() is not available on a multi-device batch: use the shards");
        return HY_ERR_INVALID_ARG;
    }
    if (b == nullptr || out == nullptr) {
        hy::detail::set_last_error("Null pointer passed to hy_batch_get_ptrs()");
        return HY_ERR_INVALID_ARG;
    }
    const shard &s = *b->shards[0];
    out->state = s.d_state;
    out->pars = s.d_pars;
    out->t_hi = s.d_t_hi;
    out->t_lo = s.d_t_lo;
    out->last_h = s.d_last_h;
    out->tc = s.d_tc; // null until a step with write_tc / a dense output has been requested
    out->d_out = s.d_d_out;
    out->step_outcome = reinterpret_cast<int64_t *>(s.d_step_outcome);
    out->prop_outcome = reinterpret_cast<int64_t *>(s.d_prop_outcome);
    out->prop_min_h = s.d_prop_min_h;
    out->prop_max_h = s.d_prop_max_h;
    out->prop_n_steps = reinterpret_cast<uint64_t *>(s.d_prop_n_steps);
    return HY_OK;
}

int hy_batch_step(hy_batch *b, const double *max_delta_t, int on_device, int backward, int write_tc)
{
    try {
        if (b->sharded && on_device) {
            throw std::invalid_argument("Device-resident step limits are not available on a multi-device batch");
        }
        if (max_delta_t != nullptr && !on_device) {
            // step(max_delta_ts): NaN limits are rejected (src/taylor_adaptive_batch.cpp:1060-1075).
            for (std::uint32_t i = 0; i < b->n; ++i) {
                if (std::isnan(max_delta_t[i])) {
                    throw std::invalid_argument("Cannot use a nan max_delta_t in the step() function of an adaptive "
                                                "Taylor integrator in batch mode");
                }
            }
        }
        if (b->n_ev != 0u && !b->ev_set) {
            throw std::invalid_argument("hy_batch_set_events() must be called before stepping a batch with event equations");
        }
        for_each_shard(b, [&](shard &sh, std::size_t off, std::size_t) {
            const double *d_mdt = on_device ? max_delta_t : stage(sh, max_delta_t, off, 0);
            if (b->n_ev != 0u) {
                // A batch with event equations: every step detects events (the Taylor coefficients are always
                // written, src/taylor_adaptive_batch.cpp:776); hy_batch_get_events() returns what was found.
                sh.ev_step(d_mdt, backward);
                return;
            }
            dev::run_args R{};
            R.max_delta_t = d_mdt;
            R.default_max_delta_t
                = backward ? -std::numeric_limits<double>::infinity() : std::numeric_limits<double>::infinity();
            R.write_tc = write_tc;
            R.flags = sh.d_flags;
            R.counter = sh.d_counter;
            sh.launch(false, R);
        });
        if (b->n_ev != 0u) {
            // The events of the step, lanes ascending: the shards' lists one after the other, with the lanes of the
            // whole batch.
            b->ev_host.clear();
            for (std::size_t i = 0; i < b->shards.size(); ++i) {
                for (hy_event_rec r : b->shards[i]->ev_host) {
                    r.lane += b->shard_off[i];
                    b->ev_host.push_back(r);
                }
            }
        }
        return HY_OK;
    } catch (...) {
        return translate_exception();
    }
}

namespace
{

// The checks of propagate_until_impl() that need the CURRENT times (src/taylor_adaptive_batch.cpp:1212-1273): finite,
// and final time - current time representable (check_prop_times(): 16 bytes per lane come back from the device for them).
void check_prop_times_host(std::uint32_t n, const double *t_hi, const double *t_lo, const double *tf_hi, const double *tf_lo)
{
    for (std::uint32_t i = 0; i < n; ++i) {
        if (!std::isfinite(t_hi[i]) || !std::isfinite(t_lo[i])) {
            throw std::invalid_argument("Cannot invoke the propagate_until() function of an adaptive Taylor integrator "
                                        "in batch mode if one of the current times is not finite");
        }
    }
    for (std::uint32_t i = 0; i < n; ++i) {
        // (Same arithmetic as the device: Knuth two-sum of the high parts is enough to detect the overflow.)
        const double rem = tf_hi[i] - t_hi[i] + ((tf_lo != nullptr ? tf_lo[i] : 0.) - t_lo[i]);
        if (!std::isfinite(rem)) {
            throw std::invalid_argument("The final time passed to the propagate_until() function of an adaptive Taylor "
                                        "integrator in batch mode results in an overflow condition");
        }
    }
}

void check_prop_times(hy_batch *b, const double *tf_hi, const double *tf_lo)
{
    std::vector<double> t_hi(b->n), t_lo(b->n);
    if (hy_batch_download(b, nullptr, t_hi.data(), t_lo.data(), nullptr) != HY_OK) {
        throw cuda_error(hy_last_error());
    }
    check_prop_times_host(b->n, t_hi.data(), t_lo.data(), tf_hi, tf_lo);
}

// Argument checks of propagate_until_impl(), src/taylor_adaptive_batch.cpp:1212-1241.
void check_prop_args(std::uint32_t n, const double *t_final_hi, const double *t_final_lo, const double *max_delta_t)
{
    for (std::uint32_t i = 0; i < n; ++i) {
        if (!std::isfinite(t_final_hi[i]) || (t_final_lo != nullptr && !std::isfinite(t_final_lo[i]))) {
            throw std::invalid_argument("A non-finite time was passed to the propagate_until() function of an "
                                        "adaptive Taylor integrator in batch mode");
        }
        if (max_delta_t != nullptr) {
            if (std::isnan(max_delta_t[i])) {
                throw std::invalid_argument("A nan max_delta_t was passed to the propagate_until() function of an "
                                            "adaptive Taylor integrator in batch mode");
            }
            if (max_delta_t[i] <= 0) {
                throw std::invalid_argument("A non-positive max_delta_t was passed to the propagate_until() "
                                            "function of an adaptive Taylor integrator in batch mode");
            }
        }
    }
}

} // namespace

int hy_batch_propagate_until(hy_batch *b, const double *t_final_hi, const double *t_final_lo, const double *max_delta_t,
                             uint64_t max_steps, int write_tc)
{
    try {
        if (b != nullptr && b->n_ev != 0u) {
            throw hy::detail::not_implemented_error("A batch with event equations is propagated by the front end's lock-step "
                                                    "loop over hy_batch_step(), not by the device-resident propagation");
        }
        if (t_final_hi == nullptr) {
            throw std::invalid_argument("Null final times passed to hy_batch_propagate_until()");
        }
        check_prop_args(b->n, t_final_hi, t_final_lo, max_delta_t);
        check_prop_times(b, t_final_hi, t_final_lo);
        return propagate(b, t_final_hi, t_final_lo, max_delta_t, 0, max_steps, write_tc, nullptr);
    } catch (...) {
        return translate_exception();
    }
}

// propagate_until() on HOST buffers in one call: upload of state / parameters / times, propagation, download of state,
// times, last_h and the per-lane results (the outputs may alias the inputs). On a batch of several shards (hy_batch_create_multi(): several devices, or the
// SAME device listed several times) every shard runs its copies and its kernel on its own stream from its own host
// thread: with k shards on one device the copies of a shard overlap the kernels of the others, and only 1 / k of the
// transfers stays exposed. The checks on the current times are done on the caller's arrays (no read-back), the state is
// downloaded right after the shard's kernel; only last_h (and the outcomes, if the iteration limit was hit) wait for the
// global exits across the shards.
int hy_batch_propagate_until_host(hy_batch *b, const double *state_in, const double *pars, const double *t_hi_in,
                                  const double *t_lo_in, const double *t_final_hi, const double *t_final_lo,
                                  const double *max_delta_t, uint64_t max_steps, double *state, double *t_hi, double *t_lo,
                                  double *last_h, int64_t *outcome, double *min_h, double *max_h, uint64_t *n_steps)
{
    try {
        if (b == nullptr || state_in == nullptr || t_hi_in == nullptr || t_lo_in == nullptr || t_final_hi == nullptr) {
            throw std::invalid_argument("Null pointer passed to hy_batch_propagate_until_host()");
        }
        if (b->n_ev != 0u) {
            throw hy::detail::not_implemented_error("A batch with event equations is propagated by the front end's lock-step "
                                                    "loop over hy_batch_step(), not by the device-resident propagation");
        }
        check_prop_args(b->n, t_final_hi, t_final_lo, max_delta_t);
        check_prop_times_host(b->n, t_hi_in, t_lo_in, t_final_hi, t_final_lo);
        const std::size_t pitch = b->n;
        std::vector<prop_ctx> ctx(b->shards.size());
        const auto download_main = [&](shard &sh, std::size_t off) {
            rows_d2h(sh, state, sh.d_state, sh.n_eq, pitch, off);
            rows_d2h(sh, t_hi, sh.d_t_hi, 1u, pitch, off);
            rows_d2h(sh, t_lo, sh.d_t_lo, 1u, pitch, off);
            rows_d2h(sh, reinterpret_cast<long long *>(outcome), sh.d_prop_outcome, 1u, pitch, off);
            rows_d2h(sh, min_h, sh.d_prop_min_h, 1u, pitch, off);
            rows_d2h(sh, max_h, sh.d_prop_max_h, 1u, pitch, off);
            rows_d2h(sh, reinterpret_cast<unsigned long long *>(n_steps), sh.d_prop_n_steps, 1u, pitch, off);
        };
        for_each_shard(b, [&](shard &sh, std::size_t off, std::size_t i) {
            rows_h2d(sh, sh.d_state, state_in, sh.n_eq, pitch, off);
            rows_h2d(sh, sh.d_pars, pars, sh.n_pars, pitch, off);
            rows_h2d(sh, sh.d_t_hi, t_hi_in, 1u, pitch, off);
            rows_h2d(sh, sh.d_t_lo, t_lo_in, 1u, pitch, off);
            const double *d_hi = stage(sh, t_final_hi, off, 0);
            const double *d_lo = stage(sh, t_final_lo, off, 1);
            const double *d_mdt = stage(sh, max_delta_t, off, 2);
            propagate_phase1(sh, d_hi, d_lo, d_mdt, max_steps, 0, ctx[i]);
            // (Speculative: a non-finite lane anywhere makes every shard run again, see below.)
            download_main(sh, off);
        });
        bool any_nf = false, any_limit = false;
        unsigned long long cap = ~0ull, loop_len = 0;
        for (const auto &c : ctx) {
            if (c.fl.any_nf != 0u) {
                any_nf = true;
                cap = std::min(cap, c.fl.min_nf_iter);
            }
        }
        if (any_nf) {
            for_each_shard(b, [&](shard &sh, std::size_t, std::size_t i) {
                HY_CUDA_CHECK(cudaStreamSynchronize(sh.stream));
                propagate_replay(sh, ctx[i], cap);
            });
        }
        for (const auto &c : ctx) {
            any_limit = any_limit || c.fl.any_limit != 0u;
            loop_len = std::max(loop_len, c.fl.max_iter);
        }
        for_each_shard(b, [&](shard &sh, std::size_t off, std::size_t) {
            propagate_finish(sh, any_nf, any_limit, loop_len, 0);
            if (any_nf || any_limit) {
                download_main(sh, off);
            }
            rows_d2h(sh, last_h, sh.d_last_h, 1u, pitch, off);
            HY_CUDA_CHECK(cudaStreamSynchronize(sh.stream));
        });
        return HY_OK;
    } catch (...) {
        return translate_exception();
    }
}

int hy_batch_propagate_until_dev(hy_batch *b, const double *d_t_final_hi, const double *d_t_final_lo,
                                 const double *d_max_delta_t, uint64_t max_steps, int write_tc, int *any_nf_or_limit)
{
    try {
        if (b != nullptr && b->n_ev != 0u) {
            throw hy::detail::not_implemented_error("A batch with event equations is propagated by the front end's lock-step "
                                                    "loop over hy_batch_step(), not by the device-resident propagation");
        }
        if (b->sharded) {
            throw std::invalid_argument("hy_batch_propagate_until_dev() is not available on a multi-device batch");
        }
        if (d_t_final_hi == nullptr) {
            throw std::invalid_argument("Null final times passed to hy_batch_propagate_until_dev()");
        }
        return propagate(b, d_t_final_hi, d_t_final_lo, d_max_delta_t, 1, max_steps, write_tc, any_nf_or_limit);
    } catch (...) {
        return translate_exception();
    }
}

// propagate_grid() (src/taylor_adaptive_batch.cpp:1545-2055). The reference's algorithm is kept as it is: an
// initial propagate_until(grid[0]) with write_tc, then lock-step iterations of {dense output at every grid point
// covered by the last step; one step clamped to the last grid point}. The per-lane work runs on the device (one
// step launch + two small kernels per iteration); the host only reads the two loop flags.
namespace
{

// The argument checks of propagate_grid_impl() (src/taylor_adaptive_batch.cpp:1575-1670); reads the current times back.
void check_grid(hy_batch *b, const double *grid, uint64_t n_pts, const double *max_delta_t)
{
    const std::uint32_t n = b->n;
    if (n_pts == 0u) {
        throw std::invalid_argument("Cannot invoke propagate_grid() in an adaptive Taylor integrator in batch mode "
                                    "if the time grid is empty");
    }
    if (n_pts > 0xffffffffull) {
        throw std::overflow_error("Too many grid points passed to propagate_grid()");
    }
    // The current time must be finite (:1590-1594).
    std::vector<double> t_hi(n), t_lo(n);
    {
        // (Through the download entry point, which gathers the lanes of every shard.)
        if (hy_batch_download(b, nullptr, t_hi.data(), t_lo.data(), nullptr) != HY_OK) {
            throw cuda_error(hy_last_error());
        }
        for (std::uint32_t i = 0; i < n; ++i) {
            if (!std::isfinite(t_hi[i]) || !std::isfinite(t_lo[i])) {
                throw std::invalid_argument("Cannot invoke propagate_grid() in an adaptive Taylor integrator in "
                                            "batch mode if the current time is not finite");
            }
        }
    }
    if (max_delta_t != nullptr) {
        for (std::uint32_t i = 0; i < n; ++i) {
            if (std::isnan(max_delta_t[i])) {
                throw std::invalid_argument("A nan max_delta_t was passed to the propagate_grid() function of an "
                                            "adaptive Taylor integrator in batch mode");
            }
            if (max_delta_t[i] <= 0) {
                throw std::invalid_argument("A non-positive max_delta_t was passed to the propagate_grid() "
                                            "function of an adaptive Taylor integrator in batch mode");
            }
        }
    }
    // Grid checks, :1619-1656: finite, strictly monotonic, same direction in every lane.
    constexpr auto nf_err_msg
        = "A non-finite time value was passed to propagate_grid() in an adaptive Taylor integrator in batch mode";
    constexpr auto ig_err_msg = "A non-monotonic time grid was passed to propagate_grid() in an adaptive "
                                "Taylor integrator in batch mode";
    const auto batch_nf = [&](std::uint64_t k) {
        return std::any_of(grid + k * n, grid + (k + 1u) * n, [](double t) { return !std::isfinite(t); });
    };
    if (batch_nf(0)) {
        throw std::invalid_argument(nf_err_msg);
    }
    if (n_pts > 1u) {
        // The direction is established from the first two points of lane 0.
        if (batch_nf(1)) {
            throw std::invalid_argument(nf_err_msg);
        }
        if (grid[n] == grid[0]) {
            throw std::invalid_argument(ig_err_msg);
        }
        const bool dir = grid[n] > grid[0];
        for (std::uint64_t k = 1; k < n_pts; ++k) {
            if (k > 1u && batch_nf(k)) {
                throw std::invalid_argument(nf_err_msg);
            }
            for (std::uint32_t i = 0; i < n; ++i) {
                if ((grid[k * n + i] > grid[(k - 1u) * n + i]) != dir) {
                    throw std::invalid_argument(ig_err_msg);
                }
            }
        }
    }
    // The grid must start at the current time (:1660-1670).
    for (std::uint32_t i = 0; i < n; ++i) {
        if (t_hi[i] != grid[i]) {
            throw std::invalid_argument(
                "When invoking propagate_grid(), the first element of the time grid must match the current "
                "time coordinate - however, the first element of the time grid at batch index "
                + std::to_string(i) + " has a value of " + hy::detail::fmt_double(grid[i])
                + ", while the current time coordinate is " + hy::detail::fmt_double(t_hi[i]));
        }
    }
}

} // namespace

int hy_batch_check_grid(hy_batch *b, const double *grid, uint64_t n_pts, const double *max_delta_t)
{
    try {
        if (b == nullptr || grid == nullptr) {
            throw std::invalid_argument("Null pointer passed to hy_batch_check_grid()");
        }
        check_grid(b, grid, n_pts, max_delta_t);
        return HY_OK;
    } catch (...) {
        return translate_exception();
    }
}

int hy_batch_propagate_grid(hy_batch *b, const double *grid, uint64_t n_pts, const double *max_delta_t,
                            uint64_t max_steps, double *out)
{
    double *d_grid = nullptr, *d_out = nullptr, *d_lane = nullptr;
    std::uint32_t *d_idx = nullptr;
    unsigned char *d_dir = nullptr;
    unsigned *d_gflags = nullptr;
    const auto cleanup = [&]() {
        for (void *ptr : {static_cast<void *>(d_grid), static_cast<void *>(d_out), static_cast<void *>(d_lane),
                          static_cast<void *>(d_idx), static_cast<void *>(d_dir), static_cast<void *>(d_gflags)}) {
            if (ptr != nullptr) {
                cudaFree(ptr);
            }
        }
    };
    try {
        if (b != nullptr && b->n_ev != 0u) {
            throw hy::detail::not_implemented_error("A batch with event equations is propagated by the front end's lock-step "
                                                    "loop over hy_batch_step(), not by the device-resident propagation");
        }
        if (b == nullptr || grid == nullptr || out == nullptr) {
            throw std::invalid_argument("Null pointer passed to hy_batch_propagate_grid()");
        }
        if (b->sharded) {
            throw hy::detail::not_implemented_error("propagate_grid() is not available on a multi-device batch");
        }
        shard &sh = *b->shards[0];
        device_guard guard(sh.device);
        const std::uint32_t n = sh.n;
        check_grid(b, grid, n_pts, max_delta_t);

        const std::size_t n_out = static_cast<std::size_t>(n_pts) * sh.n_eq * n, state_doubles = std::size_t(sh.n_eq) * n;
        HY_CUDA_CHECK(cudaMalloc(&d_grid, sizeof(double) * n_pts * n));
        HY_CUDA_CHECK(cudaMalloc(&d_out, sizeof(double) * n_out));
        HY_CUDA_CHECK(cudaMalloc(&d_lane, sizeof(double) * 4u * n)); // rem_hi, rem_lo, dt_limit, max_delta_t
        HY_CUDA_CHECK(cudaMalloc(&d_idx, sizeof(std::uint32_t) * n));
        HY_CUDA_CHECK(cudaMalloc(&d_dir, n));
        HY_CUDA_CHECK(cudaMalloc(&d_gflags, sizeof(unsigned) * 4u));
        HY_CUDA_CHECK(cudaMemcpyAsync(d_grid, grid, sizeof(double) * n_pts * n, cudaMemcpyHostToDevice, sh.stream));
        if (max_delta_t != nullptr) {
            HY_CUDA_CHECK(cudaMemcpyAsync(d_lane + 3u * n, max_delta_t, sizeof(double) * n, cudaMemcpyHostToDevice,
                                          sh.stream));
        }
        dev::k_fill_double<<<static_cast<unsigned>((n_out + 255u) / 256u), 256, 0, sh.stream>>>(
            d_out, n_out, std::numeric_limits<double>::quiet_NaN());
        HY_CUDA_CHECK(cudaGetLastError());
        const unsigned gb = (n + 127u) / 128u;
        const auto finish = [&]() {
            HY_CUDA_CHECK(cudaMemcpyAsync(out, d_out, sizeof(double) * n_out, cudaMemcpyDeviceToHost, sh.stream));
            HY_CUDA_CHECK(cudaStreamSynchronize(sh.stream));
            cleanup();
            return HY_OK;
        };

        // Up to the first grid point (a zero-length step when the time is already there: it brings the Taylor
        // coefficients up to date), :1697-1706.
        {
            const double *d_mdt = max_delta_t != nullptr ? d_lane + 3u * n : nullptr;
            const int rc = propagate(b, d_grid, nullptr, d_mdt, 1, max_steps, 1, nullptr);
            if (rc != HY_OK) {
                cleanup();
                return rc;
            }
            std::vector<long long> oc(n);
            HY_CUDA_CHECK(cudaMemcpyAsync(oc.data(), sh.d_prop_outcome, sizeof(long long) * n, cudaMemcpyDeviceToHost,
                                          sh.stream));
            HY_CUDA_CHECK(cudaStreamSynchronize(sh.stream));
            if (std::any_of(oc.begin(), oc.end(), [](long long v) { return v != HY_OUTCOME_TIME_LIMIT; })) {
                // Outcomes kept, counters reset (:1709-1722).
                dev::k_fill_double<<<gb, 128, 0, sh.stream>>>(sh.d_prop_min_h, n, std::numeric_limits<double>::infinity());
                dev::k_fill_double<<<gb, 128, 0, sh.stream>>>(sh.d_prop_max_h, n, 0.);
                HY_CUDA_CHECK(cudaMemsetAsync(sh.d_prop_n_steps, 0, sizeof(unsigned long long) * n, sh.stream));
                return finish();
            }
        }
        HY_CUDA_CHECK(cudaMemcpyAsync(d_out, sh.d_state, sizeof(double) * state_doubles, cudaMemcpyDeviceToDevice,
                                      sh.stream));

        dev::grid_state G{};
        G.grid = d_grid;
        G.n_pts = static_cast<std::uint32_t>(n_pts);
        G.out = d_out;
        G.max_delta_t = max_delta_t != nullptr ? d_lane + 3u * n : nullptr;
        G.cur_idx = d_idx;
        G.rem_hi = d_lane;
        G.rem_lo = d_lane + n;
        G.t_dir = d_dir;
        G.dt_limit = d_lane + 2u * n;
        G.flags = d_gflags;
        unsigned hflags[4] = {0u, 0u, 0u, 0u};
        const auto read_flags = [&]() {
            HY_CUDA_CHECK(cudaMemcpyAsync(hflags, d_gflags, sizeof(hflags), cudaMemcpyDeviceToHost, sh.stream));
            HY_CUDA_CHECK(cudaStreamSynchronize(sh.stream));
        };
        HY_CUDA_CHECK(cudaMemsetAsync(d_gflags, 0, sizeof(hflags), sh.stream));
        dev::k_grid_init<<<gb, 128, 0, sh.stream>>>(sh.view(), G, sh.d_prop_min_h, sh.d_prop_max_h, sh.d_prop_n_steps);
        dev::k_grid_sample<<<dim3(gb, sh.n_eq), 128, 0, sh.stream>>>(sh.prog, sh.view(), G);
        dev::k_grid_advance<<<gb, 128, 0, sh.stream>>>(sh.view(), G);
        HY_CUDA_CHECK(cudaGetLastError());
        read_flags();
        if (hflags[2] != 0u) {
            throw std::invalid_argument("The final time passed to the propagate_grid() function of an adaptive Taylor "
                                        "integrator in batch mode results in an overflow condition");
        }
        std::uint64_t iter = 0;
        bool interrupted = false;
        while (hflags[0] != 0u && !interrupted) {
            dev::run_args R{};
            R.max_delta_t = G.dt_limit;
            R.default_max_delta_t = std::numeric_limits<double>::infinity();
            R.write_tc = 1;
            R.flags = sh.d_flags;
            R.counter = sh.d_counter;
            sh.launch(false, R);
            HY_CUDA_CHECK(cudaMemsetAsync(d_gflags, 0, sizeof(unsigned) * 2u, sh.stream));
            dev::k_grid_book<<<gb, 128, 0, sh.stream>>>(sh.view(), G, sh.d_prop_outcome, sh.d_prop_min_h,
                                                        sh.d_prop_max_h, sh.d_prop_n_steps);
            dev::k_grid_sample<<<dim3(gb, sh.n_eq), 128, 0, sh.stream>>>(sh.prog, sh.view(), G);
            dev::k_grid_advance<<<gb, 128, 0, sh.stream>>>(sh.view(), G);
            HY_CUDA_CHECK(cudaGetLastError());
            read_flags();
            if (hflags[1] != 0u) {
                break; // non-finite state: nothing further is written (:1973-1978)
            }
            if (++iter == max_steps) {
                dev::k_fill_outcome<<<(n + 255u) / 256u, 256, 0, sh.stream>>>(sh.d_prop_outcome, n,
                                                                               HY_OUTCOME_STEP_LIMIT);
                interrupted = true;
            }
        }
        return finish();
    } catch (...) {
        cleanup();
        return translate_exception();
    }
}

// ------------------------------------------------------------------------------------------------
// Continuous output.
// ------------------------------------------------------------------------------------------------
struct hy_cout {
    int device = 0;
    std::uint32_t n = 0, n_eq = 0, order = 0;
    std::uint64_t n_steps = 0; // recorded iterations; times have n_steps + 2 rows (start, ..., padding)
    dev::program prog{};
    // The Taylor coefficients of the recorded iterations live in slabs of slab_iters iterations each, written in
    // place by the step kernel (no copy, no final re-pack); d_slabs is the device-side table of the slab pointers.
    std::vector<double *> slabs;
    double **d_slabs = nullptr;
    std::uint32_t slab_iters = 1;
    cudaStream_t stream = nullptr;
    double *d_t_hi = nullptr, *d_t_lo = nullptr, *d_tm = nullptr, *d_out = nullptr;
    ~hy_cout()
    {
        for (double *ptr : slabs) {
            cudaFree(ptr);
        }
        for (void *ptr : {static_cast<void *>(d_slabs), static_cast<void *>(d_t_hi), static_cast<void *>(d_t_lo),
                          static_cast<void *>(d_tm), static_cast<void *>(d_out)}) {
            if (ptr != nullptr) {
                cudaFree(ptr);
            }
        }
    }
};

namespace
{
struct callback_abort {
};
} // namespace

int hy_batch_propagate_until_cout(hy_batch *b, const double *t_final_hi, const double *t_final_lo,
                                  const double *max_delta_t, uint64_t max_steps, hy_cout **out)
{
    return hy_batch_propagate_until_cout_cb(b, t_final_hi, t_final_lo, max_delta_t, max_steps, nullptr, nullptr, out);
}

int hy_batch_propagate_until_cout_cb(hy_batch *b, const double *t_final_hi, const double *t_final_lo,
                                     const double *max_delta_t, uint64_t max_steps, hy_step_callback cb, void *user,
                                     hy_cout **out)
{
    // The recording (hy_cout) owns its device memory from the start: slabs of Taylor coefficients the step kernel
    // writes into directly, and the times of the iterations in a geometrically grown array.
    std::unique_ptr<hy_cout> co;
    double *d_lane = nullptr, *d_times = nullptr, *own_tc = nullptr;
    std::size_t times_cap = 0, times_rows = 0; // rows of 2 * n doubles (hi, lo)
    unsigned char *d_dir = nullptr;
    unsigned *d_pflags = nullptr;
    bool tc_swapped = false;
    shard *sh = nullptr;
    const auto cleanup = [&]() {
        if (tc_swapped) {
            sh->d_tc = own_tc;
        }
        for (void *ptr : {static_cast<void *>(d_lane), static_cast<void *>(d_dir), static_cast<void *>(d_pflags),
                          static_cast<void *>(d_times)}) {
            if (ptr != nullptr) {
                cudaFree(ptr);
            }
        }
    };
    try {
        if (b != nullptr && b->n_ev != 0u) {
            throw hy::detail::not_implemented_error("A batch with event equations is propagated by the front end's lock-step "
                                                    "loop over hy_batch_step(), not by the device-resident propagation");
        }
        if (b != nullptr && b->sharded) {
            throw hy::detail::not_implemented_error("Continuous output is not available on a multi-device batch");
        }
        if (b == nullptr || t_final_hi == nullptr || out == nullptr) {
            throw std::invalid_argument("Null pointer passed to hy_batch_propagate_until_cout()");
        }
        *out = nullptr;
        sh = b->shards[0].get();
        device_guard guard(sh->device);
        const std::uint32_t n = sh->n;
        check_prop_args(n, t_final_hi, t_final_lo, max_delta_t);
        // rem_hi, rem_lo, dt_limit, max_delta_t, tf_hi, tf_lo
        HY_CUDA_CHECK(cudaMalloc(&d_lane, sizeof(double) * 6u * n));
        HY_CUDA_CHECK(cudaMalloc(&d_dir, n));
        HY_CUDA_CHECK(cudaMalloc(&d_pflags, sizeof(unsigned) * 4u));
        HY_CUDA_CHECK(cudaMemcpyAsync(d_lane + 4u * n, t_final_hi, sizeof(double) * n, cudaMemcpyHostToDevice, sh->stream));
        if (t_final_lo != nullptr) {
            HY_CUDA_CHECK(cudaMemcpyAsync(d_lane + 5u * n, t_final_lo, sizeof(double) * n, cudaMemcpyHostToDevice,
                                          sh->stream));
        }
        if (max_delta_t != nullptr) {
            HY_CUDA_CHECK(cudaMemcpyAsync(d_lane + 3u * n, max_delta_t, sizeof(double) * n, cudaMemcpyHostToDevice,
                                          sh->stream));
        }
        dev::prop_state G{};
        G.tf_hi = d_lane + 4u * n;
        G.tf_lo = t_final_lo != nullptr ? d_lane + 5u * n : nullptr;
        G.max_delta_t = max_delta_t != nullptr ? d_lane + 3u * n : nullptr;
        G.rem_hi = d_lane;
        G.rem_lo = d_lane + n;
        G.t_dir = d_dir;
        G.dt_limit = d_lane + 2u * n;
        G.flags = d_pflags;
        const unsigned gb = (n + 127u) / 128u;
        const std::size_t tc_doubles = static_cast<std::size_t>(sh->n_eq) * (sh->order + 1u) * n;
        unsigned hflags[4] = {0u, 0u, 0u, 0u};
        const auto read_flags = [&]() {
            HY_CUDA_CHECK(cudaMemcpyAsync(hflags, d_pflags, sizeof(hflags), cudaMemcpyDeviceToHost, sh->stream));
            HY_CUDA_CHECK(cudaStreamSynchronize(sh->stream));
        };
        co = std::make_unique<hy_cout>();
        co->device = sh->device;
        co->n = n;
        co->n_eq = sh->n_eq;
        co->order = sh->order;
        co->prog = sh->prog;
        co->stream = sh->stream;
        // Slabs of about 64 MB (at least one iteration each).
        co->slab_iters = static_cast<std::uint32_t>(
            std::min<std::size_t>(std::max<std::size_t>((std::size_t(64) << 20) / (tc_doubles * sizeof(double)), 1u), 4096u));
        // Row 0 of the times: the starting time.
        const auto push_times = [&]() {
            if (times_rows == times_cap) {
                const std::size_t new_cap = std::max<std::size_t>(2u * times_cap, 64u);
                double *nt = nullptr;
                HY_CUDA_CHECK(cudaMalloc(&nt, sizeof(double) * 2u * n * new_cap));
                if (d_times != nullptr) {
                    HY_CUDA_CHECK(cudaMemcpyAsync(nt, d_times, sizeof(double) * 2u * n * times_rows, cudaMemcpyDeviceToDevice,
                                                  sh->stream));
                    HY_CUDA_CHECK(cudaStreamSynchronize(sh->stream));
                    HY_CUDA_CHECK(cudaFree(d_times));
                }
                d_times = nt;
                times_cap = new_cap;
            }
            double *blk = d_times + 2u * n * times_rows;
            HY_CUDA_CHECK(cudaMemcpyAsync(blk, sh->d_t_hi, sizeof(double) * n, cudaMemcpyDeviceToDevice, sh->stream));
            HY_CUDA_CHECK(cudaMemcpyAsync(blk + n, sh->d_t_lo, sizeof(double) * n, cudaMemcpyDeviceToDevice, sh->stream));
            ++times_rows;
        };
        push_times();
        sh->ensure_tc();
        own_tc = sh->d_tc;
        tc_swapped = true;
        HY_CUDA_CHECK(cudaMemsetAsync(d_pflags, 0, sizeof(hflags), sh->stream));
        dev::k_prop_init<<<gb, 128, 0, sh->stream>>>(sh->view(), G, sh->d_prop_min_h, sh->d_prop_max_h, sh->d_prop_n_steps);
        HY_CUDA_CHECK(cudaGetLastError());
        read_flags();
        if (hflags[2] != 0u) {
            throw std::invalid_argument("The final time passed to the propagate_until() function of an adaptive "
                                        "Taylor integrator in batch mode results in an overflow condition");
        }
        std::uint64_t iter = 0;
        while (true) {
            // The step kernel writes the coefficients of this iteration straight into their slot of the recording.
            if (iter / co->slab_iters == co->slabs.size()) {
                double *slab = nullptr;
                HY_CUDA_CHECK(cudaMalloc(&slab, sizeof(double) * tc_doubles * co->slab_iters));
                co->slabs.push_back(slab);
            }
            sh->d_tc = co->slabs[iter / co->slab_iters] + (iter % co->slab_iters) * tc_doubles;
            dev::run_args R{};
            R.max_delta_t = G.dt_limit;
            R.default_max_delta_t = std::numeric_limits<double>::infinity();
            R.write_tc = 1;
            R.flags = sh->d_flags;
            R.counter = sh->d_counter;
            sh->launch(false, R);
            HY_CUDA_CHECK(cudaMemsetAsync(d_pflags, 0, sizeof(unsigned) * 2u, sh->stream));
            dev::k_prop_book<<<gb, 128, 0, sh->stream>>>(sh->view(), G, sh->d_prop_outcome, sh->d_prop_min_h,
                                                         sh->d_prop_max_h, sh->d_prop_n_steps);
            HY_CUDA_CHECK(cudaGetLastError());
            read_flags();
            if (hflags[1] != 0u) {
                break; // non-finite state: this iteration is not recorded (:1462-1467)
            }
            // update_c_out(), :1320-1346.
            push_times();
            ++iter;
            if (cb != nullptr) {
                // The step callback (:1476-1500), before the exit tests like in the reference.
                HY_CUDA_CHECK(cudaStreamSynchronize(sh->stream));
                const int r = cb(user);
                if (r < 0) {
                    throw callback_abort{};
                }
                if (r == 0) {
                    dev::k_fill_outcome<<<(n + 255u) / 256u, 256, 0, sh->stream>>>(sh->d_prop_outcome, n,
                                                                                  HY_OUTCOME_CB_STOP);
                    break;
                }
            }
            if (hflags[0] == n) {
                break; // every lane reached its final time
            }
            if (iter == max_steps) {
                dev::k_fill_outcome<<<(n + 255u) / 256u, 256, 0, sh->stream>>>(sh->d_prop_outcome, n,
                                                                              HY_OUTCOME_STEP_LIMIT);
                break;
            }
        }
        // The batch's own tc array ends up with the coefficients of the last step taken, like m_tc in the reference.
        HY_CUDA_CHECK(cudaMemcpyAsync(own_tc, sh->d_tc, sizeof(double) * tc_doubles, cudaMemcpyDeviceToDevice, sh->stream));
        sh->d_tc = own_tc;
        tc_swapped = false;
        if (iter != 0u) {
            // make_c_out(), :1277-1317: the times get a padding row, +-inf by direction.
            co->n_steps = iter;
            const std::size_t rows = iter + 2u;
            HY_CUDA_CHECK(cudaMalloc(&co->d_t_hi, sizeof(double) * rows * n));
            HY_CUDA_CHECK(cudaMalloc(&co->d_t_lo, sizeof(double) * rows * n));
            HY_CUDA_CHECK(cudaMalloc(&co->d_tm, sizeof(double) * n));
            HY_CUDA_CHECK(cudaMalloc(&co->d_out, sizeof(double) * static_cast<std::size_t>(sh->n_eq) * n));
            HY_CUDA_CHECK(cudaMemcpy2DAsync(co->d_t_hi, sizeof(double) * n, d_times, sizeof(double) * 2u * n,
                                            sizeof(double) * n, iter + 1u, cudaMemcpyDeviceToDevice, sh->stream));
            HY_CUDA_CHECK(cudaMemcpy2DAsync(co->d_t_lo, sizeof(double) * n, d_times + n, sizeof(double) * 2u * n,
                                            sizeof(double) * n, iter + 1u, cudaMemcpyDeviceToDevice, sh->stream));
            HY_CUDA_CHECK(cudaMalloc(&co->d_slabs, sizeof(double *) * co->slabs.size()));
            HY_CUDA_CHECK(cudaMemcpyAsync(co->d_slabs, co->slabs.data(), sizeof(double *) * co->slabs.size(),
                                          cudaMemcpyHostToDevice, sh->stream));
            std::vector<unsigned char> dir(n);
            HY_CUDA_CHECK(cudaMemcpyAsync(dir.data(), d_dir, n, cudaMemcpyDeviceToHost, sh->stream));
            HY_CUDA_CHECK(cudaStreamSynchronize(sh->stream));
            std::vector<double> pad(n), zero(n, 0.);
            for (std::uint32_t i = 0; i < n; ++i) {
                pad[i] = dir[i] != 0 ? std::numeric_limits<double>::infinity() : -std::numeric_limits<double>::infinity();
            }
            HY_CUDA_CHECK(cudaMemcpy(co->d_t_hi + (rows - 1u) * n, pad.data(), sizeof(double) * n, cudaMemcpyHostToDevice));
            HY_CUDA_CHECK(cudaMemcpy(co->d_t_lo + (rows - 1u) * n, zero.data(), sizeof(double) * n, cudaMemcpyHostToDevice));
            *out = co.release();
        }
        HY_CUDA_CHECK(cudaStreamSynchronize(sh->stream));
        cleanup();
        return HY_OK;
    } catch (const callback_abort &) {
        cleanup();
        hy::detail::set_last_error("A host callback aborted the propagation");
        return HY_ERR_CALLBACK;
    } catch (...) {
        cleanup();
        return translate_exception();
    }
}

// A recording driven from OUTSIDE the library: the front ends' host lock-step loops (integrators with events, whose
// callbacks are host code: src/taylor_adaptive_batch.cpp:1372-1527 with update_c_out() at :1320-1346) append the Taylor
// coefficients and times of every iteration they complete.
struct hy_cout_rec {
    std::unique_ptr<hy_cout> co;
    double *d_times = nullptr; // rows of 2 * n doubles (hi, lo)
    std::size_t times_cap = 0, times_rows = 0, tc_doubles = 0;
    std::uint64_t iter = 0;
    ~hy_cout_rec()
    {
        if (d_times != nullptr) {
            cudaFree(d_times);
        }
    }
};

namespace
{

void rec_push_times(shard &sh, hy_cout_rec *r)
{
    const std::uint32_t n = sh.n;
    if (r->times_rows == r->times_cap) {
        const std::size_t new_cap = std::max<std::size_t>(2u * r->times_cap, 64u);
        double *nt = nullptr;
        HY_CUDA_CHECK(cudaMalloc(&nt, sizeof(double) * 2u * n * new_cap));
        if (r->d_times != nullptr) {
            HY_CUDA_CHECK(cudaMemcpyAsync(nt, r->d_times, sizeof(double) * 2u * n * r->times_rows, cudaMemcpyDeviceToDevice,
                                          sh.stream));
            HY_CUDA_CHECK(cudaStreamSynchronize(sh.stream));
            HY_CUDA_CHECK(cudaFree(r->d_times));
        }
        r->d_times = nt;
        r->times_cap = new_cap;
    }
    double *blk = r->d_times + 2u * n * r->times_rows;
    HY_CUDA_CHECK(cudaMemcpyAsync(blk, sh.d_t_hi, sizeof(double) * n, cudaMemcpyDeviceToDevice, sh.stream));
    HY_CUDA_CHECK(cudaMemcpyAsync(blk + n, sh.d_t_lo, sizeof(double) * n, cudaMemcpyDeviceToDevice, sh.stream));
    ++r->times_rows;
}

} // namespace

int hy_cout_rec_begin(hy_batch *b, hy_cout_rec **out)
{
    try {
        if (b == nullptr || out == nullptr) {
            throw std::invalid_argument("Null pointer passed to hy_cout_rec_begin()");
        }
        if (b->sharded) {
            throw hy::detail::not_implemented_error("Continuous output is not available on a multi-device batch");
        }
        *out = nullptr;
        shard &sh = *b->shards[0];
        device_guard guard(sh.device);
        auto r = std::make_unique<hy_cout_rec>();
        r->tc_doubles = static_cast<std::size_t>(sh.n_eq) * (sh.order + 1u) * sh.n;
        r->co = std::make_unique<hy_cout>();
        r->co->device = sh.device;
        r->co->n = sh.n;
        r->co->n_eq = sh.n_eq;
        r->co->order = sh.order;
        r->co->prog = sh.prog;
        r->co->stream = sh.stream;
        r->co->slab_iters = static_cast<std::uint32_t>(std::min<std::size_t>(
            std::max<std::size_t>((std::size_t(64) << 20) / (r->tc_doubles * sizeof(double)), 1u), 4096u));
        rec_push_times(sh, r.get()); // row 0: the starting time
        HY_CUDA_CHECK(cudaStreamSynchronize(sh.stream));
        *out = r.release();
        return HY_OK;
    } catch (...) {
        return translate_exception();
    }
}

int hy_cout_rec_append(hy_batch *b, hy_cout_rec *r)
{
    try {
        if (b == nullptr || r == nullptr || r->co == nullptr || b->sharded || r->co->n != b->n
            || b->shards[0]->d_tc == nullptr) {
            throw std::invalid_argument("Invalid arguments passed to hy_cout_rec_append() (the last step must have "
                                        "written its Taylor coefficients)");
        }
        shard &sh = *b->shards[0];
        device_guard guard(sh.device);
        auto &co = *r->co;
        if (r->iter / co.slab_iters == co.slabs.size()) {
            double *slab = nullptr;
            HY_CUDA_CHECK(cudaMalloc(&slab, sizeof(double) * r->tc_doubles * co.slab_iters));
            co.slabs.push_back(slab);
        }
        // (The rows of the state variables come first in the batch's tc array; those of event equations are not recorded.)
        HY_CUDA_CHECK(cudaMemcpyAsync(co.slabs[r->iter / co.slab_iters] + (r->iter % co.slab_iters) * r->tc_doubles, sh.d_tc,
                                      sizeof(double) * r->tc_doubles, cudaMemcpyDeviceToDevice, sh.stream));
        rec_push_times(sh, r);
        ++r->iter;
        return HY_OK;
    } catch (...) {
        return translate_exception();
    }
}

void hy_cout_rec_destroy(hy_cout_rec *r)
{
    delete r;
}

// make_c_out() (:1277-1317): forward[lane] != 0 for lanes integrated forwards in time (the padding row of the times is
// +-inf by direction). *out = NULL if nothing was recorded. The recorder is destroyed either way.
int hy_cout_rec_finish(hy_batch *b, hy_cout_rec *rp, const unsigned char *forward, hy_cout **out)
{
    std::unique_ptr<hy_cout_rec> r(rp);
    try {
        if (b == nullptr || rp == nullptr || forward == nullptr || out == nullptr) {
            throw std::invalid_argument("Null pointer passed to hy_cout_rec_finish()");
        }
        *out = nullptr;
        shard &sh = *b->shards[0];
        device_guard guard(sh.device);
        const std::uint32_t n = sh.n;
        const std::uint64_t iter = r->iter;
        if (iter != 0u) {
            auto &co = *r->co;
            co.n_steps = iter;
            const std::size_t rows = iter + 2u;
            HY_CUDA_CHECK(cudaMalloc(&co.d_t_hi, sizeof(double) * rows * n));
            HY_CUDA_CHECK(cudaMalloc(&co.d_t_lo, sizeof(double) * rows * n));
            HY_CUDA_CHECK(cudaMalloc(&co.d_tm, sizeof(double) * n));
            HY_CUDA_CHECK(cudaMalloc(&co.d_out, sizeof(double) * static_cast<std::size_t>(sh.n_eq) * n));
            HY_CUDA_CHECK(cudaMemcpy2DAsync(co.d_t_hi, sizeof(double) * n, r->d_times, sizeof(double) * 2u * n,
                                            sizeof(double) * n, iter + 1u, cudaMemcpyDeviceToDevice, sh.stream));
            HY_CUDA_CHECK(cudaMemcpy2DAsync(co.d_t_lo, sizeof(double) * n, r->d_times + n, sizeof(double) * 2u * n,
                                            sizeof(double) * n, iter + 1u, cudaMemcpyDeviceToDevice, sh.stream));
            HY_CUDA_CHECK(cudaMalloc(&co.d_slabs, sizeof(double *) * co.slabs.size()));
            HY_CUDA_CHECK(cudaMemcpyAsync(co.d_slabs, co.slabs.data(), sizeof(double *) * co.slabs.size(),
                                          cudaMemcpyHostToDevice, sh.stream));
            HY_CUDA_CHECK(cudaStreamSynchronize(sh.stream));
            std::vector<double> pad(n), zero(n, 0.);
            for (std::uint32_t i = 0; i < n; ++i) {
                pad[i] = forward[i] != 0 ? std::numeric_limits<double>::infinity() : -std::numeric_limits<double>::infinity();
            }
            HY_CUDA_CHECK(cudaMemcpy(co.d_t_hi + (rows - 1u) * n, pad.data(), sizeof(double) * n, cudaMemcpyHostToDevice));
            HY_CUDA_CHECK(cudaMemcpy(co.d_t_lo + (rows - 1u) * n, zero.data(), sizeof(double) * n, cudaMemcpyHostToDevice));
            *out = r->co.release();
        }
        HY_CUDA_CHECK(cudaStreamSynchronize(sh.stream));
        return HY_OK;
    } catch (...) {
        return translate_exception();
    }
}

int hy_cout_eval(hy_cout *c, const double *tm, double *out)
{
    try {
        if (c == nullptr || tm == nullptr || out == nullptr) {
            throw std::invalid_argument("Null pointer passed to hy_cout_eval()");
        }
        for (std::uint32_t i = 0; i < c->n; ++i) {
            if (!std::isfinite(tm[i])) {
                throw std::invalid_argument("Cannot compute the continuous output in batch mode for the batch index "
                                            + std::to_string(i) + " at the non-finite time "
                                            + hy::detail::fmt_double(tm[i]));
            }
        }
        device_guard guard(c->device);
        HY_CUDA_CHECK(cudaMemcpyAsync(c->d_tm, tm, sizeof(double) * c->n, cudaMemcpyHostToDevice, c->stream));
        dev::k_cout_eval<<<(c->n + 127u) / 128u, 128, 0, c->stream>>>(
            c->prog, c->n, static_cast<std::uint32_t>(c->n_steps + 2u), c->d_slabs, c->slab_iters, c->d_t_hi, c->d_t_lo,
            c->d_tm, c->d_out);
        HY_CUDA_CHECK(cudaGetLastError());
        HY_CUDA_CHECK(cudaMemcpyAsync(out, c->d_out, sizeof(double) * static_cast<std::size_t>(c->n_eq) * c->n,
                                      cudaMemcpyDeviceToHost, c->stream));
        HY_CUDA_CHECK(cudaStreamSynchronize(c->stream));
        return HY_OK;
    } catch (...) {
        return translate_exception();
    }
}

int hy_cout_get_bounds(const hy_cout *c, double *lb, double *ub)
{
    try {
        if (c == nullptr || lb == nullptr || ub == nullptr) {
            throw std::invalid_argument("Null pointer passed to hy_cout_get_bounds()");
        }
        device_guard guard(c->device);
        HY_CUDA_CHECK(cudaMemcpy(lb, c->d_t_hi, sizeof(double) * c->n, cudaMemcpyDeviceToHost));
        HY_CUDA_CHECK(cudaMemcpy(ub, c->d_t_hi + c->n_steps * c->n, sizeof(double) * c->n, cudaMemcpyDeviceToHost));
        return HY_OK;
    } catch (...) {
        return translate_exception();
    }
}

int hy_cout_download(const hy_cout *c, double *times_hi, double *times_lo, double *tcs)
{
    try {
        if (c == nullptr) {
            throw std::invalid_argument("Null pointer passed to hy_cout_download()");
        }
        device_guard guard(c->device);
        const std::size_t n = c->n, rows = static_cast<std::size_t>(c->n_steps) + 2u;
        if (times_hi != nullptr) {
            HY_CUDA_CHECK(cudaMemcpy(times_hi, c->d_t_hi, sizeof(double) * rows * n, cudaMemcpyDeviceToHost));
        }
        if (times_lo != nullptr) {
            HY_CUDA_CHECK(cudaMemcpy(times_lo, c->d_t_lo, sizeof(double) * rows * n, cudaMemcpyDeviceToHost));
        }
        if (tcs != nullptr) {
            // One iteration = [n_eq][order + 1][batch] doubles; the slabs hold slab_iters iterations each, the last
            // one possibly fewer.
            const std::size_t it_doubles = static_cast<std::size_t>(c->n_eq) * (c->order + 1u) * n;
            for (std::size_t s = 0; s < c->slabs.size(); ++s) {
                const std::size_t first = s * c->slab_iters;
                if (first >= c->n_steps) {
                    break;
                }
                const std::size_t count = std::min<std::size_t>(c->slab_iters, c->n_steps - first);
                HY_CUDA_CHECK(cudaMemcpy(tcs + first * it_doubles, c->slabs[s], sizeof(double) * count * it_doubles,
                                         cudaMemcpyDeviceToHost));
            }
        }
        return HY_OK;
    } catch (...) {
        return translate_exception();
    }
}

uint64_t hy_cout_n_steps(const hy_cout *c)
{
    return c != nullptr ? c->n_steps : 0u;
}

void hy_cout_destroy(hy_cout *c)
{
    delete c;
}

int hy_batch_d_output(hy_batch *b, const double *tau, double *out)
{
    try {
        for_each_shard(b, [&](shard &sh, std::size_t off, std::size_t) {
            const double *d_tau = stage(sh, tau, off, 0);
            sh.ensure_tc();
            dev::k_d_output<<<(sh.n + 127u) / 128u, 128, 0, sh.stream>>>(sh.prog, sh.n, sh.d_tc, d_tau, sh.d_d_out);
            HY_CUDA_CHECK(cudaGetLastError());
            ++sh.n_launches;
            rows_d2h(sh, out, sh.d_d_out, sh.n_eq, b->n, off);
            HY_CUDA_CHECK(cudaStreamSynchronize(sh.stream));
        });
        return HY_OK;
    } catch (...) {
        return translate_exception();
    }
}

/* ---- E. events ---- */
int hy_batch_set_events(hy_batch *b, uint32_t n_te, const int32_t *dirs, const double *cooldowns, double tol)
{
    try {
        if (b == nullptr || dirs == nullptr || (n_te != 0u && cooldowns == nullptr)) {
            throw std::invalid_argument("Null pointer passed to hy_batch_set_events()");
        }
        // (Directions, cooldowns and tolerance are per event, not per lane: every shard gets them all.)
        each_shard_in_order(b, [&](shard &sh, std::size_t, std::size_t) {
            HY_CUDA_CHECK(cudaStreamSynchronize(sh.stream));
            sh.ev_setup(n_te, dirs, cooldowns, tol);
        });
        b->n_te = n_te;
        b->ev_set = true;
        b->ev_host.clear();
        return HY_OK;
    } catch (...) {
        return translate_exception();
    }
}

uint32_t hy_batch_n_events(const hy_batch *b)
{
    return b == nullptr ? 0u : static_cast<uint32_t>(b->ev_host.size());
}

int hy_batch_get_events(const hy_batch *b, hy_event_rec *out, uint32_t cap)
{
    if (b == nullptr || (out == nullptr && cap != 0u)) {
        hy::detail::set_last_error("Null pointer passed to hy_batch_get_events()");
        return HY_ERR_INVALID_ARG;
    }
    const std::size_t m = std::min<std::size_t>(cap, b->ev_host.size());
    std::copy(b->ev_host.begin(), b->ev_host.begin() + static_cast<std::ptrdiff_t>(m), out);
    return HY_OK;
}

int hy_batch_download_tc_events(hy_batch *b, double *out)
{
    try {
        if (b == nullptr || out == nullptr) {
            throw std::invalid_argument("Null pointer passed to hy_batch_download_tc_events()");
        }
        for_each_shard(b, [&](shard &sh, std::size_t off, std::size_t) {
            if (sh.n_ev == 0u || sh.d_tc == nullptr) {
                throw std::invalid_argument("No Taylor coefficients of event equations are available");
            }
            const std::size_t rows = static_cast<std::size_t>(sh.order + 1u) * sh.n_ev;
            rows_d2h(sh, out, sh.d_tc + static_cast<std::size_t>(sh.order + 1u) * sh.n * sh.n_eq, rows, b->n, off);
            HY_CUDA_CHECK(cudaStreamSynchronize(sh.stream));
        });
        return HY_OK;
    } catch (...) {
        return translate_exception();
    }
}

int hy_batch_reset_cooldowns(hy_batch *b, int64_t lane)
{
    try {
        if (b == nullptr) {
            throw std::invalid_argument("Null batch");
        }
        if (!b->ev_set) {
            throw std::invalid_argument("No events are defined for this integrator");
        }
        if (lane >= static_cast<int64_t>(b->n)) {
            throw std::invalid_argument("Cannot reset the cooldowns at batch index " + std::to_string(lane)
                                        + ": the batch size for this integrator is only " + std::to_string(b->n));
        }
        each_shard_in_order(b, [&](shard &sh, std::size_t off, std::size_t) {
            const auto lo = static_cast<int64_t>(off), hi = lo + static_cast<int64_t>(sh.n);
            const std::size_t m = static_cast<std::size_t>(b->n_te) * sh.n;
            if (m != 0u && (lane < 0 || (lane >= lo && lane < hi))) {
                dev::k_ev_reset_cd<<<static_cast<unsigned>((m + 255u) / 256u), 256, 0, sh.stream>>>(
                    sh.eva, sh.n, lane < 0 ? 0xffffffffu : static_cast<std::uint32_t>(lane - lo));
                HY_CUDA_CHECK(cudaGetLastError());
            }
        });
        return HY_OK;
    } catch (...) {
        return translate_exception();
    }
}

int hy_batch_get_cooldowns(hy_batch *b, uint8_t *active, double *spent, double *cooldown)
{
    try {
        if (b == nullptr || !b->ev_set) {
            throw std::invalid_argument("No events are defined for this integrator");
        }
        // [n_te][batch] arrays: every shard fills its columns.
        each_shard_in_order(b, [&](shard &sh, std::size_t off, std::size_t) {
            const std::size_t m = static_cast<std::size_t>(b->n_te) * sh.n;
            std::vector<double> cd(2u * m);
            if (m != 0u) {
                rows_d2h(sh, active, sh.eva.cd_on, b->n_te, b->n, off);
                HY_CUDA_CHECK(cudaMemcpyAsync(cd.data(), sh.eva.cd, sizeof(double) * 2u * m, cudaMemcpyDeviceToHost,
                                              sh.stream));
            }
            HY_CUDA_CHECK(cudaStreamSynchronize(sh.stream));
            for (std::uint32_t k = 0; k < b->n_te; ++k) {
                for (std::uint32_t l = 0; l < sh.n; ++l) {
                    spent[static_cast<std::size_t>(k) * b->n + off + l] = cd[(static_cast<std::size_t>(k) * 2u) * sh.n + l];
                    cooldown[static_cast<std::size_t>(k) * b->n + off + l]
                        = cd[(static_cast<std::size_t>(k) * 2u + 1u) * sh.n + l];
                }
            }
        });
        return HY_OK;
    } catch (...) {
        return translate_exception();
    }
}

int hy_batch_set_cooldowns(hy_batch *b, const uint8_t *active, const double *spent, const double *cooldown)
{
    try {
        if (b == nullptr || !b->ev_set) {
            throw std::invalid_argument("No events are defined for this integrator");
        }
        if (b->n_te != 0u && (active == nullptr || spent == nullptr || cooldown == nullptr)) {
            throw std::invalid_argument("Null pointer passed to hy_batch_set_cooldowns()");
        }
        each_shard_in_order(b, [&](shard &sh, std::size_t off, std::size_t) {
            const std::size_t m = static_cast<std::size_t>(b->n_te) * sh.n;
            if (m != 0u) {
                std::vector<double> cd(2u * m);
                for (std::uint32_t k = 0; k < b->n_te; ++k) {
                    for (std::uint32_t l = 0; l < sh.n; ++l) {
                        cd[(static_cast<std::size_t>(k) * 2u) * sh.n + l] = spent[static_cast<std::size_t>(k) * b->n + off + l];
                        cd[(static_cast<std::size_t>(k) * 2u + 1u) * sh.n + l]
                            = cooldown[static_cast<std::size_t>(k) * b->n + off + l];
                    }
                }
                rows_h2d(sh, sh.eva.cd_on, active, b->n_te, b->n, off);
                HY_CUDA_CHECK(cudaMemcpyAsync(sh.eva.cd, cd.data(), sizeof(double) * 2u * m, cudaMemcpyHostToDevice,
                                              sh.stream));
                HY_CUDA_CHECK(cudaStreamSynchronize(sh.stream));
            }
        });
        return HY_OK;
    } catch (...) {
        return translate_exception();
    }
}

int hy_batch_launch_count(const hy_batch *b, uint64_t *n_launches)
{
    if (b == nullptr || n_launches == nullptr) {
        hy::detail::set_last_error("Null pointer passed to hy_batch_launch_count()");
        return HY_ERR_INVALID_ARG;
    }
    *n_launches = 0u;
    for (const auto &sh : b->shards) {
        *n_launches += sh->n_launches;
    }
    return HY_OK;
}

} // extern "C"
