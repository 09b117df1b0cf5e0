// Federated GLM log-likelihood + gradient on the 5th-gen tensor cores (tcgen05 + TMEM + TMA).
//
// Per 128-row tile of the bf16 design matrix X (read from HBM exactly ONCE per evaluation):
//
//   TMA        X[128 x P] -> smem, 128B-swizzled 64-feature panels (cp.async.bulk.tensor)
//   MMA #1     eta[128 x N1] = X_tile (A, K-major) . Theta^T (B, K-major)      -> TMEM
//              Theta holds, per MCMC chain, a 3-way bf16 split (hi, mid, lo) of the fp32
//              coefficients, so eta keeps ~fp32 accuracy although the operands are bf16.
//   epilogue   tcgen05.ld eta; link + log-likelihood; residual r = dll/deta;
//              r is split into (hi, lo) bf16 and stored to smem as the B operand of MMA #2
//   MMA #2     G[P x N2] += X_tile^T (A, **MN-major view of the very same smem tile**) . R
//              accumulated in TMEM across tiles, flushed to fp64 registers every kFlush tiles
//
// so the gradient GEMM costs no second pass over X.  Chains are batched along N (the MMA is
// otherwise idle: the kernel is HBM-bound), which is what makes tensor cores pay here.
// Roles: warp 0 = TMA producer, warp 1 = MMA #1 issuer, warps 2-5 = epilogue, warp 6 = MMA #2
// issuer (separate issuers so the gradient MMA of tile t never queues behind the TMA of tile t+1).
// The federation prologue/epilogue (theta broadcast, NVLink reduce) is fed_comm.cuh.
//
// Workload: BASELINE.json "federated logistic GLM, 10M rows x 256 features per shard, bf16".
// Nothing comparable exists in the reference (its model is /root/reference/demo_node.py:31-43).
#include <vector>

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "fed_comm.cuh"
#include "models.h"
#include "tc_common.cuh"
#include "chunks.h"

namespace tc {

constexpr int kTileM = 128;          // rows per tile (UMMA M for MMA #1, UMMA K-extent for MMA #2)
constexpr int kPanel = 64;           // features per 128-byte swizzle span
constexpr int kPanelBytes = kTileM * 128;  // 16 KB
// warps: 0 TMA, 1 MMA#1 issuer, 2-5 epilogue group 0, 6 MMA#2 issuer, 7.. further epilogue groups
constexpr int kMaxChunk = 32;        // tiles per chunk at most (= tiles accumulated in TMEM in fp32 before a flush)
constexpr int kMinChunk = 4;
constexpr int kRing = 16;            // published chunks the consumers may lag behind (needs only ~3)
constexpr int kLLRows = 16;          // epilogue warps at most (per-warp log-likelihood slots)

struct SmemLayout {
    uint32_t stages, stage_bytes, off_theta_b, theta_b_bytes, off_r, r_bytes, off_theta_f, off_icpt, off_phi, off_ring,
        off_bars, off_tmem, total, preload;
};
// r_bufs: residual (R) buffers between the epilogue and MMA #2 — 2 normally; 1 for 16 chains, where the 8 KB
// buy the third TMA stage (the epilogue of 16 chains is long enough to hide the short MMA #2 it then waits for).
// phi_bytes: the per-chain PhiChain table of the families with fitted parameters (0 otherwise).
__host__ __device__ inline SmemLayout smem_layout(int P, int n1, int n2, int n_theta, int n_groups, int chains, int r_bufs,
                                                 int phi_bytes = 0) {
    SmemLayout L;
    const uint32_t panels = P / kPanel;
    L.stage_bytes = panels * kPanelBytes;
    L.theta_b_bytes = panels * n1 * 128;
    L.r_bytes = kTileM * n2 * 2;
    // theta (fp32) is staged inside the TMA stage ring and is dead once the bf16 B operand and the intercept
    // table are built, so it costs no shared memory of its own.
    const uint32_t fixed = L.theta_b_bytes + r_bufs * L.r_bytes + ((chains * n_groups * 4 + 15) & ~15) + ((phi_bytes + 15) & ~15) +
                           kRing * 24 + 192 + 64 + 1024 /*alignment slack*/;
    uint32_t stages = (227u * 1024u - fixed) / L.stage_bytes;
    if (stages > 4) stages = 4;
    L.stages = stages;
    uint32_t o = stages * L.stage_bytes;
    L.off_theta_b = o; o += L.theta_b_bytes;
    L.off_r = o; o += r_bufs * L.r_bytes;
    // theta (fp32) sits in the LAST stage when it fits into one: the TMA warp fills the first stages - 1 stages
    // with this CTA's first tiles BEFORE theta has arrived (`preload`), the last stage is free once the B
    // operand is built.  (larger theta: stage 0 onwards, needs n_theta * 4 <= stages * stage_bytes, no preload)
    const bool theta_in_last = (uint32_t)n_theta * 4u <= L.stage_bytes && stages >= 2;
    L.off_theta_f = theta_in_last ? (stages - 1) * L.stage_bytes : 0;
    L.preload = theta_in_last ? stages - 1 : 0;
    L.off_icpt = o; o += (chains * n_groups * 4 + 15) & ~15;
    L.off_phi = o; o += (phi_bytes + 15) & ~15;
    L.off_ring = o; o += kRing * 24;   // published chunks + one mbarrier per ring slot
    L.off_bars = o; o += 192;
    L.off_tmem = o; o += 64;
    L.total = o + 1024;
    return L;
}

// KC = chains per launch.  N1 = pad16(3 KC) eta columns, N2 = pad16(2 KC) residual columns.
template <int KC>
struct Cfg {
    static constexpr int N1 = ((3 * KC + 15) / 16) * 16;
    static constexpr int N2 = ((2 * KC + 15) / 16) * 16;
    // Epilogue warp groups (128 threads each).  The per-tile epilogue is a serial chain, so it is
    // parallelised two ways: EGC groups split the chains of a tile (KC >= 4), and EGT = 2 groups
    // ping-pong on alternate tiles so that two tiles' chains overlap.  Group g: chains of
    // cg = g % EGC, tiles of parity tp = g / EGC.
    static constexpr int EGC = KC >= 4 ? 2 : 1;
    static constexpr int EGT = 2;
    static constexpr int EG = EGC * EGT;
    static constexpr int KH = KC / EGC;                 // chains per group
    static constexpr int kArrive = 128 * EGC;           // arrivals per eta/R/G barrier phase
    static constexpr int kThreads = 224 + (EG - 1) * 128;
    static constexpr int RB = KC >= 16 ? 1 : 2;         // R buffers (see smem_layout)
};

// doubles per CTA row of the partial array: (hi, lo) pairs of the n_vals outputs, then the per-warp slots of
// the values that a whole warp contributes to — [kLLRows][n_out][KC][1 + G + D]: log-likelihood, the G
// intercept gradients and the D family-parameter gradients of every (output block, chain)
__host__ __device__ constexpr size_t partial_row_doubles(int n_vals, int kc, int n_out, int n_groups, int n_family_params = 0) {
    return 2 * ((size_t)n_vals + (size_t)kLLRows * n_out * kc * (1 + n_groups + n_family_params));
}

// (hi, lo) += x on a pair that only this thread touches during the launch
__device__ __forceinline__ void dd_accumulate(double* slot, double x) {
    double2 cur = *reinterpret_cast<double2*>(slot);
    fed::dd_add(cur.x, cur.y, x, 0.0);
    *reinterpret_cast<double2*>(slot) = cur;
}

// Work is handed out in CHUNKS of consecutive tiles of one segment (host-built table: 32 tiles while much
// work is left, shrinking to 4 towards the end; always an even number, a segment with an odd tile count
// gets one empty tile).  The TMA warp claims chunks from a global counter and publishes them to the other
// roles through a small shared-memory ring, so CTAs on faster SMs simply take more chunks: no CTA waits on
// a statically assigned straggler.  Everything a chunk contributes (fp32 TMEM accumulation over its tiles,
// per-thread fp32 sums) depends on the chunk alone, and chunk results are combined as double-double pairs
// (fed::dd_add), so the evaluation stays reproducible although the assignment is not.
//
// kPhi: the families with fitted parameters (normal, student_t, negative_binomial; tc_common.cuh), selected at
// run time among themselves.  theta = [intercept[G], beta[P], phi[D]] and the result [LL, gi[G], g[P], dphi[D]] per
// chain; the D gradients fold exactly like LL.  A separate instantiation, so the other families keep their code.
template <int KC, bool kPhi>
__global__ void __launch_bounds__(Cfg<KC>::kThreads, 1)
fed_glm_tc_kernel(FedComm comm, const GlmSegment* __restrict__ segs_g, GlmParams prm, const CUtensorMap* __restrict__ tmaps,
                  const GlmChunk* __restrict__ chunks, int n_chunks, unsigned int* __restrict__ work_counter) {
    constexpr int N1 = Cfg<KC>::N1;
    constexpr int N2 = Cfg<KC>::N2;
    constexpr int EG = Cfg<KC>::EG;
    constexpr int KH = Cfg<KC>::KH;
    constexpr int EGC = Cfg<KC>::EGC;
    constexpr int kArrive = Cfg<KC>::kArrive;
    constexpr int RB = Cfg<KC>::RB;
    static_assert(Cfg<KC>::EGT == 2, "tile parity <-> eta / R buffer");
    static_assert(EG * 4 <= kLLRows, "per-warp LL slots");
    extern __shared__ unsigned char smem_dyn[];
    // 1 KB alignment (128B-swizzled TMA tiles) by offsetting INSIDE the shared array: the pointer keeps its
    // shared address space, so the compiler emits LDS / STS instead of generic LD / ST for everything below
    unsigned char* smem = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);

    const int P = prm.n_features;     // real number of features (theta / result layout)
    const int PP = (P + 127) & ~127;  // features the tile is padded to: TMA zero-fills the columns past P, their
                                      // Theta rows are zero and their gradient rows are never stored
    const int G = prm.n_groups;
    const int NH = PP / 128;          // 128-feature halves (UMMA M of MMA #2)
    const int panels = PP / kPanel;
    const SmemLayout L = smem_layout(PP, N1, N2, comm.n_theta, G, KC, RB, kPhi ? KC * (int)sizeof(PhiChain) : 0);
    const int S = (int)L.stages;
    const int nch = prm.n_chains < KC ? prm.n_chains : KC;  // chains actually present in theta
    const int D = kPhi ? prm.n_family_params : 0;
    const int TS = G + P + D;         // theta per chain: [intercept[G], beta[P], phi[D]]
    const int NV1 = 1 + G + P + D;    // outputs per chain: [LL, gi[G], g[P], dphi[D]]

    unsigned char* theta_b = smem + L.off_theta_b;
    unsigned char* r_buf = smem + L.off_r;
    float* theta_f = reinterpret_cast<float*>(smem + L.off_theta_f);  // valid until the setup barrier only
    float* icpt = reinterpret_cast<float*>(smem + L.off_icpt);        // [KC][G] intercepts
    PhiChain* phi_tab = reinterpret_cast<PhiChain*>(smem + L.off_phi); // [KC] (kPhi only)
    int4* ring = reinterpret_cast<int4*>(smem + L.off_ring);          // (segment or -1, first row, tiles, -)
    uint64_t* bar_ring = reinterpret_cast<uint64_t*>(smem + L.off_ring + kRing * 16);   // slot j % kRing: chunk j published
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L.off_bars);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + L.off_tmem);
    uint64_t* bar_full = bars;            // [4]
    uint64_t* bar_empty = bars + 4;       // [4]
    uint64_t* bar_eta_full = bars + 8;    // [2]
    uint64_t* bar_eta_empty = bars + 10;  // [2]
    uint64_t* bar_r_full = bars + 12;     // [2]
    uint64_t* bar_r_empty = bars + 14;    // [2]
    uint64_t* bar_g_full = bars + 16;     // [2]
    uint64_t* bar_g_empty = bars + 18;    // [2]

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    constexpr uint32_t kTmemCols = (2 * N1 + 2 * 4 * N2) <= 128 ? 128 : ((2 * N1 + 2 * 4 * N2) <= 256 ? 256 : 512);

    // ---------------- theta-independent setup: runs BEFORE the dependency wait inside fed::prologue, i.e. it
    // overlaps with the tail of the previous evaluation when launched with programmatic stream serialization
    for (int i = threadIdx.x; i < (int)(RB * L.r_bytes / 16); i += blockDim.x)
        reinterpret_cast<uint4*>(r_buf)[i] = make_uint4(0, 0, 0, 0);
    if (threadIdx.x == 0) {
        *pipeline_fault() = 0;
        for (int i = 0; i < kRing; ++i) mbar_init(&bar_ring[i], 1);
        for (int i = 0; i < 4; ++i) { mbar_init(&bar_full[i], 1); mbar_init(&bar_empty[i], 1); }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&bar_eta_full[i], 1);
            mbar_init(&bar_eta_empty[i], kArrive);
            mbar_init(&bar_r_full[i], kArrive);
            mbar_init(&bar_r_empty[i], 1);
            mbar_init(&bar_g_full[i], 1);
            mbar_init(&bar_g_empty[i], kArrive);
        }
        fence_barrier_init();
    }
    if (warp == 0 && lane == 0)
        for (int i = 0; i < prm.n_segments; ++i) tma_prefetch_desc(&tmaps[i]);
    if (warp == 1) tmem_alloc(tmem_slot, kTmemCols);
    // Early loads: X does not depend on theta.  The TMA warp waits for the previous evaluation to retire (its
    // last CTA re-arms the work counter), claims this CTA's first chunk and fills all stages but the one theta
    // is staged in, so the tensor core has `preload` tiles waiting when theta arrives (peers see theta several
    // microseconds after they became resident: root's PCIe read + the NVLink broadcast).
    unsigned int claim0 = 0;
    int preloaded = 0;
    if (warp == 0) {
        __syncwarp();   // lane 0's mbarrier inits
        fed::pdl_wait();
        if (lane == 0) claim0 = atomicAdd(work_counter, 1u);
        claim0 = __shfl_sync(0xffffffffu, claim0, 0);
        if (claim0 < (unsigned int)n_chunks) {
            const GlmChunk ch = chunks[claim0];
            preloaded = ch.n_tiles < (int)L.preload ? ch.n_tiles : (int)L.preload;
            if (!prm.early_loads) preloaded = 0;
            if (elect_one()) {
                for (int t = 0; t < preloaded; ++t) {
                    mbar_expect_tx(&bar_full[t], L.stage_bytes);
                    for (int pnl = 0; pnl < panels; ++pnl)
                        tma_load_2d(smem + (size_t)t * L.stage_bytes + pnl * kPanelBytes, &tmaps[ch.seg], pnl * kPanel,
                                    (ch.first_tile + t) * kTileM, &bar_full[t]);
                }
            }
            __syncwarp();
        }
    }
    tc_fence_before();

    fed::Prologue pro = fed::prologue(comm, theta_f);   // contains __syncthreads()
    const bool active = !pro.stop && !pro.timed_out;
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int NOUT = prm.n_out;       // output blocks (1 = everything summed; else one per node)
    const int NS1 = 1 + G + D;        // warp-level values per (block, chain): LL, the G intercept and D phi gradients
    const size_t row_doubles = partial_row_doubles(comm.n_vals, KC, NOUT, G, D);
    double* out = comm.cta_partials + (size_t)blockIdx.x * row_doubles;   // this CTA's running sums, (hi, lo) pairs
    double* ll_slots = out + 2 * (size_t)comm.n_vals;                     // [kLLRows][NOUT][KC][1 + G + D] pairs

    if (active) {
        // ---------------- theta-dependent setup --------------------------------------------------
        for (size_t i = threadIdx.x; i < row_doubles / 2; i += blockDim.x) reinterpret_cast<double2*>(out)[i] = make_double2(0.0, 0.0);
        for (int i = threadIdx.x; i < KC * G; i += blockDim.x)
            icpt[i] = (i / G) < nch ? theta_f[(i / G) * TS + (i % G)] : 0.f;
        if constexpr (kPhi) {
            for (int k = threadIdx.x; k < KC; k += blockDim.x)
                phi_tab[k] = k < nch ? phi_chain(prm.family, theta_f + k * TS + G + P) : PhiChain{0.0, 0.0, 0.0, {1.f, 1.f, 1.f, 1.f}};
        }
        // Theta^T as the K-major, 128B-swizzled B operand of MMA #1: row n = 3*chain + term
        for (int idx = threadIdx.x; idx < panels * N1 * 8; idx += blockDim.x) {
            const int j = idx & 7;              // 16-byte chunk (8 features) within the 128-byte row
            const int n = (idx >> 3) % N1;
            const int pnl = idx / (8 * N1);
            const int chain = n / 3, term = n % 3;
            uint32_t packed[4] = {0, 0, 0, 0};
            if (chain < nch) {
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    const int f = pnl * kPanel + j * 8 + e;
                    const float v = f < P ? theta_f[chain * TS + G + f] : 0.f;
                    const __nv_bfloat16 hi = __float2bfloat16_rn(v);
                    const float rem1 = v - __bfloat162float(hi);
                    const __nv_bfloat16 mid = __float2bfloat16_rn(rem1);
                    const __nv_bfloat16 lo = __float2bfloat16_rn(rem1 - __bfloat162float(mid));
                    const __nv_bfloat16 pick = term == 0 ? hi : (term == 1 ? mid : lo);
                    const uint32_t bits = (uint32_t)__bfloat16_as_ushort(pick);
                    packed[e >> 1] |= bits << ((e & 1) * 16);
                }
            }
            uint4* dst = reinterpret_cast<uint4*>(theta_b + pnl * (N1 * 128) + n * 128 + ((j ^ (n & 7)) * 16));
            *dst = make_uint4(packed[0], packed[1], packed[2], packed[3]);
        }
        fence_proxy_async();
        __syncthreads();
        if (threadIdx.x == 0) fed::stamp(comm, 2);
        const uint32_t tmem_eta = tmem_base;                 // 2 buffers x N1 columns
        const uint32_t tmem_g = tmem_base + 2 * N1;          // 2 buffers x NH x N2 columns

        // Consumers: the j-th chunk of this CTA, or x < 0 when the producer found the work counter exhausted.
        // (an mbarrier per ring slot: the producer arrives after writing the entry — release —, the consumers wait
        // on the slot's phase — acquire; slot j % kRing is reused every kRing chunks, consumers lag ~3 at most)
        auto next_chunk = [&](int j) -> int4 {
            mbar_wait(&bar_ring[j & (kRing - 1)], (uint32_t)((j / kRing) & 1));
            if (*pipeline_fault()) return make_int4(-1, 0, 0, 0);   // a stalled pipeline ends every role loop
            return ring[j & (kRing - 1)];
        };

        if (warp == 0) {
            // ================= TMA producer + chunk scheduler ==================================
            // The role loops are warp-uniform (all 32 lanes wait and count); only the issue is predicated on
            // elect.sync, so the compiler keeps addresses / descriptors in uniform registers.
            Ring stage;
            unsigned int claim = claim0, ahead = 0;   // the first chunk was claimed before theta arrived
            for (int j = 0;; ++j) {
                const bool have = claim < (unsigned int)n_chunks;
                GlmChunk ch{};
                if (have) ch = chunks[claim];
                if (lane == 0) {
                    ring[j & (kRing - 1)] = have ? make_int4(ch.seg, ch.first_tile * kTileM, ch.n_tiles, 0) : make_int4(-1, 0, 0, 0);
                    mbar_arrive(&bar_ring[j & (kRing - 1)]);
                    if (have) ahead = atomicAdd(work_counter, 1u);   // next claim: the round trip hides behind this chunk
                }
                __syncwarp();
                if (!have) break;
                for (int t = 0; t < ch.n_tiles; ++t) {
                    const int st = stage.idx;
                    if (j == 0 && t < preloaded) {   // already in flight (early loads)
                        stage.advance(S);
                        continue;
                    }
                    mbar_wait(&bar_empty[st], stage.phase ^ 1);
                    if (j == 0 && t == preloaded && lane == 0) fed::stamp(comm, 3);
                    const int row0 = (ch.first_tile + t) * kTileM;
                    unsigned char* dst = smem + (size_t)st * L.stage_bytes;
                    if (elect_one()) {
                        mbar_expect_tx(&bar_full[st], L.stage_bytes);
                        for (int pnl = 0; pnl < panels; ++pnl)
                            tma_load_2d(dst + pnl * kPanelBytes, &tmaps[ch.seg], pnl * kPanel, row0, &bar_full[st]);
                    }
                    __syncwarp();
                    stage.advance(S);
                }
                claim = __shfl_sync(0xffffffffu, ahead, 0);
            }
            if (lane == 0) fed::stamp(comm, 4);
        } else if (warp == 1) {
            // ================= MMA #1 issuer: eta = X . Theta^T ================================
            constexpr uint32_t idesc1 = make_idesc(128, N1, 0, 0);
            // descriptors: constant fields once, the 14-bit (address >> 4) field added per MMA
            const uint64_t desc_k = make_desc(0, 16, 1024, 2);
            const uint32_t theta_b_a4 = smem_u32(theta_b) >> 4;
            const uint32_t x_base_a4 = smem_u32(smem) >> 4;
            const uint32_t stage_a4 = L.stage_bytes >> 4;
            Ring stage, buf;   // TMA stages (S), eta buffers (2)
            for (int j = 0;; ++j) {
                const int4 ch = next_chunk(j);
                if (ch.x < 0) break;
                for (int t = 0; t < ch.z; ++t) {
                    mbar_wait(&bar_eta_empty[buf.idx], buf.phase ^ 1);
                    mbar_wait(&bar_full[stage.idx], stage.phase);
                    tc_fence_after();
                    const uint32_t x_a4 = x_base_a4 + (uint32_t)stage.idx * stage_a4;
                    const uint32_t d_eta = tmem_eta + buf.idx * N1;
                    if (elect_one()) {
                        for (int pnl = 0; pnl < panels; ++pnl) {
#pragma unroll
                            for (int ks = 0; ks < kPanel / 16; ++ks) {
                                const uint64_t adesc = desc_k | (uint64_t)(x_a4 + ((pnl * kPanelBytes + ks * 32) >> 4));
                                const uint64_t bdesc = desc_k | (uint64_t)(theta_b_a4 + ((pnl * (N1 * 128) + ks * 32) >> 4));
                                umma_bf16(d_eta, adesc, bdesc, idesc1, (pnl | ks) ? 1u : 0u);
                            }
                        }
                        umma_commit(&bar_eta_full[buf.idx]);
                    }
                    __syncwarp();
                    stage.advance(S);
                    buf.advance(2);
                }
            }
        } else if (warp == 6) {
            // ================= MMA #2 issuer: G += X^T . R ======================================
            constexpr uint32_t idesc2 = make_idesc(128, N2, 1, 1);
            constexpr uint32_t r_lbo = (N2 / 8) * 128;  // stride between 8-row K groups of R
            // A = X^T: MN-major (features contiguous), 128B swizzle.
            // LBO = stride between 64-feature panels, SBO = stride between 8-row groups.
            const uint64_t desc_x = make_desc(0, kPanelBytes, 1024, 2);
            // B = R: MN-major (chain columns contiguous), no swizzle.
            // LBO = stride between 8-row K groups, SBO = stride between 8-column groups.
            const uint64_t desc_r = make_desc(0, r_lbo, 128, 0);
            const uint32_t r_a4 = smem_u32(r_buf) >> 4;
            const uint32_t x_base_a4 = smem_u32(smem) >> 4;
            const uint32_t stage_a4 = L.stage_bytes >> 4;
            Ring stage, buf, gbuf;   // gbuf: TMEM gradient accumulator of the current chunk (2, alternating)
            for (int j = 0;; ++j) {
                const int4 ch = next_chunk(j);
                if (ch.x < 0) break;
                const int gb = gbuf.idx;
                mbar_wait(&bar_g_empty[gb], gbuf.phase ^ 1);   // the epilogue has drained this accumulator
                for (int t = 0; t < ch.z; ++t) {
                    const bool last = t == ch.z - 1;
                    mbar_wait(&bar_r_full[buf.idx], buf.phase);
                    tc_fence_after();
                    const uint32_t x_a4 = x_base_a4 + (uint32_t)stage.idx * stage_a4;
                    const uint32_t rb_a4 = r_a4 + (uint32_t)buf.idx * (L.r_bytes >> 4);
                    if (elect_one()) {
                        for (int h = 0; h < NH; ++h) {
#pragma unroll
                            for (int ks = 0; ks < kTileM / 16; ++ks) {
                                const uint64_t adesc = desc_x | (uint64_t)(x_a4 + (((2 * h) * kPanelBytes + ks * 2 * 1024) >> 4));
                                const uint64_t bdesc = desc_r | (uint64_t)(rb_a4 + ((ks * 2 * r_lbo) >> 4));
                                umma_bf16(tmem_g + (gb * NH + h) * N2, adesc, bdesc, idesc2, (t == 0 && ks == 0) ? 0u : 1u);
                            }
                        }
                        umma_commit(&bar_empty[stage.idx]);   // X stage may be refilled
                        // R may be rewritten.  Two buffers: one barrier per buffer.  One buffer: the tiles of
                        // the two epilogue groups alternate in it, and each group waits for the OTHER group's
                        // tile to be consumed — one barrier per tile parity, so that a group can never be two
                        // phases ahead of the barrier it waits on (parity waits alias after two phases).
                        umma_commit(&bar_r_empty[RB == 2 ? buf.idx : (t & 1)]);
                        if (last) umma_commit(&bar_g_full[gb]);
                    }
                    __syncwarp();
                    stage.advance(S);
                    buf.advance(RB);
                }
                gbuf.advance(2);
            }
        } else {
            // ================= epilogue warps: group 0 = warps 2-5, group g >= 1 = warps 7+4(g-1) .. =====
            const int eg = warp <= 5 ? 0 : (warp - 7) / 4 + 1;
            const int ew = eg * 4 + (warp <= 5 ? warp - 2 : (warp - 7) % 4);   // epilogue warp ordinal: LL slot row
            const int cg = eg % EGC;                // which chains
            const int tp = eg / EGC;                // which tile parity (chunks are even => also this group's eta/R buffer)
            const int q = warp & 3;                 // TMEM lane quarter this warp may access
            const int row = q * 32 + lane;          // row of the tile == TMEM lane
            const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
            const int k0 = cg * KH;                 // first chain of this group
            const uint32_t r_lbo = (N2 / 8) * 128;
            // columns fetched per request (power-of-two shapes; the surplus columns are allocated TMEM, ignored)
            constexpr int kEtaCols = KH == 1 ? 4 : (KH == 2 ? 8 : (KH == 4 ? 16 : 24));
            constexpr int kGCols = KH <= 2 ? 4 : (KH == 4 ? 8 : 16);
            constexpr bool kPrefetchSlots = KH <= 2;   // few enough registers to fetch the warp's slots a whole chunk early
            const int b = tp;                       // eta / R buffer of this group's tiles
            uint32_t bph = 0;                       // its phase: flips after every tile of this group
            Ring gbuf;
            for (int j = 0;; ++j) {
                const int4 ch = next_chunk(j);
                if (ch.x < 0) break;
                const float* __restrict__ seg_y = segs_g[ch.x].y;   // segment table: global, read once per chunk
                const long long seg_rows = segs_g[ch.x].n_rows;
                const int seg_group = segs_g[ch.x].group;
                const int og = segs_g[ch.x].out_group;               // output block of this chunk's segment
                // this warp's (hi, lo) slots of the chunk's output block: LL at +0, intercept gradient g at +(1 + g)
                double* slot0 = ll_slots + 2 * ((((size_t)ew * NOUT + og) * KC + k0) * NS1);
                double2 pre_l[kPrefetchSlots ? KH : 1], pre_g[kPrefetchSlots ? KH : 1];
                if constexpr (kPrefetchSlots) {
                    if (lane == 0) {
#pragma unroll
                        for (int k = 0; k < KH; ++k)
                            if ((k0 + k) < nch) {
                                pre_l[k] = *reinterpret_cast<const double2*>(slot0 + 2 * (size_t)k * NS1);
                                pre_g[k] = *reinterpret_cast<const double2*>(slot0 + 2 * (size_t)k * NS1 + 2 * (1 + seg_group));
                            }
                    }
                }
                float ll_acc[KH], gi_cur[KH];
                float ph_acc[kPhi ? KH : 1][2];   // row parts of dLL/dphi (kPhi)
#pragma unroll
                for (int k = 0; k < KH; ++k) ll_acc[k] = gi_cur[k] = 0.f;
                if constexpr (kPhi) {
#pragma unroll
                    for (int k = 0; k < KH; ++k) ph_acc[k][0] = ph_acc[k][1] = 0.f;
                }
                for (int t = tp; t < ch.z; t += 2) {
                    const long long grow = (long long)ch.y + (long long)t * kTileM + row;
                    const bool valid = grow < seg_rows;
                    const float y = valid ? __ldg(seg_y + grow) : 0.f;

                    mbar_wait(&bar_eta_full[b], bph);
                    tc_fence_after();
                    float ev[kEtaCols];
                    tmem_ld_cols<kEtaCols>(tmem_eta + lane_addr + b * N1 + 3 * k0, ev);   // one TMEM round trip
                    tc_fence_before();
                    mbar_arrive(&bar_eta_empty[b]);

                    // link, likelihood, residual -> (hi, lo) bf16 columns of R
                    uint32_t rpk[KH];
#pragma unroll
                    for (int k = 0; k < KH; ++k) {
                        const float eta = (ev[3 * k] + ev[3 * k + 1]) + ev[3 * k + 2];
                        float ll = 0.f, r = 0.f;
                        if constexpr (kPhi) {
                            float d0 = 0.f, d1 = 0.f;
                            if (valid && (k0 + k) < nch)
                                link_loglik_phi(prm.family, y, eta + icpt[(k0 + k) * G + seg_group], phi_tab[k0 + k].p, ll, r, d0, d1);
                            ph_acc[k][0] += d0;
                            ph_acc[k][1] += d1;
                        } else {
                            if (valid && (k0 + k) < nch)
                                link_loglik(prm.family, y, eta + icpt[(k0 + k) * G + seg_group], ll, r);
                        }
                        ll_acc[k] += ll;
                        gi_cur[k] += r;
                        const __nv_bfloat16 hi = __float2bfloat16_rn(r);
                        const __nv_bfloat16 lo = __float2bfloat16_rn(r - __bfloat162float(hi));
                        rpk[k] = (uint32_t)__bfloat16_as_ushort(hi) | ((uint32_t)__bfloat16_as_ushort(lo) << 16);
                    }
                    // R buffer of this tile: with two buffers the group's own; with one, every tile of the CTA uses it
                    const int rb = RB == 2 ? b : 0;
                    if constexpr (RB == 2) {
                        mbar_wait(&bar_r_empty[b], bph ^ 1);
                    } else {
                        // wait until MMA #2 has consumed the previous tile (the other group's): for group 0 that is
                        // the (m)-th commit on the odd barrier before its m-th tile, for group 1 the (m+1)-th on the even
                        mbar_wait(&bar_r_empty[tp ^ 1], tp == 0 ? (bph ^ 1) : bph);
                    }
                    {
                        // chain k owns columns (2k, 2k+1): 4 bytes at (k / 4) * 128 + (k % 4) * 4 of the row
                        unsigned char* rrow = r_buf + rb * L.r_bytes + (row >> 3) * r_lbo + (row & 7) * 16;
                        if constexpr (KH == 8) {
                            *reinterpret_cast<uint4*>(rrow + (k0 / 4) * 128) = make_uint4(rpk[0], rpk[1], rpk[2], rpk[3]);
                            *reinterpret_cast<uint4*>(rrow + (k0 / 4 + 1) * 128) = make_uint4(rpk[4], rpk[5], rpk[6], rpk[7]);
                        } else if constexpr (KH == 4) {
                            *reinterpret_cast<uint4*>(rrow + (k0 / 4) * 128) = make_uint4(rpk[0], rpk[1], rpk[2], rpk[3]);
                        } else if constexpr (KH == 2) {
                            *reinterpret_cast<uint2*>(rrow + (k0 / 4) * 128 + (k0 % 4) * 4) = make_uint2(rpk[0], rpk[1]);
                        } else {
                            *reinterpret_cast<uint32_t*>(rrow + (k0 / 4) * 128 + (k0 % 4) * 4) = rpk[0];
                        }
                    }
                    fence_proxy_async();
                    mbar_arrive(&bar_r_full[rb]);
                    bph ^= 1u;
                }
                // ---- end of the chunk for this group: fold its sums into the CTA's running pairs ----------
                // per-thread fp32 sums over the chunk's tiles -> fixed butterfly over the warp (double) ->
                // lane 0 adds the warp's value to its own slot: every step depends on the chunk only.
                // The slots live in L2: all their loads are issued together (KH <= 2: already at the start of the
                // chunk, see `pre`), so the chunk boundary costs one round trip at most, not 2 KH.
                constexpr int kBatch = KH <= 4 ? KH : 4;   // chains whose slots are in flight together (register budget)
#pragma unroll
                for (int kb = 0; kb < KH; kb += kBatch) {
                    double lsum[kBatch], gsum[kBatch];
#pragma unroll
                    for (int k = 0; k < kBatch; ++k) {
                        lsum[k] = (double)ll_acc[kb + k];
                        gsum[k] = (double)gi_cur[kb + k];
#pragma unroll
                        for (int o = 16; o > 0; o >>= 1) {
                            lsum[k] += __shfl_xor_sync(0xffffffffu, lsum[k], o);
                            gsum[k] += __shfl_xor_sync(0xffffffffu, gsum[k], o);
                        }
                    }
                    if (lane == 0) {
                        double2 cl[kBatch], cg[kBatch];
#pragma unroll
                        for (int k = 0; k < kBatch; ++k) {
                            if constexpr (kPrefetchSlots) {
                                cl[k] = pre_l[kb + k];
                                cg[k] = pre_g[kb + k];
                            } else if ((k0 + kb + k) < nch) {
                                const double* slot = slot0 + 2 * (size_t)(kb + k) * NS1;
                                cl[k] = *reinterpret_cast<const double2*>(slot);
                                cg[k] = *reinterpret_cast<const double2*>(slot + 2 * (1 + seg_group));
                            }
                        }
#pragma unroll
                        for (int k = 0; k < kBatch; ++k)
                            if ((k0 + kb + k) < nch) {
                                double* slot = slot0 + 2 * (size_t)(kb + k) * NS1;
                                fed::dd_add(cl[k].x, cl[k].y, lsum[k], 0.0);
                                fed::dd_add(cg[k].x, cg[k].y, gsum[k], 0.0);
                                *reinterpret_cast<double2*>(slot) = cl[k];
                                *reinterpret_cast<double2*>(slot + 2 * (1 + seg_group)) = cg[k];
                            }
                    }
                }
                if constexpr (kPhi) {
                    // dphi: the same fixed butterfly and the same per-warp slots (+ 1 + G + j).  The per-chain
                    // constants of LL and dphi enter once per chunk, as (valid rows of the chunk) x c in fp64, from
                    // the first warp of the chunk's even-tile group of these chains.
                    const bool const_warp = tp == 0 && (ew & 3) == 0;
                    const long long left = seg_rows - (long long)ch.y, span = (long long)ch.z * kTileM;
                    const double n_valid = (double)(left < 0 ? 0 : (left < span ? left : span));
#pragma unroll
                    for (int k = 0; k < KH; ++k) {
                        double s0 = (double)ph_acc[k][0], s1 = (double)ph_acc[k][1];
#pragma unroll
                        for (int o = 16; o > 0; o >>= 1) {
                            s0 += __shfl_xor_sync(0xffffffffu, s0, o);
                            s1 += __shfl_xor_sync(0xffffffffu, s1, o);
                        }
                        if (lane == 0 && (k0 + k) < nch) {
                            double* slot = slot0 + 2 * (size_t)k * NS1;
                            const PhiChain& pc = phi_tab[k0 + k];
                            dd_accumulate(slot + 2 * (1 + G), s0);
                            if (D > 1) dd_accumulate(slot + 2 * (2 + G), s1);
                            if (const_warp) {
                                dd_accumulate(slot, n_valid * pc.c_ll);
                                dd_accumulate(slot + 2 * (1 + G), n_valid * pc.c_d0);
                                if (D > 1) dd_accumulate(slot + 2 * (2 + G), n_valid * pc.c_d1);
                            }
                        }
                    }
                }
                // gradient: the group that handled the chunk's last tile (odd index) drains the TMEM accumulator
                if (tp == 1) {
                    const int gb = gbuf.idx;
                    mbar_wait(&bar_g_full[gb], gbuf.phase);
                    tc_fence_after();
                    // one 128-feature half at a time keeps 16 values live instead of 64; the running pairs live in
                    // this CTA's row of the partial array (L2): one thread owns each of them
#pragma unroll
                    for (int h = 0; h < 4; ++h)
                        if (h < NH) {
                            float gv[kGCols];
                            tmem_ld_cols<kGCols>(tmem_g + lane_addr + (gb * NH + h) * N2 + 2 * k0, gv);
                            if (h == NH - 1) {
                                tc_fence_before();
                                mbar_arrive(&bar_g_empty[gb]);   // MMA #2 may start the chunk after next in this buffer
                            }
                            const bool real = h * 128 + row < P;   // rows of the padding carry zeros: nothing to add
                            double2 cur[KH];
#pragma unroll
                            for (int k = 0; k < KH; ++k)
                                cur[k] = ((k0 + k) < nch && real)
                                             ? *reinterpret_cast<const double2*>(out + 2 * (((size_t)og * nch + k0 + k) * NV1 + 1 + G + h * 128 + row))
                                             : make_double2(0.0, 0.0);
#pragma unroll
                            for (int k = 0; k < KH; ++k) {
                                fed::dd_add(cur[k].x, cur[k].y, (double)gv[2 * k] + (double)gv[2 * k + 1], 0.0);
                                if ((k0 + k) < nch && real)
                                    *reinterpret_cast<double2*>(out + 2 * (((size_t)og * nch + k0 + k) * NV1 + 1 + G + h * 128 + row)) = cur[k];
                            }
                        }
                }
                gbuf.advance(2);
            }
        }

        // ---------------- CTA partial: fold the per-warp LL slots and the intercept gradients ----------
        tc_fence_before();
        __syncthreads();
        tc_fence_after();
        fed::pdl_trigger();   // the next evaluation's CTA may take this SM as soon as we exit
        if (threadIdx.x == 0) fed::stamp(comm, 5);
        // layout per (output block, chain): [LL, gi[G], g[P], dphi[D]] as (hi, lo) pairs; g[] was accumulated in
        // place, LL, gi[] and dphi[] are the per-warp slots summed in warp order (slot 1 + G + j -> output 1 + G + P + j)
        for (int i = threadIdx.x; i < NOUT * nch * NS1; i += blockDim.x) {
            const int j = i % NS1, k = (i / NS1) % nch, o = i / (NS1 * nch);
            double hi = 0.0, lo = 0.0;
            for (int w = 0; w < EG * 4; ++w) {
                const double* slot = ll_slots + 2 * ((((size_t)w * NOUT + o) * KC + k) * NS1 + j);
                fed::dd_add(hi, lo, slot[0], slot[1]);
            }
            const int oj = (kPhi && j > G) ? j + P : j;
            out[2 * (((size_t)o * nch + k) * NV1 + oj)] = hi;
            out[2 * (((size_t)o * nch + k) * NV1 + oj) + 1] = lo;
        }
        if (threadIdx.x == 0) fed::stamp(comm, 6);
    } else if (warp == 0) {
        // nothing will be computed (stop / idle): the early loads still have to land before the CTA may exit
        for (int t = 0; t < preloaded; ++t) mbar_wait(&bar_full[t], 0u);
    }
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, kTmemCols);
    const unsigned long long status = *pipeline_fault() ? B200FED_ERR_PIPELINE : 0ull;
    const bool fin = fed::epilogue_t<true>(comm, pro, status, row_doubles, comm.group_partials);
    if (fin && threadIdx.x == 0) *work_counter = 0u;   // every CTA has stopped claiming: ready for the next launch
}

}  // namespace tc

// ------------------------------------------------------------------ host side
namespace {
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}
int chains_bucket(int k) { return k <= 1 ? 1 : (k <= 4 ? 4 : (k <= 8 ? 8 : (k <= 16 ? 16 : 0))); }
}  // namespace

// Builds one TMA descriptor per segment ([n_rows, P] bf16, box = 64 features x 128 rows, 128B swizzle) and
// the chunk table.
extern "C" int b200_glm_tc_prepare(const GlmSegment* segs_host, int n_segments, const GlmParams* prm, int sm_count,
                                   void** tmaps_dev, void** chunks_dev, int* n_chunks) {
    if (prm->n_features % 8 != 0 || prm->n_features > 384 || prm->n_features < 8) return -11;   // padded to 128s by TMA
    if (chains_bucket(prm->n_chains) == 0) return -13;
    if ((prm->ld * 2) % 16 != 0) return -14;
    EncodeTiledFn encode = get_encode();
    if (!encode) return -15;
    for (int s = 0; s < n_segments; ++s)
        if (segs_host[s].n_rows + tc::kTileM >= (1ll << 31)) return -18;   // row coordinates are 32-bit
    CUtensorMap* host = new CUtensorMap[n_segments];
    for (int s = 0; s < n_segments; ++s) {
        if (((uintptr_t)segs_host[s].X & 15) != 0) { delete[] host; return -16; }
        cuuint64_t dims[2] = {(cuuint64_t)prm->n_features, (cuuint64_t)segs_host[s].n_rows};
        cuuint64_t strides[1] = {(cuuint64_t)prm->ld * 2};
        cuuint32_t box[2] = {(cuuint32_t)tc::kPanel, (cuuint32_t)tc::kTileM};
        cuuint32_t estr[2] = {1, 1};
        CUresult r = encode(&host[s], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(segs_host[s].X), dims, strides,
                            box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                            CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { delete[] host; return -17; }
    }
    if (*tmaps_dev) cudaFree(*tmaps_dev);
    cudaError_t e = cudaMalloc(tmaps_dev, sizeof(CUtensorMap) * n_segments);
    if (e == cudaSuccess) e = cudaMemcpy(*tmaps_dev, host, sizeof(CUtensorMap) * n_segments, cudaMemcpyHostToDevice);
    delete[] host;
    if (e != cudaSuccess) return (int)e;
    const std::vector<GlmChunk> chunks = build_chunks(segs_host, n_segments, sm_count > 0 ? sm_count : 148, tc::kTileM, 2,
                                                        tc::kMaxChunk, tc::kMinChunk);
    if (*chunks_dev) cudaFree(*chunks_dev);
    e = cudaMalloc(chunks_dev, sizeof(GlmChunk) * (chunks.size() + 1));
    if (e == cudaSuccess) e = cudaMemcpy(*chunks_dev, chunks.data(), sizeof(GlmChunk) * chunks.size(), cudaMemcpyHostToDevice);
    *n_chunks = (int)chunks.size();
    return e == cudaSuccess ? 0 : (int)e;
}

// The chunk table for given segment sizes (host only; tests/test_chunk_schedule.py).  Writes up to max_chunks
// triples (seg, first_tile, n_tiles) and returns the number of chunks.
extern "C" int b200_glm_tc_chunk_table(const long long* n_rows, int n_segments, int sm_count, int multiple, int max_chunk,
                                       int min_chunk, int* out, int max_chunks) {
    std::vector<GlmSegment> segs(n_segments);
    for (int s = 0; s < n_segments; ++s) segs[s].n_rows = n_rows[s];
    const std::vector<GlmChunk> chunks = build_chunks(segs.data(), n_segments, sm_count, tc::kTileM, multiple, max_chunk, min_chunk);
    for (size_t i = 0; i < chunks.size() && (int)i < max_chunks; ++i) {
        out[3 * i + 0] = chunks[i].seg;
        out[3 * i + 1] = chunks[i].first_tile;
        out[3 * i + 2] = chunks[i].n_tiles;
    }
    return (int)chunks.size();
}

// doubles in the partial array of the tensor-core kernel: one row of (hi, lo) pairs + per-warp LL slots per CTA
extern "C" size_t b200_glm_tc_partial_row_doubles(int n_vals, int n_chains, int n_out, int n_groups, int n_family_params) {
    return tc::partial_row_doubles(n_vals, chains_bucket(n_chains), n_out > 0 ? n_out : 1, n_groups, n_family_params);
}

extern "C" int b200_launch_glm_tc(const FedComm* comm, const GlmSegment* segs_dev, const GlmParams* prm, const void* tmaps,
                                  const void* chunks_dev, int n_chunks, unsigned int* work_counter, int grid,
                                  cudaStream_t stream) {
    const int kc = chains_bucket(prm->n_chains);
    if (kc == 0) return -1;
    const CUtensorMap* maps = reinterpret_cast<const CUtensorMap*>(tmaps);
#define LAUNCH_TC(KC, PHI)                                                                                         \
    do {                                                                                                           \
        const tc::SmemLayout L = tc::smem_layout((prm->n_features + 127) & ~127, tc::Cfg<KC>::N1, tc::Cfg<KC>::N2, comm->n_theta,  \
                                                 prm->n_groups, KC, tc::Cfg<KC>::RB, PHI ? KC * (int)sizeof(tc::PhiChain) : 0); \
        if (L.stages < 2) return -2;                                                                               \
        cudaFuncSetAttribute(tc::fed_glm_tc_kernel<KC, PHI>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total); \
        cudaLaunchConfig_t cfg{};                                                                                  \
        cfg.gridDim = dim3(grid);                                                                                  \
        cfg.blockDim = dim3(tc::Cfg<KC>::kThreads);                                                                \
        cfg.dynamicSmemBytes = L.total;                                                                            \
        cfg.stream = stream;                                                                                       \
        cudaLaunchAttribute attr[1];                                                                               \
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;                                           \
        attr[0].val.programmaticStreamSerializationAllowed = 1;                                                    \
        cfg.attrs = attr;                                                                                          \
        cfg.numAttrs = tc::use_pdl() ? 1 : 0;                                                                      \
        cudaLaunchKernelEx(&cfg, tc::fed_glm_tc_kernel<KC, PHI>, *comm, segs_dev, *prm, maps,                      \
                           reinterpret_cast<const GlmChunk*>(chunks_dev), n_chunks, work_counter);                 \
    } while (0)
    if (prm->n_family_params > 0) {
        if (kc == 1) LAUNCH_TC(1, true);
        else if (kc == 4) LAUNCH_TC(4, true);
        else if (kc == 8) LAUNCH_TC(8, true);
        else LAUNCH_TC(16, true);
    } else {
        if (kc == 1) LAUNCH_TC(1, false);
        else if (kc == 4) LAUNCH_TC(4, false);
        else if (kc == 8) LAUNCH_TC(8, false);
        else LAUNCH_TC(16, false);
    }
#undef LAUNCH_TC
    return (int)cudaGetLastError();
}
