// runtime.cu -- slice handle, loader, forward scheduling and the C ABI (include/b200_slice.h).
//
// Replaces TransformerSlice / llama_eval_internal / the loader of the reference
// (distllm/tensor_processor.cpp:1488-1562, 474-809, 926-1086, 1203-1416) for a slice resident on
// one B200.  One stream per slice; the N=1 decode step is a CUDA graph replayed per token with
// the position kept in device memory.
#include "kernels.cuh"
#include "persist.cuh"
#include "fastgemm.cuh"
#include "fastgemm2.cuh"
#include "ggjt_file.hpp"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <dlfcn.h>
#include <cstdlib>
#include <map>
#include <memory>
#include <mutex>
#include <thread>
#include <vector>

namespace b200 {

constexpr int kSmemLimit = 226 * 1024;   // opt-in dynamic limit is 227 KB minus static __shared__

struct LayerW {
    PackedW qkv{}, wo{}, w13{}, w2{};
    PackedW wo_p{}, w2_p{};      // persistent-kernel copies of the narrow matrices with fewer row-groups per tile (B200_PERSIST_TR)
    // F16-weight slices
    uint16_t * f_q = nullptr, * f_k = nullptr, * f_v = nullptr, * f_o = nullptr, * f_1 = nullptr, * f_2 = nullptr, * f_3 = nullptr;
    float * attn_norm = nullptr, * ffn_norm = nullptr;
};

struct GraphKey { const float * in; float * out; int host; bool operator<(const GraphKey & o) const {
    return in != o.in ? in < o.in : (out != o.out ? out < o.out : host < o.host); } };

// A step over several sessions (batched or mixed, see plan_step): segment i is len_i consecutive tokens of one session, the
// columns of the step are the segments back to back.
struct StepPlan {
    std::vector<int2> segs;            // (session, len)
    std::vector<int4> cols;            // column -> (session, position, T = n_past + len of its segment, 0)
    std::vector<AttnBlock> blocks;     // head size 128: query blocks of the chunks on k_attn128_tiled
    std::vector<int> clist;            // head size 128: the other columns (k_attn128<false>)
    int t_rows = 0;                    // largest T among the tiled chunks
    bool ones = true;                  // every segment is one token: the batched-step schedule (fused RoPE + attention)
};

}  // namespace b200

using namespace b200;

struct b200_slice {
    int device = 0, n_sm = 148;
    cudaStream_t stream = nullptr;
    int E = 0, H = 0, D = 0, FF = 0, L = 0, first_layer = 0, n_ctx = 512, wtype = 0;
    // sessions (SURVEY 8f N3): independent sequences sharing the weights, each with its own KV cache and position.
    // Session 0 is the reference's single global context (tensor_processor.cpp:1491, 1992).
    int n_sessions = 1, cur = 0;
    std::vector<int> past;                 // n_past per session
    int * d_npast = nullptr;               // [n_sessions], device copy (graph replays read it)
    size_t sess_stride = 0;                // elements between two sessions' KV caches
    // multi-session step: s->plan's tables on the device; cols != nullptr while such a step is being enqueued
    int4 * d_cols = nullptr; const int4 * cols = nullptr; AttnBlock * d_blocks = nullptr; int * d_clist = nullptr;
    StepPlan plan;
    std::vector<LayerW> layers;
    std::vector<void *> allocs;
    uint16_t * kc = nullptr, * vc = nullptr, * q16 = nullptr;
    float * xa = nullptr, * xb = nullptr, * qkv = nullptr, * att = nullptr, * ffin = nullptr, * gate = nullptr;
    float * d_in = nullptr, * d_out = nullptr, * h_in = nullptr, * h_out = nullptr;
    float2 * cs = nullptr; uint16_t * texp = nullptr, * tsilu = nullptr;
    int * aq_att = nullptr, * aq_gate = nullptr; float * da_att = nullptr, * da_gate = nullptr;   // pre-quantised activations
    int nbqE = 0, nbqF = 0;
    int soffE = 0, soffF = 0;              // Q4_1 slices (Q8_1 activations): floats between the scale plane and the block-sum plane of da_*
    int * aq_x = nullptr; float * da_x = nullptr; int * nq_counter = nullptr; double * nq_partial = nullptr;   // normalised+quantised layer input (last-CTA epilogue)
    std::map<GraphKey, cudaGraphExec_t> graphs;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr; bool timed = false;
    int64_t launches = 0, weight_bytes = 0;
    bool use_ring = true, use_graph = true, use_pdl = false, use_nq = true, f16_ring = true, use_tiled_attn = true, use_n8 = false, f16_mc = true; int f16_mc_cols = 4;
    bool skip_attention = false;   // measurement aid: replay only the weight matmuls of a step (bench.py roofline)
    bool fast_prefill = false; int fast_min_tokens = 32; uint16_t * xh = nullptr;   // tcgen05 prefill (fast mode)
    int fast_version = 2;                                                               // 2: fastgemm2.cuh (TMA tensor map, N = 256), 1: fastgemm.cuh
    int opt_ns = 0, opt_cta_per_sm = 0, opt_nc = 0, opt_pre = 3, opt_nomath = 0;   // read once at load (environment)
    float ema_token_ms = 0.f;              // host-buffer decode calls: smoothed device time of one token (sleep-then-poll wait)
    std::mutex mu;
    // per-kernel-class event timing (b200_slice_profile): class 0 qkv, 1 rope, 2 attention, 3 wo, 4 w13, 5 w2, 6 advance
    bool profiling = false; int cur_class = 0;
    std::vector<cudaEvent_t> prof_ev; std::vector<int> prof_cls; size_t prof_used = 0;
    cudaEvent_t mark[2] = {nullptr, nullptr};
    // debug timeline
    unsigned long long * trace = nullptr; int trace_next = 0; std::vector<int> trace_cls, trace_ctas;
    // layer-slice pipeline over NCCL (see b200_pipeline_*)
    void * nccl_comm = nullptr; int pp_rank = 0, pp_world = 1; float * d_final = nullptr;
    // peer-memory hand-off (b200_pipeline_mailbox_*): my mailbox, and my ring neighbours' mailboxes mapped over NVLink
    uint8_t * mb_block = nullptr; size_t mb_slot_floats = 0;
    uint8_t * mb_next = nullptr, * mb_prev = nullptr; bool mb_on = false;
    bool send_pending = false; PeerSendArgs send_args{}; int send_ctas = 1;      // enqueue_layers launches the send right behind the last matmul
    // single-token steps fold the send into the slice's last matmul (EPI_RESID_SEND): rows leave for the next rank's inbox
    // as they are computed, no k_peer_send launch on the critical path
    bool fold_send = false, use_fold = true;
    std::map<GraphKey, cudaGraphExec_t> pp_graphs;
    // persistent single-token step (persist.cuh)
    bool use_persist = false; int persist_tr = 4, persist_ns = 0, persist_ctas = 0;
    int * p_cnt = nullptr; std::map<GraphKey, PLayer *> p_tables; unsigned long long * p_trace = nullptr;
};

namespace b200 {

static int env_int(const char * name, int dflt) { const char * v = getenv(name); return v ? atoi(v) : dflt; }

template <typename T> static int dev_alloc(b200_slice * s, T ** p, size_t n) {
    void * q = nullptr;
    cudaError_t e = cudaMalloc(&q, n * sizeof(T));
    if (e != cudaSuccess) return fail(B200_ECUDA, "cudaMalloc(%zu) failed: %s", n * sizeof(T), cudaGetErrorString(e));
    s->allocs.push_back(q); *p = (T *) q; return 0;
}

// ---------------------------------------------------------------- per-launch event brackets
static void prof_begin(b200_slice * s) {
    if (!s->profiling) return;
    if (s->prof_used + 2 > s->prof_ev.size()) {
        for (int i = 0; i < 2; i++) { cudaEvent_t e; cudaEventCreate(&e); s->prof_ev.push_back(e); }
    }
    cudaEventRecord(s->prof_ev[s->prof_used], s->stream);
}
static void prof_end(b200_slice * s) {
    if (!s->profiling) return;
    cudaEventRecord(s->prof_ev[s->prof_used + 1], s->stream);
    s->prof_cls.push_back(s->cur_class);
    s->prof_used += 2;
}

// ---------------------------------------------------------------- kernel dispatch
template <int WT, int G, int NC, int PRO, int EPI, bool RING>
static int launch_gemv_t(b200_slice * s, GemvArgs a) {
    constexpr int CB = chunk_bytes(WT);
    constexpr int TR = kWPC * G;
    auto kern = k_gemv<WT, G, NC, PRO, EPI, RING>;
    static bool attr_set[16] = {false};
    const size_t stage = (size_t) kQS * TR * CB;
    const size_t act = (size_t) NC * act_bytes_per_col(a.W.nbq, WT) + 34 * 8 + kWPC * 8 + (size_t) NC * 128 + 64 +
                       ((NC == 1 && PRO == PRO_NORM) ? (size_t) a.W.K * 4 : 0);
    // Ring depth: as deep as possible while EVERY tile of the matrix still gets a co-resident CTA (no second wave):
    // wide matrices (qkv 384 tiles, w1|w3 688) run 3-5 small-ring CTAs per SM, narrow ones (wo, w2: 128 tiles) one
    // CTA per SM with a deep ring.  B200_NS overrides.
    int NS = 0;
    if (RING) {
        const int ncolg = (a.N + NC - 1) / NC;
        int need = (a.W.n_tiles * ncolg + s->n_sm - 1) / s->n_sm;
        if (need > 5) need = 5;
        const size_t budget = (size_t) kSmemLimit / need - 1024;
        NS = s->opt_ns > 0 ? s->opt_ns : (budget > act ? (int)((budget - act) / stage) : 2);
        if (NS < 2) NS = 2;
        if (NS > 16) NS = 16;
        while (NS > 2 && NS * stage + act > (size_t) kSmemLimit) NS--;
    }
    const size_t smem = NS * stage + act;
    if (smem > (size_t) kSmemLimit) return fail(B200_EINVAL, "gemv needs %zu B of shared memory (K=%d, NC=%d)", smem, a.W.K, NC);
    if (!attr_set[s->device & 15]) {
        B200_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
        // without this the driver's carve-out heuristic leaves room for only 2 CTAs/SM however small the ring is
        B200_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        attr_set[s->device & 15] = true;
    }
    a.NS = NS; a.dbg_nomath = s->opt_nomath; a.pre_stages = s->opt_pre;
    a.trace = nullptr;
    if (s->trace && s->trace_next < 512) { a.trace = s->trace + (size_t) s->trace_next * 1024 * 8; s->trace_next++; s->trace_cls.push_back(s->cur_class); }
    int per_sm = s->opt_cta_per_sm > 0 ? s->opt_cta_per_sm : (int)(kSmemLimit / (smem + 1024));
    if (per_sm < 1) per_sm = 1;
    if (per_sm > 6) per_sm = 6;
    const int ncol = (a.N + NC - 1) / NC;
    int gx = a.W.n_tiles;
    const int cap = s->n_sm * per_sm;
    if (gx > cap) gx = cap;
    cudaLaunchConfig_t cfg{};
    if (a.trace) s->trace_ctas.push_back(gx * ncol);
    cfg.gridDim = dim3(gx, ncol, 1);
    cfg.blockDim = dim3(RING ? kConsumers + 32 : kConsumers, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s->stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = s->use_pdl ? 1 : 0;
    prof_begin(s);
    B200_CUDA(cudaLaunchKernelEx(&cfg, kern, a));
    prof_end(s);
    s->launches++;
    return 0;
}

// narrow matrices of a single-token step: 8 threads per row (k_gemv_n8), one CTA per tile, deep ring
template <int WT, int EPI>
static int launch_gemv8_t(b200_slice * s, GemvArgs a) {
    constexpr int CB = chunk_bytes(WT);
    auto kern = k_gemv_n8<WT, EPI>;
    static bool attr_set[16] = {false};
    const size_t stage = (size_t) kQS * 4 * CB;
    const size_t act = (size_t) a.W.nbq * 144 + 34 * 8 + 64;
    // every tile gets a co-resident CTA (13B: 160 tiles -> two CTAs on some SMs, each with half the ring)
    const int need = (a.W.n_tiles + s->n_sm - 1) / s->n_sm;
    const size_t budget = (size_t) kSmemLimit / need - 1024;
    int NS = s->opt_ns > 0 ? s->opt_ns : (budget > act ? (int)((budget - act) / stage) : 2);
    if (NS > 16) NS = 16;
    if (NS < 2) NS = 2;
    const size_t smem = NS * stage + act;
    if (smem > (size_t) kSmemLimit) return fail(B200_EINVAL, "gemv8 needs %zu B of shared memory (K=%d)", smem, a.W.K);
    if (!attr_set[s->device & 15]) {
        B200_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
        B200_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        attr_set[s->device & 15] = true;
    }
    a.NS = NS; a.dbg_nomath = s->opt_nomath; a.pre_stages = s->opt_pre;
    a.trace = nullptr;
    if (s->trace && s->trace_next < 512) { a.trace = s->trace + (size_t) s->trace_next * 1024 * 8; s->trace_next++; s->trace_cls.push_back(s->cur_class); }
    const int gx = a.W.n_tiles;
    if (a.trace) s->trace_ctas.push_back(gx);
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(gx, 1, 1);
    cfg.blockDim = dim3(kN8Consumers + 32, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s->stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = s->use_pdl ? 1 : 0;
    prof_begin(s);
    B200_CUDA(cudaLaunchKernelEx(&cfg, kern, a));
    prof_end(s);
    s->launches++;
    return 0;
}
// applies to: one column, ring on, Q4_0 / Q8_0, the matrix is narrow enough that k_gemv would run <= 1 CTA per SM
static bool gemv8_applicable(const b200_slice * s, const PackedW & W, int N) {
    return s->use_n8 && N == 1 && !s->cols && s->use_ring && (W.wtype == kWT_Q4_0 || W.wtype == kWT_Q8_0) && W.TR == 4 &&
           W.n_tiles <= s->n_sm * 3 / 2;
}
template <int EPI>
static int launch_gemv8(b200_slice * s, const GemvArgs & a) {
    if (a.W.wtype == kWT_Q4_0) return launch_gemv8_t<kWT_Q4_0, EPI>(s, a);
    return launch_gemv8_t<kWT_Q8_0, EPI>(s, a);
}

template <int WT, int G, int PRO, int EPI>
static int launch_gemv_nc(b200_slice * s, const GemvArgs & a) {
    if (a.N == 1) return s->use_ring ? launch_gemv_t<WT, G, 1, PRO, EPI, true>(s, a) : launch_gemv_t<WT, G, 1, PRO, EPI, false>(s, a);
    if (!s->use_ring) return launch_gemv_t<WT, G, 8, PRO, EPI, false>(s, a);
    // Columns per CTA.  A multi-column step is issue-bound (every column repeats the dp4a -> fadd -> fma chains), so it
    // needs warps, not bytes: 8 columns per CTA amortise the nibble unpacking best, but a small batch (<= 8 columns)
    // over a narrow matrix (wo / w2: 128-160 tiles) would then run ONE 4-warp CTA per SM.  Take the widest column
    // group that still puts >= 3 CTAs on every SM; the extra column groups re-read the tile from L2, not from HBM
    // (they are co-resident and walk the tiles in the same order).
    const int want = 3 * s->n_sm, nt = a.W.n_tiles;
    const int force = s->opt_nc;
    if (force == 8 || (!force && nt * ((a.N + 7) / 8) >= want)) return launch_gemv_t<WT, G, 8, PRO, EPI, true>(s, a);
    if (force == 4 || (!force && nt * ((a.N + 3) / 4) >= want)) return launch_gemv_t<WT, G, 4, PRO, EPI, true>(s, a);
    return launch_gemv_t<WT, G, 2, PRO, EPI, true>(s, a);
}

template <int G, int PRO, int EPI>
static int launch_gemv(b200_slice * s, const GemvArgs & a) {
    if (a.W.wtype == kWT_Q4_0) return launch_gemv_nc<kWT_Q4_0, G, PRO, EPI>(s, a);
    if (a.W.wtype == kWT_Q4_1) return launch_gemv_nc<kWT_Q4_1, G, PRO, EPI>(s, a);
    return launch_gemv_nc<kWT_Q8_0, G, PRO, EPI>(s, a);
}

template <typename K, typename A>
static int launch_simple(b200_slice * s, K kern, dim3 grid, dim3 block, size_t smem, const A & args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s->stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = s->use_pdl ? 1 : 0;
    prof_begin(s);
    B200_CUDA(cudaLaunchKernelEx(&cfg, kern, args));
    prof_end(s);
    s->launches++;
    return 0;
}

template <int PRO, int EPI>
static int launch_f16(b200_slice * s, GemvF16Args a) {
    auto kern = k_gemv_f16<PRO, EPI>;
    static bool attr_set[16] = {false};
    const size_t smem = (size_t) a.K * 2 + 16;
    if (!attr_set[s->device & 15]) {
        B200_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
        attr_set[s->device & 15] = true;
    }
    if (a.N == 1 && s->use_ring && s->f16_ring && (a.K & 255) == 0) {
        // single-token steps: TMA-ring variant (weights stream from before the dependency wait, two CTAs per SM)
        auto rk = k_gemv_f16_ring<PRO, EPI>;
        static bool rattr[16] = {false};
        if (!rattr[s->device & 15]) {
            B200_CUDA(cudaFuncSetAttribute(rk, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
            B200_CUDA(cudaFuncSetAttribute(rk, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
            rattr[s->device & 15] = true;
        }
        const int nc8 = (a.K / 32 + 7) / 8;
        const size_t fixed = (size_t) nc8 * 1024 + 64 + 64;
        int NS = s->opt_ns > 0 ? s->opt_ns : (int)(((size_t) 112 * 1024 - fixed) / ((size_t) kF16Warps * (kF16Stage + 16)));
        if (NS < 2) NS = 2;
        if (NS > 12) NS = 12;
        const size_t rsmem = (size_t) kF16Warps * NS * kF16Stage + (size_t) nc8 * 1024 + (size_t) 2 * kF16Warps * NS * 8 + 64;
        const int n_tiles = (a.rows + kF16Warps - 1) / kF16Warps;
        int per_sm = (int)(kSmemLimit / (rsmem + 1024)); if (per_sm < 1) per_sm = 1; if (per_sm > 4) per_sm = 4;
        int rgx = n_tiles < s->n_sm * per_sm ? n_tiles : s->n_sm * per_sm;
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3(rgx, 1, 1); cfg.blockDim = dim3(kF16Warps * 32 + 32, 1, 1); cfg.dynamicSmemBytes = rsmem; cfg.stream = s->stream;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = at; cfg.numAttrs = s->use_pdl ? 1 : 0;
        prof_begin(s);
        B200_CUDA(cudaLaunchKernelEx(&cfg, rk, a, NS));
        prof_end(s);
        s->launches++;
        return 0;
    }
    int gx = (a.rows + 7) / 8;
    if (a.N >= 2 && s->f16_mc) {
        gx = (a.rows + 15) / 16;                         // 8 warps x 2 rows per CTA
        // multi-token call: 8 (or 4) columns per CTA share every weight load (k_gemv_f16_mc)
        // 4 columns per CTA keep the activation block at 64 KB for K = 4096: three CTAs (24 warps) per SM; B200_F16_MC=8 forces 8
        const bool c8 = s->f16_mc_cols == 8 && a.N > 4 && (size_t) a.K * 4 * 8 + 64 <= (size_t) 200 * 1024;
        const int nc = c8 ? 8 : 4;
        const size_t msmem = (size_t) a.K * 4 * nc + 64;
        if (msmem <= (size_t) 72 * 1024 || (c8 && msmem <= (size_t) kSmemLimit)) {
            static bool mattr[16] = {false};
            if (!mattr[s->device & 15]) {
                B200_CUDA(cudaFuncSetAttribute(k_gemv_f16_mc<PRO, EPI, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
                B200_CUDA(cudaFuncSetAttribute(k_gemv_f16_mc<PRO, EPI, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
                mattr[s->device & 15] = true;
            }
            const int ncolg = (a.N + nc - 1) / nc;
            int per_sm = (int)(kSmemLimit / (msmem + 1024)); if (per_sm < 1) per_sm = 1;
            int mgx = gx; const int mcap = (s->n_sm * per_sm + ncolg - 1) / ncolg;
            if (mgx > mcap) mgx = mcap < 1 ? 1 : mcap;
            if (c8) return launch_simple(s, k_gemv_f16_mc<PRO, EPI, 8>, dim3(mgx, ncolg, 1), dim3(256, 1, 1), msmem, a);
            return launch_simple(s, k_gemv_f16_mc<PRO, EPI, 4>, dim3(mgx, ncolg, 1), dim3(256, 1, 1), msmem, a);
        }
    }
    gx = (a.rows + 7) / 8;
    const int cap = s->n_sm * 8;
    if (gx > cap) gx = cap;
    return launch_simple(s, kern, dim3(gx, a.N, 1), dim3(256, 1, 1), smem, a);
}

static int launch_norm_quant(b200_slice * s, const float * x, int ldx, const float * norm_w, int N) {
    NormQuantArgs q{x, ldx, norm_w, s->E, s->aq_x, s->da_x, s->nbqE, s->soffE};
    if (s->wtype == kWT_Q4_0) return launch_simple(s, k_norm_quant<kWT_Q4_0>, dim3(N, 1, 1), dim3(256, 1, 1), 0, q);
    if (s->wtype == kWT_Q4_1) return launch_simple(s, k_norm_quant<kWT_Q4_1>, dim3(N, 1, 1), dim3(256, 1, 1), 0, q);
    return launch_simple(s, k_norm_quant<kWT_Q8_0>, dim3(N, 1, 1), dim3(256, 1, 1), 0, q);
}

// ---------------------------------------------------------------- fast-mode prefill (tcgen05), see fastgemm.cuh
template <bool NORM>
static int launch_prep(b200_slice * s, const float * x, int ldx, const float * norm_w, int K, int N) {
    PrepArgs p{x, ldx, norm_w, s->xh, K, N};
    return launch_simple(s, k_prep_q8_f16<NORM>, dim3(N, 1, 1), dim3(256, 1, 1), 0, p);
}
template <int EPI>
static int launch_fast_gemm(b200_slice * s, const PackedW & W, const float * resid, int ldr, float * y, int ldy, int N, int out_rows) {
    static bool attr_set[16] = {false};
    auto kern = k_gemm_q4_tc<EPI>;
    if (!attr_set[s->device & 15]) {
        B200_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kFgSmem));
        attr_set[s->device & 15] = true;
    }
    FastGemmArgs a{}; a.W = W; a.xh = s->xh; a.resid = resid; a.ldr = ldr; a.y = y; a.ldy = ldy; a.N = N; a.out_rows = out_rows;
    a.tsilu = s->tsilu;
    const int groups = W.n_tiles * W.TR;                     // 8-row groups in packed order
    return launch_simple(s, kern, dim3((groups + 15) / 16, (N + kFgN - 1) / kFgN, 1), dim3(160, 1, 1), kFgSmem, a);
}

// second-generation tcgen05 prefill matmul (fastgemm2.cuh): 128 x 256 tiles, activations through a tensor-map TMA
typedef CUresult (*TensorMapEncodeFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                      const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                      CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static TensorMapEncodeFn tensor_map_encode() {
    static TensorMapEncodeFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void * p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
            fn = (TensorMapEncodeFn) p;
    });
    return fn;
}

template <int WT, int EPI, int NT>
static int launch_fast_gemm2_t(b200_slice * s, const PackedW & W, const float * resid, int ldr, float * y, int ldy, int N, int out_rows) {
    TensorMapEncodeFn enc = tensor_map_encode();
    if (!enc) return fail(B200_ECUDA, "cuTensorMapEncodeTiled is not available from this driver");
    // activations xh [N][K] fp16, K innermost; box = 64 halfs (128 B, the swizzle span) x 256 token rows; rows >= N read as zeros
    CUtensorMap map;
    const cuuint64_t dims[2] = {(cuuint64_t) W.K, (cuuint64_t) N};
    const cuuint64_t strides[1] = {(cuuint64_t) W.K * 2};
    const cuuint32_t box[2] = {64, (cuuint32_t) NT};
    const cuuint32_t estr[2] = {1, 1};
    CUresult cr = enc(&map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, (void *) s->xh, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                      CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS) return fail(B200_ECUDA, "cuTensorMapEncodeTiled failed (%d) for K=%d N=%d", (int) cr, W.K, N);
    auto kern = k_gemm_tc2<WT, EPI, NT>;
    static bool attr_set[16] = {false};
    if (!attr_set[s->device & 15]) {
        B200_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, f2_smem(WT, NT)));
        attr_set[s->device & 15] = true;
    }
    FastGemm2Args a{}; a.W = W; a.resid = resid; a.ldr = ldr; a.y = y; a.ldy = ldy; a.N = N; a.out_rows = out_rows; a.tsilu = s->tsilu;
    const int groups = W.n_tiles * W.TR;                     // 8-row groups in packed order
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((groups + 15) / 16, (N + NT - 1) / NT, 1); cfg.blockDim = dim3(kF2Threads, 1, 1);
    cfg.dynamicSmemBytes = f2_smem(WT, NT); cfg.stream = s->stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = s->use_pdl ? 1 : 0;
    prof_begin(s);
    B200_CUDA(cudaLaunchKernelEx(&cfg, kern, a, map));
    prof_end(s);
    s->launches++;
    return 0;
}
// tile: 0 picks the token tile below; 128 / 256 force it (v2 only; b200_debug_fast_matmul)
template <int EPI>
static int launch_fast_any(b200_slice * s, const PackedW & W, const float * resid, int ldr, float * y, int ldy, int N, int out_rows,
                           int tile = 0) {
    if (s->fast_version >= 2) {
        // 256-token tiles halve the dequantisation per flop; a matrix whose 128-row tiles x 256-token tiles would leave SMs idle
        // (wo, w2: 32 row tiles) takes 128-token tiles and three stages instead
        const int mtiles = (W.n_tiles * W.TR + 15) / 16;
        const bool wide = tile ? tile == 256 : (long long) mtiles * ((N + 255) / 256) >= s->n_sm || N <= 128;
        if (W.wtype == kWT_Q4_0) return wide ? launch_fast_gemm2_t<kWT_Q4_0, EPI, 256>(s, W, resid, ldr, y, ldy, N, out_rows)
                                             : launch_fast_gemm2_t<kWT_Q4_0, EPI, 128>(s, W, resid, ldr, y, ldy, N, out_rows);
        return wide ? launch_fast_gemm2_t<kWT_Q8_0, EPI, 256>(s, W, resid, ldr, y, ldy, N, out_rows)
                    : launch_fast_gemm2_t<kWT_Q8_0, EPI, 128>(s, W, resid, ldr, y, ldy, N, out_rows);
    }
    return launch_fast_gemm<EPI>(s, W, resid, ldr, y, ldy, N, out_rows);
}

// The slice's weights suit the tcgen05 matmuls: Q4_0 (v1, v2) or Q8_0 (v2), and qkv / wo / w1|w3 are whole 16-group M tiles.
static bool fast_weights_ok(const b200_slice * s, const LayerW & Lw) {
    return (s->wtype == kWT_Q4_0 || (s->wtype == kWT_Q8_0 && s->fast_version >= 2)) && (Lw.qkv.n_tiles * Lw.qkv.TR) % 16 == 0 &&
           (Lw.wo.n_tiles * Lw.wo.TR) % 16 == 0 && (Lw.w13.n_tiles * Lw.w13.TR) % 16 == 0;
}

// A call runs in fast mode only as a prompt chunk of one sequence: single-token steps and batched steps (one token for each of
// several sessions, s->cols) promise results bit-identical to exact mode, so they never take it, whatever fast_min_tokens says.
static bool fast_applicable(const b200_slice * s, const LayerW & Lw, int N) {
    return s->fast_prefill && N > 1 && !s->cols && N >= s->fast_min_tokens && fast_weights_ok(s, Lw);
}

// ---------------------------------------------------------------- persistent single-token step (persist.cuh)
static bool persist_applicable(const b200_slice * s, int N) {
    return s->use_persist && N == 1 && !s->cols && s->D == 128 && (s->wtype == kWT_Q4_0 || s->wtype == kWT_Q8_0) && !s->skip_attention &&
           !s->profiling && s->E / 32 <= kPConsumers && s->p_cnt != nullptr;
}

static PMat pmat_of(const PackedW & W, int G) {
    PMat m{};
    m.data = W.data; m.n_tiles = W.n_tiles; m.nbq = W.nbq; m.TR = W.TR; m.tile_bytes = W.tile_bytes;
    m.sq = kQS / G;                           // quads per ring stage: one stage = 16 chunks = one slot
    return m;
}

// The layer table of a step (weights + this call's buffers) lives in device memory; it depends on (in, out, session), so
// it is built once per such triple -- OUTSIDE any stream capture, which is why forward paths call this before capturing.
static int persist_prepare(b200_slice * s, const float * in, float * out) {
    GraphKey key{in, out, s->cur};
    if (s->p_tables.count(key)) return 0;
    std::vector<PLayer> tab(s->L);
    const float * cur = in;
    const int E = s->E;
    const size_t sess_off = (size_t) s->cur * s->sess_stride;
    for (int il = 0; il < s->L; il++) {
        LayerW & Lw = s->layers[il];
        PLayer & P = tab[il];
        P.qkv = pmat_of(Lw.qkv, 1);
        P.wo = pmat_of(Lw.wo, 1);
        P.w13 = pmat_of(Lw.w13, 2);
        P.w2 = pmat_of(Lw.w2, 1);
        P.attn_norm = Lw.attn_norm; P.ffn_norm = Lw.ffn_norm;
        float * nxt = (il == s->L - 1) ? out : ((il & 1) ? s->xb : s->xa);
        P.x_in = cur; P.x_out = nxt;
        P.kc = s->kc + sess_off + (size_t) il * s->n_ctx * E; P.vc = s->vc + sess_off + (size_t) il * s->n_ctx * E;
        cur = nxt;
    }
    PLayer * d = nullptr;
    int rc = dev_alloc(s, &d, (size_t) s->L);
    if (rc) return rc;
    B200_CUDA(cudaMemcpy(d, tab.data(), tab.size() * sizeof(PLayer), cudaMemcpyHostToDevice));
    s->p_tables[key] = d;
    return 0;
}

static int launch_persistent(b200_slice * s, const float * in, float * out) {
    auto it = s->p_tables.find(GraphKey{in, out, s->cur});
    if (it == s->p_tables.end()) return fail(B200_EINVAL, "persistent step: layer table not prepared");
    PersistArgs a{};
    a.layers = it->second; a.L = s->L;
    a.E = s->E; a.FF = s->FF; a.H = s->H; a.n_ctx = s->n_ctx; a.nb_E = s->E / 32; a.nbqE = s->nbqE; a.nbqF = s->nbqF;
    a.n_past = s->d_npast + s->cur;
    a.qkv = s->qkv; a.att = s->att; a.ffin = s->ffin;
    a.aq_att = s->aq_att; a.da_att = s->da_att; a.aq_gate = s->aq_gate; a.da_gate = s->da_gate;
    a.dscale = s->wtype == kWT_Q4_0 ? 0.0625f : 1.0f;
    a.cs = s->cs; a.texp = s->texp; a.tsilu = s->tsilu;
    a.cnt = s->p_cnt;
    a.kq_scale = 1.0f / sqrtf((float) s->E / (float) s->H);
    a.trace = s->p_trace;
    const int nbq_max = s->nbqF > s->nbqE ? s->nbqF : s->nbqE;
    const size_t limit = 227 * 1024;
    int NS = s->persist_ns > 0 ? s->persist_ns : 48;          // ring slots of the CTA: all the shared memory that is left
    while (NS > 4 && p_smem_layout(s->wtype, NS, nbq_max, s->E, s->n_ctx).total > limit) NS--;
    const PSmem lay = p_smem_layout(s->wtype, NS, nbq_max, s->E, s->n_ctx);
    if (lay.total > limit) return fail(B200_EINVAL, "persistent step needs %zu B of shared memory", lay.total);
    a.NS = NS;
    static bool attr_set[16] = {false};
    if (!attr_set[s->device & 15]) {
        B200_CUDA(cudaFuncSetAttribute(k_decode_persistent<kWT_Q4_0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) limit));
        B200_CUDA(cudaFuncSetAttribute(k_decode_persistent<kWT_Q8_0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) limit));
        attr_set[s->device & 15] = true;
    }
    // progress counters start at zero every step
    B200_CUDA(cudaMemsetAsync(s->p_cnt, 0, (size_t) s->L * kPPhases * 4, s->stream));
    int grid = s->persist_ctas > 0 ? s->persist_ctas : s->n_sm;      // one CTA per SM, all co-resident (they wait on each other)
    if (grid > s->n_sm) grid = s->n_sm;
    if (grid < s->H) return fail(B200_EINVAL, "persistent step needs at least n_head (%d) CTAs", s->H);
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid, 1, 1); cfg.blockDim = dim3(kPThreads, 1, 1); cfg.dynamicSmemBytes = lay.total; cfg.stream = s->stream;
    s->cur_class = 0;
    prof_begin(s);
    if (s->wtype == kWT_Q4_0) B200_CUDA(cudaLaunchKernelEx(&cfg, k_decode_persistent<kWT_Q4_0>, a));
    else                      B200_CUDA(cudaLaunchKernelEx(&cfg, k_decode_persistent<kWT_Q8_0>, a));
    prof_end(s);
    s->launches++;
    return 0;
}

// query-tiled prompt attention over grid_y query blocks; ta.t_rows = the largest T the blocks see
static int launch_attn_tiled(b200_slice * s, AttnTiledArgs ta, int grid_y) {
    ta.t_pad = (ta.t_rows + 31) & ~31;
    const size_t tsm = (size_t) ta.t_rows * kAttnRow + (size_t) kAttnQB * ta.t_pad * 6 + 4 * 8 * 128 * 4 + kAttnQB * 256 + 64;
    static bool tattr[16] = {false};
    if (!tattr[s->device & 15]) {
        B200_CUDA(cudaFuncSetAttribute(k_attn128_tiled, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
        tattr[s->device & 15] = true;
    }
    return launch_simple(s, k_attn128_tiled, dim3(s->H, grid_y, 1), dim3(512, 1, 1), tsm, ta);
}

// ---------------------------------------------------------------- one forward over the slice
// Enqueue every layer for N tokens at device-side position *d_npast (tensor_processor.cpp:537-766).
static int enqueue_layers(b200_slice * s, const float * in, int N, float * out) {
    const int E = s->E, FF = s->FF, H = s->H, D = s->D;
    const float * cur = in;
    const bool persist = persist_applicable(s, N);
    if (persist) { int rc = launch_persistent(s, in, out); if (rc) return rc; }
    for (int il = 0; il < (persist ? 0 : s->L); il++) {
        LayerW & Lw = s->layers[il];
        // grid-barrier norm+quant epilogue: decode only (every CTA of wo / w2 must be co-resident: 1 tile per CTA)
        const bool fast = fast_applicable(s, Lw, N);
        const bool nq = s->use_nq && N == 1 && !s->cols && s->wtype != kWT_F16 && Lw.wo.n_tiles <= 256 && Lw.wo.n_tiles <= s->n_sm * 2;
        float * nxt = (il == s->L - 1) ? out : ((il & 1) ? s->xb : s->xa);
        // cols mode (batched independent sequences): the kernels add session * sess_stride themselves
        const size_t sess_off = s->cols ? 0 : (size_t) s->cur * s->sess_stride;
        uint16_t * kc = s->kc + sess_off + (size_t) il * s->n_ctx * E, * vc = s->vc + sess_off + (size_t) il * s->n_ctx * E;
        int * d_npast = s->d_npast + s->cur;
        int rc;
        s->cur_class = 0;
        if (s->wtype == kWT_F16) {
            GemvF16Args f{}; f.K = E; f.x = cur; f.ldx = E; f.norm_w = Lw.attn_norm; f.N = N; f.tsilu = s->tsilu;
            f.rows = 3 * E; f.ldy = 3 * E;       // wq | wk | wv are packed back to back: one launch, one RMSNorm prologue
            f.W = Lw.f_q; f.y = s->qkv;         if ((rc = launch_f16<PRO_NORM, EPI_STORE>(s, f))) return rc;
        } else if (fast) {
            if ((rc = launch_prep<true>(s, cur, E, Lw.attn_norm, E, N))) return rc;
            if ((rc = launch_fast_any<FG_STORE>(s, Lw.qkv, nullptr, 0, s->qkv, 3 * E, N, 3 * E))) return rc;
        } else {
            GemvArgs g{}; g.W = Lw.qkv; g.x = cur; g.ldx = E; g.norm_w = Lw.attn_norm; g.y = s->qkv; g.ldy = 3 * E;
            g.N = N; g.out_rows = 3 * E; g.tsilu = s->tsilu; g.aq_in = s->aq_x; g.da_in = s->da_x; g.in_soff = s->soffE;
            // layers after the first get their input already normalised + quantised by the previous w2's last CTA
            if (il > 0 && nq) { if ((rc = launch_gemv<1, PRO_PREQ, EPI_STORE>(s, g))) return rc; }
            else if (N > 1) {
                // multi-token call: normalise + quantise every row ONCE instead of once per 32-row tile (k_norm_quant)
                if ((rc = launch_norm_quant(s, cur, E, Lw.attn_norm, N))) return rc;
                if ((rc = launch_gemv<1, PRO_PREQ, EPI_STORE>(s, g))) return rc;
            }
            else                     { if ((rc = launch_gemv<1, PRO_NORM, EPI_STORE>(s, g))) return rc; }
        }
        if (s->skip_attention) {
            // measurement aid: the matmul kernels of the step back to back, attention left out
        } else if (D == 128) {
            // head size 128: cluster kernel; for N = 1 RoPE + KV append are fused into its prologue
            constexpr int kChunk = 1024;     // query tokens per launch (grid.y)
            // scores + probabilities, then (single-token kernels) the staged K / V rows: up to 128 local rows = 512 positions
            const size_t sc_bytes = (((size_t)((s->n_ctx + 3) & ~3) * 4 + (size_t)((s->n_ctx + 7) & ~7) * 2) + 15) & ~(size_t) 15;
            int pf_rows = 8 * ((s->n_ctx + 31) / 32);
            if (pf_rows > 128) pf_rows = 128;
            const size_t asm_plain = sc_bytes + 64, asm_bytes = sc_bytes + (size_t) 2 * pf_rows * kAttnRow + 32 * 64 + 64;
            const size_t asm_lut = asm_bytes + 65536;            // + the exp table's negative half (single-token steps only)
            Attn128Args aa{};
            aa.pf_rows = pf_rows;
            aa.qkv = s->qkv; aa.q16 = s->q16; aa.kc = kc; aa.vc = vc; aa.n_past = d_npast; aa.E = E; aa.H = H; aa.N = N;
            aa.cols = s->cols; aa.sess_stride = s->sess_stride;
            aa.cs = s->cs; aa.texp = s->texp; aa.out = s->att;
            aa.n_ctx = s->n_ctx; aa.kq_scale = 1.0f / sqrtf((float) E / (float) H);
            const bool preq = s->wtype != kWT_F16;
            const float dsc = wt_nibbles(s->wtype) ? 0.0625f : 1.0f;
            if (preq) { aa.aq_out = s->aq_att; aa.da_out = s->da_att; aa.out_nbq = s->nbqE; aa.out_dscale = dsc; aa.out_soff = s->soffE; }
            AttnTiledArgs ta{};
            ta.q16 = s->q16; ta.kc = kc; ta.vc = vc; ta.n_past = d_npast; ta.E = E; ta.H = H; ta.N = N; ta.texp = s->texp; ta.out = s->att;
            if (preq) { ta.aq_out = s->aq_att; ta.da_out = s->da_att; ta.out_nbq = s->nbqE; ta.out_dscale = dsc; ta.out_soff = s->soffE; }
            ta.kq_scale = aa.kq_scale;
            if (s->cols && s->plan.ones) {
                // every column is an independent N = 1 step: the fused (RoPE + append) kernel, one cluster row per column
                s->cur_class = 2;
                for (int n0 = 0; n0 < N; n0 += kChunk) {
                    aa.n0 = n0;
                    const int cnt = N - n0 < kChunk ? N - n0 : kChunk;
                    if ((rc = launch_simple(s, k_attn128<true>, dim3(4 * H, cnt, 1), dim3(256, 1, 1), asm_bytes, aa))) return rc;
                }
            } else if (s->cols) {
                // mixed step: every RoPE + KV append first (a chunk's queries read the rows the other columns of their segment
                // append), then the tiled kernel over the query blocks of the chunks whose context fits the staged window, and
                // the cluster kernel over every other column
                s->cur_class = 1;
                RopeArgs ra{s->qkv, E, H, D, N, d_npast, s->cs, s->q16, kc, vc, s->cols, s->sess_stride};
                if ((rc = launch_simple(s, k_rope_append, dim3((E / 2 + 255) / 256, N, 1), dim3(256, 1, 1), 0, ra))) return rc;
                s->cur_class = 2;
                if (!s->plan.blocks.empty()) {
                    ta.blocks = s->d_blocks; ta.sess_stride = s->sess_stride; ta.t_rows = s->plan.t_rows;
                    if ((rc = launch_attn_tiled(s, ta, (int) s->plan.blocks.size()))) return rc;
                }
                aa.colmap = s->d_clist;
                const int ncl = (int) s->plan.clist.size();
                for (int n0 = 0; n0 < ncl; n0 += kChunk) {
                    aa.n0 = n0;
                    const int cnt = ncl - n0 < kChunk ? ncl - n0 : kChunk;
                    if ((rc = launch_simple(s, k_attn128<false>, dim3(4 * H, cnt, 1), dim3(256, 1, 1), asm_plain, aa))) return rc;
                }
            } else if (N == 1) {
                s->cur_class = 2;
                aa.n0 = 0;
                if (s->trace && s->trace_next < 512) { aa.trace = s->trace + (size_t) s->trace_next * 1024 * 8; s->trace_next++; s->trace_cls.push_back(2); s->trace_ctas.push_back(4 * H); }
                aa.lut_smem = 1;
                if ((rc = launch_simple(s, k_attn128<true>, dim3(4 * H, 1, 1), dim3(256, 1, 1), asm_lut, aa))) return rc;
            } else if (s->use_tiled_attn && s->past[s->cur] + N <= kAttnTMax) {
                // prompt chunk whose whole context fits the staged window: query-tiled kernel, K / V read once per 16 queries
                s->cur_class = 1;
                RopeArgs ra{s->qkv, E, H, D, N, d_npast, s->cs, s->q16, kc, vc, nullptr, 0};
                if ((rc = launch_simple(s, k_rope_append, dim3((E / 2 + 255) / 256, N, 1), dim3(256, 1, 1), 0, ra))) return rc;
                s->cur_class = 2;
                ta.t_rows = s->past[s->cur] + N;
                if ((rc = launch_attn_tiled(s, ta, (N + kAttnQB - 1) / kAttnQB))) return rc;
            } else {
                s->cur_class = 1;
                RopeArgs ra{s->qkv, E, H, D, N, d_npast, s->cs, s->q16, kc, vc, nullptr, 0};
                if ((rc = launch_simple(s, k_rope_append, dim3((E / 2 + 255) / 256, N, 1), dim3(256, 1, 1), 0, ra))) return rc;
                s->cur_class = 2;
                for (int n0 = 0; n0 < N; n0 += kChunk) {
                    aa.n0 = n0;
                    const int cnt = N - n0 < kChunk ? N - n0 : kChunk;
                    if ((rc = launch_simple(s, k_attn128<false>, dim3(4 * H, cnt, 1), dim3(256, 1, 1), asm_plain, aa))) return rc;
                }
            }
        } else {
            s->cur_class = 1;
            RopeArgs ra{s->qkv, E, H, D, N, d_npast, s->cs, s->q16, kc, vc, s->cols, s->sess_stride};
            if ((rc = launch_simple(s, k_rope_append, dim3((E / 2 + 255) / 256, N, 1), dim3(256, 1, 1), 0, ra))) return rc;
            s->cur_class = 2;
            AttnArgs aa{s->q16, kc, vc, d_npast, E, H, D, N, s->texp, s->att, 1.0f / sqrtf((float) E / (float) H), s->cols, s->sess_stride};
            const size_t asm_bytes = (size_t)((s->n_ctx + 3) & ~3) * 4 + (size_t)((s->n_ctx + 7) & ~7) * 2 + (size_t) 4 * D * 8 * 4 + 64;
            if ((rc = launch_simple(s, k_attention, dim3(H, N, 1), dim3(512, 1, 1), asm_bytes, aa))) return rc;
        }
        if (s->wtype == kWT_F16) {
            GemvF16Args f{}; f.K = E; f.x = s->att; f.ldx = E; f.N = N; f.tsilu = s->tsilu;
            s->cur_class = 3;
            f.rows = E; f.W = Lw.f_o; f.resid = cur; f.ldr = E; f.y = s->ffin; f.ldy = E;
            if ((rc = launch_f16<PRO_PLAIN, EPI_RESID>(s, f))) return rc;
            s->cur_class = 4;
            GemvF16Args g{}; g.K = E; g.x = s->ffin; g.ldx = E; g.norm_w = Lw.ffn_norm; g.N = N; g.tsilu = s->tsilu;
            g.rows = FF; g.W = Lw.f_1; g.W2 = Lw.f_3; g.y = s->gate; g.ldy = FF;
            if ((rc = launch_f16<PRO_NORM, EPI_GATE>(s, g))) return rc;
            s->cur_class = 5;
            GemvF16Args w{}; w.K = FF; w.x = s->gate; w.ldx = FF; w.N = N; w.tsilu = s->tsilu;
            w.rows = E; w.W = Lw.f_2; w.resid = s->ffin; w.ldr = E; w.y = nxt; w.ldy = E;
            if ((rc = launch_f16<PRO_PLAIN, EPI_RESID>(s, w))) return rc;
        } else if (fast) {
            s->cur_class = 3;
            if ((rc = launch_prep<false>(s, s->att, E, nullptr, E, N))) return rc;
            if ((rc = launch_fast_any<FG_RESID>(s, Lw.wo, cur, E, s->ffin, E, N, E))) return rc;
            s->cur_class = 4;
            if ((rc = launch_prep<true>(s, s->ffin, E, Lw.ffn_norm, E, N))) return rc;
            if ((rc = launch_fast_any<FG_GATE>(s, Lw.w13, nullptr, 0, s->gate, FF, N, FF))) return rc;
            s->cur_class = 5;
            if ((rc = launch_prep<false>(s, s->gate, FF, nullptr, FF, N))) return rc;
            if ((rc = launch_fast_any<FG_RESID>(s, Lw.w2, s->ffin, E, nxt, E, N, E))) return rc;
        } else {
            const float dsc = wt_nibbles(s->wtype) ? 0.0625f : 1.0f;
            s->cur_class = 3;
            GemvArgs o{}; o.W = Lw.wo; o.x = s->att; o.ldx = E; o.resid = cur; o.ldr = E; o.y = s->ffin; o.ldy = E;
            o.N = N; o.out_rows = E; o.tsilu = s->tsilu; o.aq_in = s->aq_att; o.da_in = s->da_att; o.in_soff = s->soffE; o.out_soff = s->soffE;
            o.nq_norm_w = Lw.ffn_norm; o.nq_counter = s->nq_counter; o.nq_partial = s->nq_partial; o.aq_out = s->aq_x; o.da_out = s->da_x; o.out_nbq = s->nbqE; o.out_dscale = dsc;
            if (D == 128) {
                if (nq) { if ((rc = launch_gemv<1, PRO_PREQ, EPI_RESID_NQ>(s, o))) return rc; }
                else if (gemv8_applicable(s, Lw.wo, N)) { if ((rc = launch_gemv8<EPI_RESID>(s, o))) return rc; }
                else    { if ((rc = launch_gemv<1, PRO_PREQ, EPI_RESID>(s, o))) return rc; }
            } else {
                if (nq) { if ((rc = launch_gemv<1, PRO_PLAIN, EPI_RESID_NQ>(s, o))) return rc; }
                else    { if ((rc = launch_gemv<1, PRO_PLAIN, EPI_RESID>(s, o))) return rc; }
            }
            s->cur_class = 4;
            GemvArgs g{}; g.W = Lw.w13; g.x = s->ffin; g.ldx = E; g.norm_w = Lw.ffn_norm; g.y = s->gate; g.ldy = FF;
            g.N = N; g.out_rows = FF; g.tsilu = s->tsilu; g.aq_in = s->aq_x; g.da_in = s->da_x; g.in_soff = s->soffE; g.out_soff = s->soffF;
            g.aq_out = s->aq_gate; g.da_out = s->da_gate; g.out_nbq = s->nbqF; g.out_dscale = dsc;
            if (nq) { if ((rc = launch_gemv<2, PRO_PREQ, EPI_GATEQ>(s, g))) return rc; }
            else if (N > 1) {
                if ((rc = launch_norm_quant(s, s->ffin, E, Lw.ffn_norm, N))) return rc;
                if ((rc = launch_gemv<2, PRO_PREQ, EPI_GATEQ>(s, g))) return rc;
            }
            else    { if ((rc = launch_gemv<2, PRO_NORM, EPI_GATEQ>(s, g))) return rc; }
            s->cur_class = 5;
            GemvArgs w{}; w.W = Lw.w2; w.resid = s->ffin; w.ldr = E; w.y = nxt; w.ldy = E;
            w.N = N; w.out_rows = E; w.tsilu = s->tsilu; w.aq_in = s->aq_gate; w.da_in = s->da_gate; w.in_soff = s->soffF; w.out_soff = s->soffE;
            if (il + 1 < s->L && nq) {
                w.nq_norm_w = s->layers[il + 1].attn_norm; w.nq_counter = s->nq_counter; w.nq_partial = s->nq_partial; w.aq_out = s->aq_x; w.da_out = s->da_x;
                w.out_nbq = s->nbqE; w.out_dscale = dsc;
                if ((rc = launch_gemv<1, PRO_PREQ, EPI_RESID_NQ>(s, w))) return rc;
            } else if (s->fold_send && il == s->L - 1) {
                w.mb_mine = (MailboxHdr *) s->mb_block;
                w.mb_peer_inbox = (uint2 *)(s->mb_next + sizeof(MailboxHdr)); w.mb_slot_elems = s->mb_slot_floats;
                if (gemv8_applicable(s, Lw.w2, N)) rc = launch_gemv8<EPI_RESID_SEND>(s, w);
                else if (s->wtype == kWT_Q4_0) rc = launch_gemv_t<kWT_Q4_0, 1, 1, PRO_PREQ, EPI_RESID_SEND, true>(s, w);
                else if (s->wtype == kWT_Q4_1) rc = launch_gemv_t<kWT_Q4_1, 1, 1, PRO_PREQ, EPI_RESID_SEND, true>(s, w);
                else                           rc = launch_gemv_t<kWT_Q8_0, 1, 1, PRO_PREQ, EPI_RESID_SEND, true>(s, w);
                if (rc) return rc;
            } else if (gemv8_applicable(s, Lw.w2, N)) { if ((rc = launch_gemv8<EPI_RESID>(s, w))) return rc; }
            else if ((rc = launch_gemv<1, PRO_PREQ, EPI_RESID>(s, w))) return rc;
        }
        cur = nxt;
    }
    if (s->send_pending) {
        // pipeline hand-off: the activation leaves for the next slice's GPU right behind the last matmul
        s->send_pending = false;
        s->cur_class = 6;
        int rc = launch_simple(s, k_peer_send, dim3(s->send_ctas, 1, 1), dim3(1024, 1, 1), 0, s->send_args);
        if (rc) return rc;
    }
    {
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3(1); cfg.blockDim = dim3(32); cfg.stream = s->stream;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = at; cfg.numAttrs = s->use_pdl ? 1 : 0;
        s->cur_class = 6;
        prof_begin(s);
        if (s->cols) B200_CUDA(cudaLaunchKernelEx(&cfg, k_advance_segs, s->d_npast, s->cols, N));
        else if (s->fold_send) B200_CUDA(cudaLaunchKernelEx(&cfg, k_advance_sent, s->d_npast + s->cur, N, (MailboxHdr *) s->mb_block));
        else         B200_CUDA(cudaLaunchKernelEx(&cfg, k_advance, s->d_npast + s->cur, N));
        prof_end(s);
        s->launches++;
    }
    return 0;
}

// N = 1: replay a captured graph (host variant adds the H2D / D2H copies as graph nodes)
static int run_decode_graph(b200_slice * s, const float * in, float * out, bool host) {
    GraphKey key{in, out, (host ? 1 : 0) | (s->skip_attention ? 2 : 0) | (s->send_pending ? 4 : 0) | (s->cur << 3)};
    auto it = s->graphs.find(key);
    const int per_step = persist_applicable(s, 1) ? 2 : (s->D == 128 ? 5 : 6) * s->L + 1;
    if (persist_applicable(s, 1)) { int rc = persist_prepare(s, host ? s->d_in : in, host ? s->d_out : out); if (rc) return rc; }
    if (it == s->graphs.end()) {
        const int64_t before = s->launches;
        cudaGraph_t g = nullptr;
        B200_CUDA(cudaStreamBeginCapture(s->stream, cudaStreamCaptureModeThreadLocal));
        int rc = 0;
        if (host) {
            cudaMemcpyAsync(s->d_in, s->h_in, (size_t) s->E * 4, cudaMemcpyHostToDevice, s->stream);
            rc = enqueue_layers(s, s->d_in, 1, s->d_out);
            cudaMemcpyAsync(s->h_out, s->d_out, (size_t) s->E * 4, cudaMemcpyDeviceToHost, s->stream);
        } else {
            rc = enqueue_layers(s, in, 1, out);
        }
        cudaError_t e = cudaStreamEndCapture(s->stream, &g);
        s->launches = before;
        if (rc) { if (g) cudaGraphDestroy(g); return rc; }
        if (e != cudaSuccess) return fail(B200_ECUDA, "graph capture failed: %s", cudaGetErrorString(e));
        cudaGraphExec_t ge = nullptr;
        e = cudaGraphInstantiate(&ge, g, 0);
        cudaGraphDestroy(g);
        if (e != cudaSuccess) return fail(B200_ECUDA, "cudaGraphInstantiate failed: %s", cudaGetErrorString(e));
        if (s->graphs.size() >= 64)      // one graph per (buffers, session): enough for a node serving dozens of sessions
            { for (auto & kv : s->graphs) cudaGraphExecDestroy(kv.second); s->graphs.clear(); }
        it = s->graphs.emplace(key, ge).first;
    }
    B200_CUDA(cudaGraphLaunch(it->second, s->stream));
    s->launches += per_step;
    return 0;
}

static int forward_locked(b200_slice * s, const float * in, int N, float * out, bool host, int session = 0) {
    if (N <= 0) return fail(B200_EINVAL, "n_tokens must be positive (got %d)", N);
    if (session < 0 || session >= s->n_sessions) return fail(B200_EINVAL, "session %d outside [0, %d)", session, s->n_sessions);
    if (s->past[session] + N > s->n_ctx)
        return fail(B200_ECONTEXT, "context overflow: n_past %d + n_tokens %d > n_ctx %d", s->past[session], N, s->n_ctx);
    B200_CUDA(cudaSetDevice(s->device));
    s->cur = session; s->cols = nullptr;
    B200_CUDA(cudaEventRecord(s->ev0, s->stream));
    int rc;
    if (host) {
        if (N == 1 && s->use_graph && !s->profiling) {
            memcpy(s->h_in, in, (size_t) s->E * 4);
            if ((rc = run_decode_graph(s, nullptr, nullptr, true))) return rc;
            B200_CUDA(cudaEventRecord(s->ev1, s->stream));
            // A decoded token is ~1 ms of GPU work.  A blocking synchronize adds the wake-up latency of the driver's
            // interrupt path to every token; polling from the start burns a core for the whole token.  So: sleep through
            // ~70 % of the smoothed token time, poll the rest, and block if the token takes unusually long.
            if (s->ema_token_ms > 0.2f)
                std::this_thread::sleep_for(std::chrono::microseconds((long)(700.f * s->ema_token_ms)));
            for (int spin = 0; spin < 100000; spin++) if (cudaEventQuery(s->ev1) != cudaErrorNotReady) break;
            B200_CUDA(cudaStreamSynchronize(s->stream));
            { float ms = 0.f; if (cudaEventElapsedTime(&ms, s->ev0, s->ev1) == cudaSuccess && ms > 0.f)
                  s->ema_token_ms = s->ema_token_ms > 0.f ? 0.8f * s->ema_token_ms + 0.2f * ms : ms; }
            memcpy(out, s->h_out, (size_t) s->E * 4);
        } else {
            B200_CUDA(cudaMemcpyAsync(s->d_in, in, (size_t) N * s->E * 4, cudaMemcpyHostToDevice, s->stream));
            if (persist_applicable(s, N) && (rc = persist_prepare(s, s->d_in, s->d_out))) return rc;
            if ((rc = enqueue_layers(s, s->d_in, N, s->d_out))) return rc;
            B200_CUDA(cudaEventRecord(s->ev1, s->stream));
            B200_CUDA(cudaMemcpyAsync(out, s->d_out, (size_t) N * s->E * 4, cudaMemcpyDeviceToHost, s->stream));
            B200_CUDA(cudaStreamSynchronize(s->stream));
        }
    } else {
        if (N == 1 && s->use_graph && !s->profiling) { if ((rc = run_decode_graph(s, in, out, false))) return rc; }
        else {
            if (persist_applicable(s, N) && (rc = persist_prepare(s, in, out))) return rc;
            if ((rc = enqueue_layers(s, in, N, out))) return rc;
        }
        B200_CUDA(cudaEventRecord(s->ev1, s->stream));
    }
    s->timed = true;
    s->past[session] += N;
    return 0;
}

// A step over n_seg DISTINCT sessions in a single pass: segment i is n_tokens[i] consecutive tokens of sessions[i] (n_tokens
// == nullptr: one token each, the batched step).  The weight matmuls see all columns at once (weights read once); RoPE, KV
// append and attention run per column against that session's cache.  Column n of segment i carries T_i = n_past_i + len_i,
// the row length the reference's V.p of that call splits into 32-slot body and double tail, so every segment's rows are
// bit-identical to a forward of that session alone.  Checks every segment before anything is enqueued: a rejected step changes
// nothing.  Fills s->plan; *rows = the step's column count.
static int plan_step(b200_slice * s, const int * sessions, const int * n_tokens, int n_seg, int * rows) {
    if (n_seg <= 0 || n_seg > s->n_sessions) return fail(B200_EINVAL, "step over %d sessions with %d sessions", n_seg, s->n_sessions);
    std::vector<char> seen(s->n_sessions, 0);
    long long total = 0;
    for (int i = 0; i < n_seg; i++) {
        const int k = sessions[i], len = n_tokens ? n_tokens[i] : 1;
        if (k < 0 || k >= s->n_sessions) return fail(B200_EINVAL, "session %d outside [0, %d)", k, s->n_sessions);
        if (seen[k]) return fail(B200_EINVAL, "session %d listed twice in one step", k);
        if (len <= 0) return fail(B200_EINVAL, "segment %d of session %d has %d tokens", i, k, len);
        seen[k] = 1;
        total += len;
    }
    if (total > s->n_ctx) return fail(B200_EINVAL, "step of %lld tokens exceeds n_ctx %d", total, s->n_ctx);
    for (int i = 0; i < n_seg; i++) {
        const int k = sessions[i], len = n_tokens ? n_tokens[i] : 1;
        if (s->past[k] + len > s->n_ctx)
            return fail(B200_ECONTEXT, "context overflow: session %d n_past %d + %d > n_ctx %d", k, s->past[k], len, s->n_ctx);
    }
    StepPlan & P = s->plan;
    P.segs.clear(); P.cols.clear(); P.blocks.clear(); P.clist.clear(); P.t_rows = 0; P.ones = true;
    for (int i = 0; i < n_seg; i++) {
        const int k = sessions[i], len = n_tokens ? n_tokens[i] : 1, p0 = s->past[k], T = p0 + len, c0 = (int) P.cols.size();
        P.segs.push_back(make_int2(k, len));
        P.ones = P.ones && len == 1;
        for (int j = 0; j < len; j++) P.cols.push_back(make_int4(k, p0 + j, T, 0));
        // head size 128: the same choice a prompt chunk of this session alone gets (enqueue_layers, N > 1)
        if (s->D == 128 && len > 1 && s->use_tiled_attn && T <= kAttnTMax) {
            for (int j = 0; j < len; j += kAttnQB) P.blocks.push_back(AttnBlock{c0 + j, std::min(kAttnQB, len - j), k, p0 + j, T});
            P.t_rows = std::max(P.t_rows, T);
        } else {
            for (int j = 0; j < len; j++) P.clist.push_back(c0 + j);
        }
    }
    *rows = (int) total;
    return 0;
}

// Copy s->plan's tables to the device and put the slice in multi-session mode (s->cols) for enqueue_layers.
static int upload_plan(b200_slice * s) {
    const StepPlan & P = s->plan;
    // pageable sources: the driver stages them before returning, so the next plan may overwrite the vectors
    B200_CUDA(cudaMemcpyAsync(s->d_cols, P.cols.data(), P.cols.size() * sizeof(int4), cudaMemcpyHostToDevice, s->stream));
    if (!P.ones && !P.blocks.empty())
        B200_CUDA(cudaMemcpyAsync(s->d_blocks, P.blocks.data(), P.blocks.size() * sizeof(AttnBlock), cudaMemcpyHostToDevice, s->stream));
    if (!P.ones && !P.clist.empty())
        B200_CUDA(cudaMemcpyAsync(s->d_clist, P.clist.data(), P.clist.size() * sizeof(int), cudaMemcpyHostToDevice, s->stream));
    s->cur = 0; s->cols = s->d_cols;
    return 0;
}

static void commit_plan(b200_slice * s) { for (const int2 & g : s->plan.segs) s->past[g.x] += g.y; }

// Enqueue the step s->plan describes (N columns) and advance its sessions.
static int run_plan(b200_slice * s, int N, const float * in, float * out, bool host) {
    int rc;
    B200_CUDA(cudaSetDevice(s->device));
    B200_CUDA(cudaEventRecord(s->ev0, s->stream));
    if ((rc = upload_plan(s))) { s->cols = nullptr; return rc; }
    if (host) {
        B200_CUDA(cudaMemcpyAsync(s->d_in, in, (size_t) N * s->E * 4, cudaMemcpyHostToDevice, s->stream));
        rc = enqueue_layers(s, s->d_in, N, s->d_out);
        s->cols = nullptr;
        if (rc) return rc;
        B200_CUDA(cudaEventRecord(s->ev1, s->stream));
        B200_CUDA(cudaMemcpyAsync(out, s->d_out, (size_t) N * s->E * 4, cudaMemcpyDeviceToHost, s->stream));
        B200_CUDA(cudaStreamSynchronize(s->stream));
    } else {
        rc = enqueue_layers(s, in, N, out);
        s->cols = nullptr;
        if (rc) return rc;
        B200_CUDA(cudaEventRecord(s->ev1, s->stream));
    }
    s->timed = true;
    commit_plan(s);
    return 0;
}

static int mixed_locked(b200_slice * s, const int * sessions, const int * n_tokens, int n_seg, const float * in, float * out, bool host) {
    int N = 0;
    const int rc = plan_step(s, sessions, n_tokens, n_seg, &N);
    return rc ? rc : run_plan(s, N, in, out, host);
}

// ---------------------------------------------------------------- loader
// file (mmap, page cache) --reader thread--> pinned staging ring --DMA--> device scratch ring --k_repack--> packed HBM.
// Three slots are in flight: while slot j is repacked on the GPU, slot j+1 is on the PCIe bus and the reader thread is
// faulting slot j+2 in from the page cache.  Nothing synchronises the stream per matrix; a slot is reused once the
// event recorded behind its repack kernel has completed (the reader thread waits for it).
struct LoadJob {
    const GgjtTensor * src[3] = {nullptr, nullptr, nullptr};
    int nsrc = 0;
    int kind = 0;                 // 0: block-quantised matrix (k_repack), 1: F16 (k_repack_f16), 2: raw copy, 3: Q6_K (k_repack_q6k)
    int mode = 0, G = 1;
    PackedW * out = nullptr;      // kind 0
    PackedW * out2 = nullptr; int TR2 = 0;   // kind 0: a second packing of the same matrix with TR2 row-groups per tile
    uint16_t ** outf = nullptr; uint16_t * into = nullptr;   // kind 1
    uint8_t * raw_dst = nullptr;  // kind 2
    size_t bytes() const { size_t n = 0; for (int i = 0; i < nsrc; i++) n += (src[i]->nbytes + 255) & ~(size_t) 255; return n; }
};

struct LoadPipe {
    static constexpr int NB = 3;
    uint8_t * pinned[NB] = {nullptr, nullptr, nullptr};
    uint8_t * scratch[NB] = {nullptr, nullptr, nullptr};
    cudaEvent_t ev[NB] = {nullptr, nullptr, nullptr};
    size_t slot_bytes = 0;
    ~LoadPipe() {
        for (int i = 0; i < NB; i++) {
            if (pinned[i]) cudaFreeHost(pinned[i]);
            if (scratch[i]) cudaFree(scratch[i]);
            if (ev[i]) cudaEventDestroy(ev[i]);
        }
    }
};

static int run_load_jobs(b200_slice * s, const GgjtFile & f, std::vector<LoadJob> & jobs) {
    if (jobs.empty()) return 0;
    LoadPipe lp;
    for (const LoadJob & j : jobs) lp.slot_bytes = std::max(lp.slot_bytes, j.bytes());
    lp.slot_bytes += 4096;
    for (int i = 0; i < LoadPipe::NB; i++) {
        B200_CUDA(cudaMallocHost((void **) &lp.pinned[i], lp.slot_bytes));
        B200_CUDA(cudaMalloc((void **) &lp.scratch[i], lp.slot_bytes));
        B200_CUDA(cudaEventCreateWithFlags(&lp.ev[i], cudaEventDisableTiming));
    }
    posix_fadvise(f.fd, 0, 0, POSIX_FADV_SEQUENTIAL);       // a cold file: deep kernel read-ahead in front of the preads
    std::mutex mu; std::condition_variable cv;
    size_t filled = 0, consumed = 0; bool abort_flag = false;
    const int device = s->device;
    std::thread reader([&] {
        cudaSetDevice(device);
        for (size_t j = 0; j < jobs.size(); j++) {
            const int slot = (int)(j % LoadPipe::NB);
            {
                std::unique_lock<std::mutex> lk(mu);
                cv.wait(lk, [&] { return abort_flag || consumed + LoadPipe::NB > j; });
                if (abort_flag) return;
            }
            if (j >= LoadPipe::NB) cudaEventSynchronize(lp.ev[slot]);    // the slot's previous repack has read its scratch
            // pread straight into the pinned slot: page-cache copy without the per-4-KiB minor faults a private file
            // mapping costs; the job is cut in two so a second thread overlaps its copy
            struct Piece { uint8_t * dst; size_t off, n; };
            std::vector<Piece> pieces;
            size_t off = 0;
            for (int i = 0; i < jobs[j].nsrc; i++) {
                const GgjtTensor & t = *jobs[j].src[i];
                const size_t half = (t.nbytes / 2) & ~(size_t) 4095;
                pieces.push_back({lp.pinned[slot] + off, t.offset, half});
                pieces.push_back({lp.pinned[slot] + off + half, t.offset + half, t.nbytes - half});
                off += (t.nbytes + 255) & ~(size_t) 255;
            }
            auto pull = [&](int first) {
                for (size_t k = first; k < pieces.size(); k += 2) {
                    size_t done = 0;
                    while (done < pieces[k].n) {
                        const ssize_t got = pread(f.fd, pieces[k].dst + done, pieces[k].n - done, (off_t)(pieces[k].off + done));
                        if (got <= 0) { memcpy(pieces[k].dst + done, f.base + pieces[k].off + done, pieces[k].n - done); break; }
                        done += (size_t) got;
                    }
                }
            };
            std::thread helper(pull, 1);
            pull(0);
            helper.join();
            { std::lock_guard<std::mutex> lk(mu); filled = j + 1; }
            cv.notify_all();
        }
    });
    int rc = 0;
    for (size_t j = 0; j < jobs.size() && !rc; j++) {
        const int slot = (int)(j % LoadPipe::NB);
        LoadJob & job = jobs[j];
        { std::unique_lock<std::mutex> lk(mu); cv.wait(lk, [&] { return filled > j; }); }
        cudaError_t e = cudaMemcpyAsync(lp.scratch[slot], lp.pinned[slot], job.bytes(), cudaMemcpyHostToDevice, s->stream);
        if (e != cudaSuccess) { rc = fail(B200_ECUDA, "weight upload failed: %s", cudaGetErrorString(e)); break; }
        if (job.kind == 0) {
            const int wt = (int) job.src[0]->type;
            const int K = (int) job.src[0]->ne[0], rows_per = (int) job.src[0]->ne[1];
            const int nb = K / 32, nbq = ((nb + 3) / 4 + kQS - 1) / kQS * kQS, TR = kWPC * job.G;
            const int total_groups = (rows_per + 7) / 8 * job.nsrc;
            const int n_tiles = (total_groups + TR - 1) / TR;
            const long long tile_bytes = (long long) nbq * TR * chunk_bytes(wt);
            uint8_t * dst = nullptr;
            if ((rc = dev_alloc(s, &dst, (size_t) n_tiles * tile_bytes))) break;
            RepackArgs ra{};
            size_t off = 0;
            for (int i = 0; i < job.nsrc; i++) { ra.src[i] = lp.scratch[slot] + off; off += (job.src[i]->nbytes + 255) & ~(size_t) 255; }
            ra.mode = job.mode; ra.wtype = wt; ra.rows_per_src = rows_per; ra.nb = nb; ra.nbq = nbq; ra.TR = TR; ra.n_tiles = n_tiles;
            ra.dst = dst;
            k_repack<<<s->n_sm * 8, 256, 0, s->stream>>>(ra);
            PackedW * out = job.out;
            out->data = dst; out->wtype = wt; out->rows = rows_per * job.nsrc; out->K = K; out->nb = nb; out->nbq = nbq; out->TR = TR;
            out->n_tiles = n_tiles; out->tile_bytes = tile_bytes;
            if (job.out2 && job.TR2 > 0) {
                const int TR2 = job.TR2, n_tiles2 = (total_groups + TR2 - 1) / TR2;
                // quads per ring stage of the persistent kernel: sq * TR2 <= 16; pad nbq so a whole number of stages fits
                int sq = 16 / TR2; while (sq > 4 && nbq % sq) sq >>= 1;
                const long long tile_bytes2 = (long long) nbq * TR2 * chunk_bytes(wt);
                uint8_t * dst2 = nullptr;
                if ((rc = dev_alloc(s, &dst2, (size_t) n_tiles2 * tile_bytes2))) break;
                ra.TR = TR2; ra.n_tiles = n_tiles2; ra.dst = dst2;
                k_repack<<<s->n_sm * 8, 256, 0, s->stream>>>(ra);
                PackedW * o2 = job.out2;
                *o2 = *out; o2->data = dst2; o2->TR = TR2; o2->n_tiles = n_tiles2; o2->tile_bytes = tile_bytes2;
            }
        } else if (job.kind == 1) {
            const GgjtTensor & t = *job.src[0];
            const int K = (int) t.ne[0], rows = (int) t.ne[1];
            const int nchunk = K / 32, nc8 = (nchunk + 7) / 8;
            uint16_t * dst = job.into;
            if (!dst && (rc = dev_alloc(s, &dst, (size_t) rows * nc8 * 256 + 8))) break;
            k_repack_f16<<<s->n_sm * 8, 256, 0, s->stream>>>((const uint16_t *) lp.scratch[slot], dst, dst /*no tail: K%32==0*/, rows, K);
            *job.outf = dst;
        } else if (job.kind == 3) {
            const GgjtTensor & t = *job.src[0];
            k_repack_q6k<<<s->n_sm * 8, 256, 0, s->stream>>>(lp.scratch[slot], job.raw_dst, (int) t.ne[1], (int) t.ne[0] / 256);
        } else {
            e = cudaMemcpyAsync(job.raw_dst, lp.scratch[slot], job.src[0]->nbytes, cudaMemcpyDeviceToDevice, s->stream);
            if (e != cudaSuccess) { rc = fail(B200_ECUDA, "weight copy failed: %s", cudaGetErrorString(e)); break; }
        }
        if ((e = cudaGetLastError()) != cudaSuccess) { rc = fail(B200_ECUDA, "repack launch failed: %s", cudaGetErrorString(e)); break; }
        cudaEventRecord(lp.ev[slot], s->stream);
        { std::lock_guard<std::mutex> lk(mu); consumed = j + 1; }
        cv.notify_all();
    }
    { std::lock_guard<std::mutex> lk(mu); abort_flag = rc != 0; consumed = jobs.size() + LoadPipe::NB; }
    cv.notify_all();
    reader.join();
    cudaError_t e = cudaStreamSynchronize(s->stream);
    if (!rc && e != cudaSuccess) rc = fail(B200_ECUDA, "weight repack failed: %s", cudaGetErrorString(e));
    return rc;
}

static int build_tables(b200_slice * s) {
    // fp16 lookup tables of ggml_init (ggml.c:4300-4312), built with the host libm like the reference does
    std::vector<uint16_t> texp(65536), tsilu(65536);
    for (int i = 0; i < 65536; i++) {
        const float f = __half2float(__ushort_as_half((unsigned short) i));
        texp[i]  = __half_as_ushort(__float2half_rn(expf(f)));
        tsilu[i] = __half_as_ushort(__float2half_rn(f / (1.0f + expf(-f))));
    }
    int rc;
    if ((rc = dev_alloc(s, &s->texp, 65536)) || (rc = dev_alloc(s, &s->tsilu, 65536))) return rc;
    B200_CUDA(cudaMemcpy(s->texp, texp.data(), 65536 * 2, cudaMemcpyHostToDevice));
    B200_CUDA(cudaMemcpy(s->tsilu, tsilu.data(), 65536 * 2, cudaMemcpyHostToDevice));
    // RoPE cos/sin, theta iterated in f32 (ggml.c:12000, 12038-12044)
    const int half = s->D / 2;
    std::vector<float2> cs((size_t) s->n_ctx * half);
    const float theta_scale = powf(10000.0, -2.0f / s->D);
    for (int p = 0; p < s->n_ctx; p++) {
        float theta = (float) p;
        for (int j = 0; j < half; j++) {
            cs[(size_t) p * half + j] = make_float2(cosf(theta), sinf(theta));
            theta *= theta_scale;
        }
    }
    if ((rc = dev_alloc(s, &s->cs, cs.size()))) return rc;
    B200_CUDA(cudaMemcpy(s->cs, cs.data(), cs.size() * sizeof(float2), cudaMemcpyHostToDevice));
    return 0;
}

static int load_locked(b200_slice * s, const char * path) {
    const bool ltrace = env_int("B200_LOAD_TRACE", 0) != 0;
    auto tnow = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double t_begin = tnow(); double t_last = t_begin;
    auto lap = [&](const char * what) { if (ltrace) { const double t = tnow(); fprintf(stderr, "[b200 load] %-28s %7.3f s\n", what, t - t_last); t_last = t; } };
    std::unique_ptr<GgjtFile> fp;
    try { fp.reset(new GgjtFile(path, false)); }
    catch (const std::exception & e) { return fail(B200_EFILE, "error loading model: %s", e.what()); }
    GgjtFile & f = *fp;
    lap("parse header + tensor index");
    if (f.n_layer == 0 || f.n_head == 0 || f.n_embd % f.n_head || f.n_embd % 32)
        return fail(B200_EFILE, "not a transformer slice file (n_layer=%u n_embd=%u n_head=%u)", f.n_layer, f.n_embd, f.n_head);
    s->E = (int) f.n_embd; s->H = (int) f.n_head; s->D = s->E / s->H; s->L = (int) f.n_layer; s->first_layer = (int) f.first_layer;
    s->FF = (int)(((2 * (4 * f.n_embd) / 3 + f.n_mult - 1) / f.n_mult) * f.n_mult);   // tensor_processor.cpp:1250
    if (s->D > 128 || (s->D & 1)) return fail(B200_EFILE, "head size %d unsupported (<=128, even)", s->D);
    {
        // worst-case dynamic shared memory of the attention kernels at this n_ctx (scores f32 + probabilities f16 per
        // position, + staged rows / exp table / partials): reject the load instead of failing every forward later
        const size_t sc_bytes = (((size_t)((s->n_ctx + 3) & ~3) * 4 + (size_t)((s->n_ctx + 7) & ~7) * 2) + 15) & ~(size_t) 15;
        int pf_rows = 8 * ((s->n_ctx + 31) / 32); if (pf_rows > 128) pf_rows = 128;
        const size_t need128 = sc_bytes + (size_t) 2 * pf_rows * kAttnRow + 32 * 64 + 64 + 65536;
        const size_t need_gen = (size_t)((s->n_ctx + 3) & ~3) * 4 + (size_t)((s->n_ctx + 7) & ~7) * 2 + (size_t) 4 * s->D * 8 * 4 + 64;
        const size_t need = s->D == 128 ? need128 : need_gen, limit = s->D == 128 ? (size_t) 200 * 1024 : (size_t) kSmemLimit;
        if (need > limit)
            return fail(B200_EINVAL, "n_ctx %d needs %zu B of attention shared memory (limit %zu B): largest supported n_ctx for head size %d is %d",
                        s->n_ctx, need, limit, s->D, s->D == 128 ? (int)((limit - 2 * 128 * kAttnRow - 32 * 64 - 64 - 65536 - 16) / 6) & ~31
                                                                 : (int)((limit - (size_t) 4 * s->D * 32 - 64) / 6) & ~31);
    }
    const uint32_t E = f.n_embd, FF = (uint32_t) s->FF;
    s->layers.resize(s->L);
    int rc;
    std::vector<LoadJob> jobs;
    std::vector<float> norms;                       // all norm weights, one upload
    try {
        const std::string p0 = "layers." + std::to_string(s->first_layer);
        s->wtype = (int) f.get(p0 + ".attention.wq.weight", {E, E}).type;
        if (s->wtype != kWT_Q4_0 && s->wtype != kWT_Q4_1 && s->wtype != kWT_Q8_0 && s->wtype != kWT_F16)
            return fail(B200_EFILE, "weight type %d unsupported (Q4_0, Q4_1, Q8_0, F16)", s->wtype);
        float * d_norms = nullptr;
        if ((rc = dev_alloc(s, &d_norms, (size_t) s->L * 2 * E))) return rc;
        norms.resize((size_t) s->L * 2 * E);
        for (int i = 0; i < s->L; i++) {
            const std::string p = "layers." + std::to_string(i + s->first_layer);
            LayerW & Lw = s->layers[i];
            const GgjtTensor & an = f.get(p + ".attention_norm.weight", {E});
            const GgjtTensor & wq = f.get(p + ".attention.wq.weight", {E, E});
            const GgjtTensor & wk = f.get(p + ".attention.wk.weight", {E, E});
            const GgjtTensor & wv = f.get(p + ".attention.wv.weight", {E, E});
            const GgjtTensor & wo = f.get(p + ".attention.wo.weight", {E, E});
            const GgjtTensor & fn = f.get(p + ".ffn_norm.weight", {E});
            const GgjtTensor & w1 = f.get(p + ".feed_forward.w1.weight", {E, FF});
            const GgjtTensor & w2 = f.get(p + ".feed_forward.w2.weight", {FF, E});
            const GgjtTensor & w3 = f.get(p + ".feed_forward.w3.weight", {E, FF});
            if (an.type != GT_F32 || fn.type != GT_F32) return fail(B200_EFILE, "norm weights must be F32");
            for (const GgjtTensor * t : {&wq, &wk, &wv, &wo, &w1, &w2, &w3})
                if ((int) t->type != s->wtype) return fail(B200_EFILE, "mixed weight types in slice (%s)", t->name.c_str());
            Lw.attn_norm = d_norms + (size_t) i * 2 * E; Lw.ffn_norm = Lw.attn_norm + E;
            memcpy(norms.data() + (size_t) i * 2 * E, f.data(an), (size_t) E * 4);
            memcpy(norms.data() + (size_t) i * 2 * E + E, f.data(fn), (size_t) E * 4);
            if (s->wtype == kWT_F16) {
                const GgjtTensor * ts[7] = {&wq, &wk, &wv, &wo, &w1, &w2, &w3};
                uint16_t ** dst[7] = {&Lw.f_q, &Lw.f_k, &Lw.f_v, &Lw.f_o, &Lw.f_1, &Lw.f_2, &Lw.f_3};
                const size_t per = (size_t) E * ((E / 32 + 7) / 8) * 256;          // packed elements of one E x E matrix
                uint16_t * qkv_buf = nullptr;
                if ((rc = dev_alloc(s, &qkv_buf, 3 * per + 8))) return rc;
                for (int k = 0; k < 7; k++) {
                    LoadJob j; j.kind = 1; j.nsrc = 1; j.src[0] = ts[k]; j.outf = dst[k]; j.into = k < 3 ? qkv_buf + k * per : nullptr;
                    jobs.push_back(j);
                }
            } else {
                LoadJob a; a.nsrc = 3; a.src[0] = &wq; a.src[1] = &wk; a.src[2] = &wv; a.mode = 1; a.G = 1; a.out = &Lw.qkv; jobs.push_back(a);
                LoadJob o; o.nsrc = 1; o.src[0] = &wo; o.mode = 0; o.G = 1; o.out = &Lw.wo;
                jobs.push_back(o);
                LoadJob g; g.nsrc = 2; g.src[0] = &w1; g.src[1] = &w3; g.mode = 2; g.G = 2; g.out = &Lw.w13; jobs.push_back(g);
                LoadJob d; d.nsrc = 1; d.src[0] = &w2; d.mode = 0; d.G = 1; d.out = &Lw.w2;
                jobs.push_back(d);
            }
            s->weight_bytes += (int64_t)(an.nbytes + fn.nbytes + wq.nbytes + wk.nbytes + wv.nbytes + wo.nbytes + w1.nbytes + w2.nbytes + w3.nbytes);
        }
        B200_CUDA(cudaMemcpyAsync(d_norms, norms.data(), norms.size() * 4, cudaMemcpyHostToDevice, s->stream));
        if ((rc = run_load_jobs(s, f, jobs))) return rc;
    } catch (const std::exception & e) {
        return fail(B200_EFILE, "error loading model: %s", e.what());
    }
    lap("weights: read + upload + repack");

    const size_t nE = (size_t) s->n_ctx * E;
    s->sess_stride = (size_t) s->L * nE;
    s->past.assign(s->n_sessions, 0);
    if ((rc = dev_alloc(s, &s->kc, s->n_sessions * s->sess_stride)) || (rc = dev_alloc(s, &s->vc, s->n_sessions * s->sess_stride)) ||
        (rc = dev_alloc(s, &s->d_cols, (size_t) s->n_ctx)) || (rc = dev_alloc(s, &s->d_blocks, (size_t) s->n_ctx)) ||
        (rc = dev_alloc(s, &s->d_clist, (size_t) s->n_ctx)) ||
        (rc = dev_alloc(s, &s->q16, nE)) || (rc = dev_alloc(s, &s->xa, nE)) || (rc = dev_alloc(s, &s->xb, nE)) ||
        (rc = dev_alloc(s, &s->qkv, 3 * nE)) || (rc = dev_alloc(s, &s->att, nE)) || (rc = dev_alloc(s, &s->ffin, nE)) ||
        (rc = dev_alloc(s, &s->gate, (size_t) s->n_ctx * FF)) || (rc = dev_alloc(s, &s->d_in, nE)) ||
        (rc = dev_alloc(s, &s->d_out, nE)) || (rc = dev_alloc(s, &s->d_npast, (size_t) s->n_sessions)))
        return rc;
    if ((rc = dev_alloc(s, &s->xh, (size_t) s->n_ctx * (FF > E ? FF : E) + 64))) return rc;
    if (s->wtype != kWT_F16) {
        s->nbqE = s->layers[0].wo.nbq; s->nbqF = s->layers[0].w2.nbq;
        const size_t nq = (size_t) s->n_ctx;
        // Q4_1: every scale array carries a second plane (Q8_1's block sums s) right behind the scales
        const size_t pl = s->wtype == kWT_Q4_1 ? 2 : 1;
        if (pl == 2) { s->soffE = (int)(nq * s->nbqE * 4); s->soffF = (int)(nq * s->nbqF * 4); }
        if ((rc = dev_alloc(s, &s->aq_att, nq * s->nbqE * 32)) || (rc = dev_alloc(s, &s->da_att, pl * nq * s->nbqE * 4)) ||
            (rc = dev_alloc(s, &s->aq_gate, nq * s->nbqF * 32)) || (rc = dev_alloc(s, &s->da_gate, pl * nq * s->nbqF * 4))) return rc;
        if ((rc = dev_alloc(s, &s->aq_x, nq * s->nbqE * 32)) || (rc = dev_alloc(s, &s->da_x, pl * nq * s->nbqE * 4)) ||
            (rc = dev_alloc(s, &s->nq_counter, 2 * nq)) || (rc = dev_alloc(s, &s->nq_partial, nq * 256))) return rc;
        if ((rc = dev_alloc(s, &s->p_cnt, (size_t) s->L * kPPhases + 32))) return rc;
        B200_CUDA(cudaMemset(s->p_cnt, 0, ((size_t) s->L * kPPhases + 32) * 4));
        B200_CUDA(cudaMemset(s->aq_x, 0, nq * s->nbqE * 128)); B200_CUDA(cudaMemset(s->da_x, 0, pl * nq * s->nbqE * 16));
        B200_CUDA(cudaMemset(s->nq_counter, 0, 2 * nq * 4));
        B200_CUDA(cudaMemset(s->aq_att, 0, nq * s->nbqE * 128));  B200_CUDA(cudaMemset(s->da_att, 0, pl * nq * s->nbqE * 16));
        B200_CUDA(cudaMemset(s->aq_gate, 0, nq * s->nbqF * 128)); B200_CUDA(cudaMemset(s->da_gate, 0, pl * nq * s->nbqF * 16));
    }
    B200_CUDA(cudaMemset(s->kc, 0, s->n_sessions * s->sess_stride * 2));
    B200_CUDA(cudaMemset(s->vc, 0, s->n_sessions * s->sess_stride * 2));
    B200_CUDA(cudaMemset(s->d_npast, 0, 4 * (size_t) s->n_sessions));
    B200_CUDA(cudaMallocHost((void **) &s->h_in, (size_t) E * 4));
    B200_CUDA(cudaMallocHost((void **) &s->h_out, (size_t) E * 4));
    lap("KV cache + activations");
    if ((rc = build_tables(s))) return rc;
    lap("exp / SiLU / RoPE tables");
    if (env_int("B200_TRACE", 0)) {
        if ((rc = dev_alloc(s, &s->trace, (size_t) 512 * 1024 * 8))) return rc;
        B200_CUDA(cudaMemset(s->trace, 0, (size_t) 512 * 1024 * 8 * 8));
    }
    B200_CUDA(cudaFuncSetAttribute(k_attention, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit));
    B200_CUDA(cudaFuncSetAttribute(k_attn128<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    B200_CUDA(cudaFuncSetAttribute(k_attn128<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    B200_CUDA(cudaEventCreate(&s->ev0));
    B200_CUDA(cudaEventCreate(&s->ev1));
    B200_CUDA(cudaDeviceSynchronize());
    lap("attributes + final sync");
    if (ltrace) fprintf(stderr, "[b200 load] total %.3f s for %.2f GB of weights\n", tnow() - t_begin, s->weight_bytes / 1e9);
    return 0;
}

static void destroy(b200_slice * s) {
    cudaSetDevice(s->device);
    if (s->stream) cudaStreamSynchronize(s->stream);
    for (auto & kv : s->graphs) cudaGraphExecDestroy(kv.second);
    for (auto & kv : s->pp_graphs) cudaGraphExecDestroy(kv.second);
    if (s->mb_next) cudaIpcCloseMemHandle(s->mb_next);
    if (s->mb_prev && s->mb_prev != s->mb_next) cudaIpcCloseMemHandle(s->mb_prev);
    for (void * p : s->allocs) cudaFree(p);
    if (s->h_in) cudaFreeHost(s->h_in);
    if (s->h_out) cudaFreeHost(s->h_out);
    if (s->ev0) cudaEventDestroy(s->ev0);
    if (s->ev1) cudaEventDestroy(s->ev1);
    for (cudaEvent_t e : s->prof_ev) cudaEventDestroy(e);
    for (int i = 0; i < 2; i++) if (s->mark[i]) cudaEventDestroy(s->mark[i]);
    if (s->stream) cudaStreamDestroy(s->stream);
    delete s;
}

}  // namespace b200

// ============================================================================ C ABI
extern "C" {

const char * b200_last_error(void) { return b200::last_error_ref().c_str(); }
const char * b200_version(void) { return "b200-slice 0.1 (sm_100a, exact mode)"; }

int b200_slice_load(const char * path, int device, int n_ctx, b200_slice_t ** out) {
    return b200_slice_load_ex(path, device, n_ctx, 1, out);
}

int b200_slice_load_ex(const char * path, int device, int n_ctx, int n_sessions, b200_slice_t ** out) {
    if (!path || !out) return fail(B200_EINVAL, "b200_slice_load: null argument");
    *out = nullptr;
    if (n_sessions < 1 || n_sessions > 4096) return fail(B200_EINVAL, "n_sessions %d outside [1, 4096]", n_sessions);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(B200_ENODEV, "no CUDA device visible: the slice forward has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(B200_ENODEV, "device %d out of range (%d visible)", device, ndev);
    cudaDeviceProp prop;
    B200_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail(B200_ENODEV, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
    B200_CUDA(cudaSetDevice(device));
    b200_slice * s = new b200_slice();
    s->device = device; s->n_sm = prop.multiProcessorCount;
    s->n_ctx = n_ctx > 0 ? n_ctx : 512;               // vendor examples/common.h:28
    s->n_sessions = n_sessions;
    s->use_ring  = env_int("B200_RING", 1) != 0;
    s->use_graph = env_int("B200_GRAPH", 1) != 0;
    s->use_pdl   = env_int("B200_PDL", 1) != 0;
    s->fast_prefill = env_int("B200_FAST_PREFILL", 0) != 0; s->fast_min_tokens = env_int("B200_FAST_MIN_TOKENS", 32);
    s->fast_version = env_int("B200_FAST_V", 2);
    s->use_nq    = env_int("B200_NQ", 0) != 0;   // grid-barrier norm+quant epilogue in wo / w2 (decode): exact, opt-in (its barrier costs what it saves)
    s->opt_ns = env_int("B200_NS", 0); s->opt_cta_per_sm = env_int("B200_CTA_PER_SM", 0); s->opt_nc = env_int("B200_NC", 0);
    s->opt_pre = env_int("B200_PRE", 3); s->opt_nomath = env_int("B200_DBG_NOMATH", 0);
    s->use_tiled_attn = env_int("B200_TILED_ATTN", 1) != 0;
    s->f16_mc = env_int("B200_F16_MC", 1) != 0;      // F16 slices, multi-token calls: 4 (8) columns per CTA share the weight loads
    s->f16_mc_cols = env_int("B200_F16_MC", 1) == 8 ? 8 : 4;
    s->use_n8 = env_int("B200_N8", 0) != 0;          // single-token wo / w2: 8 threads per row (k_gemv_n8): exact, opt-in (slower: 806 vs 823 tok/s)  // prompt chunks: query-tiled attention (K / V staged once per 16 queries)
    s->f16_ring = env_int("B200_F16_RING", 1) != 0;          // F16-weight slices: TMA-ring matmul for single-token steps
    s->use_persist = env_int("B200_PERSIST", 0) != 0;         // single-token step as ONE persistent kernel (persist.cuh)
    s->persist_tr = env_int("B200_PERSIST_TR", 4); s->persist_ns = env_int("B200_PERSIST_NS", 0); s->persist_ctas = env_int("B200_PERSIST_CTAS", 0);
    if (s->persist_tr != 1 && s->persist_tr != 2 && s->persist_tr != 4) s->persist_tr = 4;
    const bool want_ptrace = env_int("B200_PTRACE", 0) != 0;
    cudaError_t e = cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) { delete s; return fail(B200_ECUDA, "cudaStreamCreate failed: %s", cudaGetErrorString(e)); }
    int rc = load_locked(s, path);
    if (rc) { destroy(s); return rc; }
    if (want_ptrace) {
        const size_t n = (size_t) s->n_sm * s->L * kPTraceSlots;
        if ((rc = dev_alloc(s, &s->p_trace, n))) { destroy(s); return rc; }
        cudaMemset(s->p_trace, 0, n * 8);
    }
    *out = s;
    return 0;
}

/* Debug timeline of the persistent step (B200_PTRACE=1 at load): [cta][layer][16] %globaltimer stamps of the LAST step. */
int b200_debug_ptrace_read(b200_slice_t * s, unsigned long long * out, size_t cap_words) {
    if (!s || !s->p_trace || !out) return 0;
    cudaSetDevice(s->device);
    cudaStreamSynchronize(s->stream);
    size_t n = (size_t) s->n_sm * s->L * kPTraceSlots;
    if (n > cap_words) n = cap_words;
    cudaMemcpy(out, s->p_trace, n * 8, cudaMemcpyDeviceToHost);
    return (int)(n / kPTraceSlots);
}

int b200_slice_unload(b200_slice_t * s) {
    if (!s) return fail(B200_EINVAL, "null handle");
    { std::lock_guard<std::mutex> lk(s->mu); }       // let a call that is inside the library finish (see the header: no NEW call may race unload)
    destroy(s);
    return 0;
}

/* Create the CUDA context of `device` (cudaSetDevice + a no-op runtime call).  The first CUDA call of a process costs
 * 0.3 s on a 1-GPU box and several seconds on an 8-GPU box; callers that time b200_slice_load can pay it up front. */
int b200_device_init(int device) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(B200_ENODEV, "no CUDA device visible: the slice forward has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(B200_ENODEV, "device %d out of range (%d visible)", device, ndev);
    B200_CUDA(cudaSetDevice(device));
    B200_CUDA(cudaFree(nullptr));
    return 0;
}

int b200_slice_clear(b200_slice_t * s) {
    if (!s) return fail(B200_EINVAL, "null handle");
    std::lock_guard<std::mutex> lk(s->mu);
    B200_CUDA(cudaSetDevice(s->device));
    B200_CUDA(cudaMemsetAsync(s->d_npast, 0, 4, s->stream));
    B200_CUDA(cudaStreamSynchronize(s->stream));
    s->past[0] = 0;
    return 0;
}

int b200_slice_rewind(b200_slice_t * s, int n_past) {
    if (!s) return fail(B200_EINVAL, "null handle");
    std::lock_guard<std::mutex> lk(s->mu);
    if (n_past < 0 || n_past > s->past[0]) return fail(B200_EINVAL, "rewind target %d outside [0, %d]", n_past, s->past[0]);
    B200_CUDA(cudaSetDevice(s->device));
    B200_CUDA(cudaMemcpyAsync(s->d_npast, &n_past, 4, cudaMemcpyHostToDevice, s->stream));
    B200_CUDA(cudaStreamSynchronize(s->stream));
    s->past[0] = n_past;
    return 0;
}

int b200_slice_info(b200_slice_t * s, b200_slice_info_t * info) {
    if (!s || !info) return fail(B200_EINVAL, "null argument");
    info->n_embd = s->E; info->n_head = s->H; info->n_ff = s->FF; info->n_layer = s->L; info->first_layer = s->first_layer;
    info->n_ctx = s->n_ctx; info->n_past = s->past[0]; info->weight_type = s->wtype; info->device = s->device;
    info->weight_bytes = s->weight_bytes; info->kv_bytes_per_pos = (int64_t) s->L * 2 * s->E * 2;
    return 0;
}

int b200_slice_forward(b200_slice_t * s, const float * in, int n_tokens, float * out) {
    if (!s || !in || !out) return fail(B200_EINVAL, "null argument");
    std::lock_guard<std::mutex> lk(s->mu);
    return forward_locked(s, in, n_tokens, out, true);
}

int b200_slice_forward_device(b200_slice_t * s, const float * d_in, int n_tokens, float * d_out, int sync) {
    if (!s || !d_in || !d_out) return fail(B200_EINVAL, "null argument");
    std::lock_guard<std::mutex> lk(s->mu);
    int rc = forward_locked(s, d_in, n_tokens, d_out, false);
    if (rc) return rc;
    if (sync) B200_CUDA(cudaStreamSynchronize(s->stream));
    return 0;
}

/* ---- sessions and batched steps (additive; SURVEY 8f N3) ---- */
int b200_session_count(b200_slice_t * s) { return s ? s->n_sessions : 0; }

int b200_session_n_past(b200_slice_t * s, int session) {
    if (!s || session < 0 || session >= s->n_sessions) return -1;
    std::lock_guard<std::mutex> lk(s->mu);
    return s->past[session];
}

int b200_session_clear(b200_slice_t * s, int session) {
    if (!s) return fail(B200_EINVAL, "null handle");
    if (session < -1 || session >= s->n_sessions) return fail(B200_EINVAL, "session %d outside [0, %d)", session, s->n_sessions);
    std::lock_guard<std::mutex> lk(s->mu);
    B200_CUDA(cudaSetDevice(s->device));
    if (session < 0) {
        B200_CUDA(cudaMemsetAsync(s->d_npast, 0, 4 * (size_t) s->n_sessions, s->stream));
        std::fill(s->past.begin(), s->past.end(), 0);
    } else {
        B200_CUDA(cudaMemsetAsync(s->d_npast + session, 0, 4, s->stream));
        s->past[session] = 0;
    }
    B200_CUDA(cudaStreamSynchronize(s->stream));
    return 0;
}

int b200_session_rewind(b200_slice_t * s, int session, int n_past) {
    if (!s) return fail(B200_EINVAL, "null handle");
    if (session < 0 || session >= s->n_sessions) return fail(B200_EINVAL, "session %d outside [0, %d)", session, s->n_sessions);
    std::lock_guard<std::mutex> lk(s->mu);
    if (n_past < 0 || n_past > s->past[session]) return fail(B200_EINVAL, "rewind target %d outside [0, %d]", n_past, s->past[session]);
    B200_CUDA(cudaSetDevice(s->device));
    B200_CUDA(cudaMemcpyAsync(s->d_npast + session, &n_past, 4, cudaMemcpyHostToDevice, s->stream));
    B200_CUDA(cudaStreamSynchronize(s->stream));
    s->past[session] = n_past;
    return 0;
}

int b200_session_forward(b200_slice_t * s, int session, const float * in, int n_tokens, float * out) {
    if (!s || !in || !out) return fail(B200_EINVAL, "null argument");
    std::lock_guard<std::mutex> lk(s->mu);
    return forward_locked(s, in, n_tokens, out, true, session);
}

int b200_session_forward_device(b200_slice_t * s, int session, const float * d_in, int n_tokens, float * d_out, int sync) {
    if (!s || !d_in || !d_out) return fail(B200_EINVAL, "null argument");
    std::lock_guard<std::mutex> lk(s->mu);
    int rc = forward_locked(s, d_in, n_tokens, d_out, false, session);
    if (rc) return rc;
    if (sync) B200_CUDA(cudaStreamSynchronize(s->stream));
    return 0;
}

int b200_batch_forward(b200_slice_t * s, const int * sessions, int n_seq, const float * in, float * out) {
    if (!s || !sessions || !in || !out) return fail(B200_EINVAL, "null argument");
    std::lock_guard<std::mutex> lk(s->mu);
    return mixed_locked(s, sessions, nullptr, n_seq, in, out, true);
}

int b200_batch_forward_device(b200_slice_t * s, const int * sessions, int n_seq, const float * d_in, float * d_out, int sync) {
    if (!s || !sessions || !d_in || !d_out) return fail(B200_EINVAL, "null argument");
    std::lock_guard<std::mutex> lk(s->mu);
    int rc = mixed_locked(s, sessions, nullptr, n_seq, d_in, d_out, false);
    if (rc) return rc;
    if (sync) B200_CUDA(cudaStreamSynchronize(s->stream));
    return 0;
}

// The mixed-step entry points are new: a caller without a device cannot have a handle, so a null handle reports why.
static int null_handle() {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(B200_ENODEV, "no CUDA device visible: the slice forward has no CPU fallback");
    return fail(B200_EINVAL, "null handle");
}

int b200_mixed_forward(b200_slice_t * s, const int * sessions, const int * n_tokens, int n_seg, const float * in, float * out) {
    if (!s) return null_handle();
    if (!sessions || !n_tokens || !in || !out) return fail(B200_EINVAL, "null argument");
    std::lock_guard<std::mutex> lk(s->mu);
    return mixed_locked(s, sessions, n_tokens, n_seg, in, out, true);
}

int b200_mixed_forward_device(b200_slice_t * s, const int * sessions, const int * n_tokens, int n_seg, const float * d_in, float * d_out,
                              int sync) {
    if (!s) return null_handle();
    if (!sessions || !n_tokens || !d_in || !d_out) return fail(B200_EINVAL, "null argument");
    std::lock_guard<std::mutex> lk(s->mu);
    int rc = mixed_locked(s, sessions, n_tokens, n_seg, d_in, d_out, false);
    if (rc) return rc;
    if (sync) B200_CUDA(cudaStreamSynchronize(s->stream));
    return 0;
}

int b200_slice_sync(b200_slice_t * s) {
    if (!s) return fail(B200_EINVAL, "null handle");
    B200_CUDA(cudaSetDevice(s->device));
    B200_CUDA(cudaStreamSynchronize(s->stream));
    return 0;
}

float b200_slice_last_ms(b200_slice_t * s) {
    if (!s || !s->timed) return -1.f;
    float ms = -1.f;
    cudaSetDevice(s->device);
    if (cudaEventSynchronize(s->ev1) != cudaSuccess) return -1.f;
    if (cudaEventElapsedTime(&ms, s->ev0, s->ev1) != cudaSuccess) return -1.f;
    return ms;
}

int64_t b200_slice_launch_count(b200_slice_t * s) { return s ? s->launches : 0; }
float * b200_slice_dev_in(b200_slice_t * s)  { return s ? s->d_in : nullptr; }
float * b200_slice_dev_out(b200_slice_t * s) { return s ? s->d_out : nullptr; }

int b200_slice_set_fast_prefill(b200_slice_t * s, int on, int min_tokens) {
    if (!s) return fail(B200_EINVAL, "null handle");
    std::lock_guard<std::mutex> lk(s->mu);
    s->fast_prefill = on != 0;
    if (min_tokens > 0) s->fast_min_tokens = min_tokens;
    return 0;
}

/* Measurement aid for bench.py's roofline: while on, a decode step launches ONLY its weight-matmul kernels (the
 * attention launch is skipped, so hidden states are meaningless and the KV cache is not appended). */
int b200_debug_skip_attention(b200_slice_t * s, int on) {
    if (!s) return fail(B200_EINVAL, "null handle");
    std::lock_guard<std::mutex> lk(s->mu);
    s->skip_attention = on != 0;
    return 0;
}

int b200_slice_mark(b200_slice_t * s, int which) {
    if (!s || which < 0 || which > 1) return fail(B200_EINVAL, "bad argument");
    B200_CUDA(cudaSetDevice(s->device));
    if (!s->mark[which]) B200_CUDA(cudaEventCreate(&s->mark[which]));
    B200_CUDA(cudaEventRecord(s->mark[which], s->stream));
    return 0;
}

float b200_slice_mark_elapsed_ms(b200_slice_t * s) {
    if (!s || !s->mark[0] || !s->mark[1]) return -1.f;
    float ms = -1.f;
    cudaSetDevice(s->device);
    if (cudaEventSynchronize(s->mark[1]) != cudaSuccess) return -1.f;
    if (cudaEventElapsedTime(&ms, s->mark[0], s->mark[1]) != cudaSuccess) return -1.f;
    return ms;
}

int b200_slice_profile(b200_slice_t * s, int enable) {
    if (!s) return fail(B200_EINVAL, "null handle");
    std::lock_guard<std::mutex> lk(s->mu);
    s->profiling = enable != 0; s->prof_used = 0; s->prof_cls.clear();
    return 0;
}

int b200_slice_profile_read(b200_slice_t * s, float * ms_by_class, int * launches_by_class, int n_class) {
    if (!s || !ms_by_class || !launches_by_class) return fail(B200_EINVAL, "null argument");
    std::lock_guard<std::mutex> lk(s->mu);
    B200_CUDA(cudaSetDevice(s->device));
    B200_CUDA(cudaStreamSynchronize(s->stream));
    for (int i = 0; i < n_class; i++) { ms_by_class[i] = 0.f; launches_by_class[i] = 0; }
    for (size_t i = 0; i < s->prof_cls.size(); i++) {
        float ms = 0.f;
        B200_CUDA(cudaEventElapsedTime(&ms, s->prof_ev[2 * i], s->prof_ev[2 * i + 1]));
        const int c = s->prof_cls[i];
        if (c < n_class) { ms_by_class[c] += ms; launches_by_class[c]++; }
    }
    s->prof_used = 0; s->prof_cls.clear();
    return 0;
}

/* Switch the in-kernel timeline on or off at run time (drops the captured decode graphs so the next step re-captures). */
int b200_debug_trace_enable(b200_slice_t * s, int on) {
    if (!s) return fail(B200_EINVAL, "null handle");
    std::lock_guard<std::mutex> lk(s->mu);
    B200_CUDA(cudaSetDevice(s->device));
    B200_CUDA(cudaStreamSynchronize(s->stream));
    for (auto & kv : s->graphs) cudaGraphExecDestroy(kv.second);
    s->graphs.clear();
    static unsigned long long * parked = nullptr;
    if (on) {
        if (!s->trace) {
            if (parked) { s->trace = parked; parked = nullptr; }
            else { int rc = dev_alloc(s, &s->trace, (size_t) 512 * 1024 * 8); if (rc) return rc; }
        }
        B200_CUDA(cudaMemset(s->trace, 0, (size_t) 512 * 1024 * 8 * 8));
        s->trace_next = 0; s->trace_cls.clear(); s->trace_ctas.clear();
    } else if (s->trace) { parked = s->trace; s->trace = nullptr; }
    return 0;
}

/* Debug timeline: when B200_TRACE=1 every matmul / attention launch of the NEXT captured graph (or un-graphed step)
 * stamps %globaltimer per CTA: [0] entry, [1] after griddepcontrol.wait, [2] prologue done, [3] exit, [4] last weight copy issued. */
int b200_debug_trace_read(b200_slice_t * s, unsigned long long * out, int * cls, int * ctas, int max_launches) {
    if (!s || !s->trace) return 0;
    cudaSetDevice(s->device);
    cudaStreamSynchronize(s->stream);
    int n = s->trace_next < max_launches ? s->trace_next : max_launches;
    cudaMemcpy(out, s->trace, (size_t) n * 1024 * 8 * 8, cudaMemcpyDeviceToHost);
    for (int i = 0; i < n; i++) { cls[i] = s->trace_cls[i]; ctas[i] = s->trace_ctas[i]; }
    return n;
}

/* Test hook: copy `count` 32-bit words of an internal activation buffer to the host after a
 * forward (0 qkv, 1 att, 2 ffin, 3 gate, 4 xa, 5 xb, 6 q16, 7 k-cache, 8 v-cache). */
int b200_debug_read(b200_slice_t * s, int which, size_t offset_words, size_t count, void * out) {
    if (!s || !out) return fail(B200_EINVAL, "null argument");
    const void * src[9] = {s->qkv, s->att, s->ffin, s->gate, s->xa, s->xb, s->q16, s->kc, s->vc};
    if (which < 0 || which > 8) return fail(B200_EINVAL, "bad buffer id %d", which);
    B200_CUDA(cudaSetDevice(s->device));
    B200_CUDA(cudaStreamSynchronize(s->stream));
    B200_CUDA(cudaMemcpy(out, (const uint32_t *) src[which] + offset_words, count * 4, cudaMemcpyDeviceToHost));
    return 0;
}

/* Test hook: ONE fast-mode weight matmul of `layer` with the launch sequence enqueue_layers uses (k_prep_q8_f16, then the
 * tcgen05 kernel), on private buffers: the KV cache and n_past are not touched.  which: 0 qkv, 1 wo, 2 w1|w3, 3 w2. */
int b200_debug_fast_matmul(b200_slice_t * s, int layer, int which, int tile, const float * x, int n_tokens, const float * resid,
                           float * y, uint16_t * xh) {
    if (!s || !x || !y || !xh) return fail(B200_EINVAL, "null argument");
    std::lock_guard<std::mutex> lk(s->mu);
    if (layer < 0 || layer >= s->L) return fail(B200_EINVAL, "layer %d outside [0, %d)", layer, s->L);
    if (which < 0 || which > 3) return fail(B200_EINVAL, "bad matrix id %d", which);
    if (n_tokens <= 0 || n_tokens > s->n_ctx) return fail(B200_EINVAL, "n_tokens %d outside [1, n_ctx %d]", n_tokens, s->n_ctx);
    if (tile != 0 && tile != 128 && !(tile == 256 && s->fast_version >= 2))
        return fail(B200_EINVAL, "token tile %d not available (fast kernel v%d)", tile, s->fast_version);
    LayerW & Lw = s->layers[layer];
    if (!fast_weights_ok(s, Lw)) return fail(B200_EINVAL, "this slice does not qualify for fast mode");
    const bool has_resid = which == 1 || which == 3;
    if (has_resid && !resid) return fail(B200_EINVAL, "wo / w2 need the residual input");
    const int E = s->E, FF = s->FF, N = n_tokens;
    const int K = which == 3 ? FF : E, rows = which == 0 ? 3 * E : (which == 2 ? FF : E);
    const size_t n_pad = (size_t)(N + 255) & ~(size_t) 255;
    B200_CUDA(cudaSetDevice(s->device));
    float * d_x = nullptr, * d_r = nullptr, * d_y = nullptr;
    auto run = [&]() -> int {
        B200_CUDA(cudaMalloc(&d_x, (size_t) N * K * 4));
        B200_CUDA(cudaMalloc(&d_y, n_pad * rows * 4));
        if (has_resid) B200_CUDA(cudaMalloc(&d_r, (size_t) N * E * 4));
        B200_CUDA(cudaMemcpyAsync(d_x, x, (size_t) N * K * 4, cudaMemcpyHostToDevice, s->stream));
        if (has_resid) B200_CUDA(cudaMemcpyAsync(d_r, resid, (size_t) N * E * 4, cudaMemcpyHostToDevice, s->stream));
        B200_CUDA(cudaMemsetAsync(d_y, 0xFF, n_pad * rows * 4, s->stream));      // sentinel: every word 0xFFFFFFFF (a NaN)
        int rc;
        switch (which) {
        case 0:
            if ((rc = launch_prep<true>(s, d_x, E, Lw.attn_norm, E, N))) return rc;
            if ((rc = launch_fast_any<FG_STORE>(s, Lw.qkv, nullptr, 0, d_y, 3 * E, N, 3 * E, tile))) return rc;
            break;
        case 1:
            if ((rc = launch_prep<false>(s, d_x, E, nullptr, E, N))) return rc;
            if ((rc = launch_fast_any<FG_RESID>(s, Lw.wo, d_r, E, d_y, E, N, E, tile))) return rc;
            break;
        case 2:
            if ((rc = launch_prep<true>(s, d_x, E, Lw.ffn_norm, E, N))) return rc;
            if ((rc = launch_fast_any<FG_GATE>(s, Lw.w13, nullptr, 0, d_y, FF, N, FF, tile))) return rc;
            break;
        default:
            if ((rc = launch_prep<false>(s, d_x, FF, nullptr, FF, N))) return rc;
            if ((rc = launch_fast_any<FG_RESID>(s, Lw.w2, d_r, E, d_y, E, N, E, tile))) return rc;
        }
        B200_CUDA(cudaMemcpyAsync(y, d_y, n_pad * rows * 4, cudaMemcpyDeviceToHost, s->stream));
        B200_CUDA(cudaMemcpyAsync(xh, s->xh, (size_t) N * K * 2, cudaMemcpyDeviceToHost, s->stream));
        B200_CUDA(cudaStreamSynchronize(s->stream));
        return 0;
    };
    const int rc = run();
    if (rc) cudaStreamSynchronize(s->stream);
    cudaFree(d_x); cudaFree(d_y); cudaFree(d_r);
    return rc;
}

}  // extern "C"


// ============================================================================ layer-slice pipeline (NCCL)
// The reference relays the activation between nodes through the client over TCP, one request per hop
// (cli_api/common.py:148-154 -> control_center.py:224-244 -> routes.py:176-195).  For slices that live on the
// GPUs of one NVSwitch box the hop is ONE ncclSend / ncclRecv of [n_tokens][n_embd] f32 on the slice's stream.
// NCCL is bound at run time (dlopen) so that the single-GPU path carries no dependency on it.
namespace b200 {
struct NcclId { char bytes[128]; };
struct NcclApi {
    void * lib = nullptr;
    int (*GetUniqueId)(NcclId *) = nullptr;
    int (*CommInitRank)(void **, int, NcclId, int) = nullptr;
    int (*Send)(const void *, size_t, int, int, void *, cudaStream_t) = nullptr;
    int (*Recv)(void *, size_t, int, int, void *, cudaStream_t) = nullptr;
    int (*CommDestroy)(void *) = nullptr;
    const char * (*GetErrorString)(int) = nullptr;
};
static NcclApi & nccl() {
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        const char * env = getenv("B200_NCCL_LIB");
        const char * names[] = {env, "libnccl.so.2", "libnccl.so"};
        for (const char * n : names) {
            if (!n) continue;
            api.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
            if (api.lib) break;
        }
        if (!api.lib) return;
        api.GetUniqueId    = (int (*)(NcclId *)) dlsym(api.lib, "ncclGetUniqueId");
        api.CommInitRank   = (int (*)(void **, int, NcclId, int)) dlsym(api.lib, "ncclCommInitRank");
        api.Send           = (int (*)(const void *, size_t, int, int, void *, cudaStream_t)) dlsym(api.lib, "ncclSend");
        api.Recv           = (int (*)(void *, size_t, int, int, void *, cudaStream_t)) dlsym(api.lib, "ncclRecv");
        api.CommDestroy    = (int (*)(void *)) dlsym(api.lib, "ncclCommDestroy");
        api.GetErrorString = (const char * (*)(int)) dlsym(api.lib, "ncclGetErrorString");
    });
    return api;
}
static int nccl_fail(const char * what, int rc) {
    NcclApi & n = nccl();
    return fail(B200_ENCCL, "%s failed: %s", what, n.GetErrorString ? n.GetErrorString(rc) : "NCCL error");
}
constexpr int kNcclFloat32 = 7;
}  // namespace b200

extern "C" {

int b200_pipeline_unique_id(void * id128) {
    NcclApi & n = nccl();
    if (!n.lib || !n.GetUniqueId) return fail(B200_ENCCL, "libnccl.so.2 not found (set B200_NCCL_LIB)");
    if (!id128) return fail(B200_EINVAL, "null id buffer");
    NcclId id;
    int rc = n.GetUniqueId(&id);
    if (rc) return nccl_fail("ncclGetUniqueId", rc);
    memcpy(id128, id.bytes, 128);
    return 0;
}

int b200_pipeline_init(b200_slice_t * s, int rank, int nranks, const void * id128) {
    if (!s || !id128 || rank < 0 || rank >= nranks) return fail(B200_EINVAL, "bad pipeline arguments");
    NcclApi & n = nccl();
    if (!n.lib || !n.CommInitRank) return fail(B200_ENCCL, "libnccl.so.2 not found (set B200_NCCL_LIB)");
    std::lock_guard<std::mutex> lk(s->mu);
    B200_CUDA(cudaSetDevice(s->device));
    NcclId id; memcpy(id.bytes, id128, 128);
    int rc = n.CommInitRank(&s->nccl_comm, nranks, id, rank);
    if (rc) return nccl_fail("ncclCommInitRank", rc);
    s->pp_rank = rank; s->pp_world = nranks;
    if (rank == 0 && !s->d_final) { int e = dev_alloc(s, &s->d_final, (size_t) s->n_ctx * s->E); if (e) return e; }
    return 0;
}

// Peer-memory variant of a pipeline step (see kernels.cuh, "Inter-slice hand-off through PEER MEMORY"): the hop is a
// store into the next rank's mailbox + a flag, issued by k_peer_send right behind this slice's last matmul and picked
// up by k_peer_recv in front of the next slice's first matmul.  For a single-token step the whole sequence
// [recv ->] layers -> send [-> recv of the ring result] is ONE captured graph per rank: no host code between slices.
static int pipeline_step_peer(b200_slice * s, const float * d_in, int n_rows, int ring, int session, bool multi) {
    const int r = s->pp_rank, W = s->pp_world;
    const size_t count = (size_t) n_rows * s->E;
    if (count > s->mb_slot_floats) return fail(B200_EINVAL, "hand-off of %zu floats exceeds the mailbox slot (%zu)", count, s->mb_slot_floats);
    const bool recv_in = r > 0, sends = r < W - 1 || ring, recv_final = r == 0 && ring == 1;   // ring 2: rank 0 collects later
    MailboxHdr * mine = (MailboxHdr *) s->mb_block;
    const uint2 * inbox = (const uint2 *)(s->mb_block + sizeof(MailboxHdr));
    PeerRecvArgs ra{mine, inbox, s->mb_slot_floats, &((MailboxHdr *) s->mb_prev)->ack, s->d_in, (int) count};
    PeerRecvArgs rf = ra; rf.dst = s->d_final;
    PeerSendArgs sa{mine, (uint2 *)(s->mb_next + sizeof(MailboxHdr)), s->mb_slot_floats, s->d_out, (int) count};
    const int xfer_ctas = (int) std::min<size_t>(32, (count + 8191) / 8192);      // one CTA per 8 K elements, at most 32
    if (!multi) { s->cur = session; s->cols = nullptr; }
    // fold the send into the slice's last matmul for plain single-token steps of quantised, head-size-128 slices
    const bool fold = s->use_fold && sends && !multi && n_rows == 1 && s->D == 128 && s->wtype != kWT_F16 && s->use_ring && !s->use_nq &&
                      !persist_applicable(s, 1) && !s->skip_attention;
    const float * in = recv_in ? s->d_in : d_in;
    int rc = 0;
    if (!multi && persist_applicable(s, n_rows) && (rc = persist_prepare(s, in, s->d_out))) return rc;
    auto body = [&]() -> int {
        int e;
        s->cur_class = 6;
        if (recv_in && (e = launch_simple(s, k_peer_recv, dim3(xfer_ctas, 1, 1), dim3(1024, 1, 1), 0, ra))) return e;
        if (sends && !fold) { s->send_args = sa; s->send_pending = true; s->send_ctas = xfer_ctas; }
        s->fold_send = fold;
        e = enqueue_layers(s, in, n_rows, s->d_out);
        s->send_pending = false; s->fold_send = false;
        if (e) return e;
        s->cur_class = 6;
        if (recv_final && (e = launch_simple(s, k_peer_recv, dim3(xfer_ctas, 1, 1), dim3(1024, 1, 1), 0, rf))) return e;
        return 0;
    };
    B200_CUDA(cudaEventRecord(s->ev0, s->stream));
    if (multi) {
        if ((rc = upload_plan(s))) { s->cols = nullptr; return rc; }
        rc = body();
        s->cols = nullptr;
        if (rc) return rc;
        commit_plan(s);
    } else if (n_rows == 1 && s->use_graph && !s->profiling) {
        GraphKey key{in, nullptr, (ring & 3) | (fold ? 4 : 0) | (session << 3)};
        auto it = s->pp_graphs.find(key);
        if (it == s->pp_graphs.end()) {
            const int64_t before = s->launches;
            cudaGraph_t g = nullptr;
            B200_CUDA(cudaStreamBeginCapture(s->stream, cudaStreamCaptureModeThreadLocal));
            rc = body();
            cudaError_t e = cudaStreamEndCapture(s->stream, &g);
            s->launches = before;
            if (rc) { if (g) cudaGraphDestroy(g); return rc; }
            if (e != cudaSuccess) return fail(B200_ECUDA, "pipeline graph capture failed: %s", cudaGetErrorString(e));
            cudaGraphExec_t ge = nullptr;
            e = cudaGraphInstantiate(&ge, g, 0);
            cudaGraphDestroy(g);
            if (e != cudaSuccess) return fail(B200_ECUDA, "cudaGraphInstantiate failed: %s", cudaGetErrorString(e));
            if (s->pp_graphs.size() >= 64) { for (auto & kv : s->pp_graphs) cudaGraphExecDestroy(kv.second); s->pp_graphs.clear(); }
            it = s->pp_graphs.emplace(key, ge).first;
        }
        B200_CUDA(cudaGraphLaunch(it->second, s->stream));
        s->launches += (persist_applicable(s, 1) ? 2 : (s->D == 128 ? 5 : 6) * s->L + 1) + (recv_in ? 1 : 0) + (sends ? 1 : 0) + (recv_final ? 1 : 0);
        s->past[session] += 1;
    } else {
        s->cur = session; s->cols = nullptr;
        if ((rc = body())) return rc;
        s->past[session] += n_rows;
    }
    B200_CUDA(cudaEventRecord(s->ev1, s->stream));
    s->timed = true;
    return 0;
}

// recv <- rank-1, the slice's layers, send -> rank+1 (ring: the last rank hands its output back to rank 0).
// sessions == nullptr: n_rows tokens of session `session`; else a step over the n_rows listed sessions, n_tokens[i] tokens of
// sessions[i] (n_tokens == nullptr: one each), as b200_mixed_forward.
static int pipeline_step_locked(b200_slice * s, const float * d_in, int n_rows, int ring, int session, const int * sessions,
                                const int * n_tokens = nullptr) {
    NcclApi & n = nccl();
    B200_CUDA(cudaSetDevice(s->device));
    int rc;
    // validate the step BEFORE anything is posted: a rejected step must not leave the peer's send unmatched
    if (sessions) {
        if ((rc = plan_step(s, sessions, n_tokens, n_rows, &n_rows))) return rc;
    } else {
        if (n_rows <= 0 || n_rows > s->n_ctx) return fail(B200_EINVAL, "n_tokens %d outside [1, n_ctx]", n_rows);
        if (session < 0 || session >= s->n_sessions) return fail(B200_EINVAL, "session %d outside [0, %d)", session, s->n_sessions);
        if (s->past[session] + n_rows > s->n_ctx)
            return fail(B200_ECONTEXT, "context overflow: n_past %d + n_tokens %d > n_ctx %d", s->past[session], n_rows, s->n_ctx);
    }
    const size_t count = (size_t) n_rows * s->E;
    const int r = s->pp_rank, W = s->pp_world;
    if (r == 0 && !d_in) return fail(B200_EINVAL, "rank 0 needs an input buffer");
    if (s->mb_on && W > 1) return pipeline_step_peer(s, d_in, n_rows, ring, session, sessions != nullptr);
    const float * in = d_in;
    if (r > 0) {
        if ((rc = n.Recv(s->d_in, count, kNcclFloat32, r - 1, s->nccl_comm, s->stream))) return nccl_fail("ncclRecv", rc);
        in = s->d_in;
    }
    if (sessions) rc = run_plan(s, n_rows, in, s->d_out, false);
    else          rc = forward_locked(s, in, n_rows, s->d_out, false, session);
    if (rc) return rc;
    if (r < W - 1) {
        if ((rc = n.Send(s->d_out, count, kNcclFloat32, r + 1, s->nccl_comm, s->stream))) return nccl_fail("ncclSend", rc);
    } else if (ring && W > 1) {
        if ((rc = n.Send(s->d_out, count, kNcclFloat32, 0, s->nccl_comm, s->stream))) return nccl_fail("ncclSend", rc);
    }
    if (r == 0 && ring == 1 && W > 1) {
        // the last slice's output comes back to the first rank (where the client-side lm_head lives)
        if ((rc = n.Recv(s->d_final, count, kNcclFloat32, W - 1, s->nccl_comm, s->stream))) return nccl_fail("ncclRecv", rc);
    }
    s->launches += (r > 0) + (r < W - 1 || (ring && W > 1)) + (r == 0 && ring == 1 && W > 1);
    return 0;
}

int b200_pipeline_step(b200_slice_t * s, const float * d_in, int n_tokens, int ring) {
    if (!s || !s->nccl_comm) return fail(B200_EINVAL, "pipeline not initialised");
    std::lock_guard<std::mutex> lk(s->mu);
    return pipeline_step_locked(s, d_in, n_tokens, ring, 0, nullptr);
}

int b200_pipeline_step_session(b200_slice_t * s, int session, const float * d_in, int n_tokens, int ring) {
    if (!s || !s->nccl_comm) return fail(B200_EINVAL, "pipeline not initialised");
    std::lock_guard<std::mutex> lk(s->mu);
    return pipeline_step_locked(s, d_in, n_tokens, ring, session, nullptr);
}

int b200_pipeline_step_batch(b200_slice_t * s, const int * sessions, int n_seq, const float * d_in, int ring) {
    if (!s || !s->nccl_comm) return fail(B200_EINVAL, "pipeline not initialised");
    if (!sessions) return fail(B200_EINVAL, "null session list");
    std::lock_guard<std::mutex> lk(s->mu);
    return pipeline_step_locked(s, d_in, n_seq, ring, 0, sessions);
}

int b200_pipeline_step_mixed(b200_slice_t * s, const int * sessions, const int * n_tokens, int n_seg, const float * d_in, int ring) {
    if (!s) return null_handle();
    if (!s->nccl_comm) return fail(B200_EINVAL, "pipeline not initialised");
    if (!sessions || !n_tokens) return fail(B200_EINVAL, "null session list");
    std::lock_guard<std::mutex> lk(s->mu);
    return pipeline_step_locked(s, d_in, n_seg, ring, 0, sessions, n_tokens);
}

/* ---- peer-memory hand-off: mailboxes mapped across processes with cudaIpc --------------------------------------- */
int b200_pipeline_mailbox_export(b200_slice_t * s, void * handle64) {
    if (!s || !handle64) return fail(B200_EINVAL, "null argument");
    std::lock_guard<std::mutex> lk(s->mu);
    B200_CUDA(cudaSetDevice(s->device));
    s->mb_slot_floats = (size_t) s->n_ctx * s->E;
    const size_t bytes = sizeof(MailboxHdr) + (size_t) kMbSlots * s->mb_slot_floats * 8;      // 8-byte {value, seq} elements
    if (!s->mb_block) {
        void * p = nullptr;
        B200_CUDA(cudaMalloc(&p, bytes));                 // a dedicated cudaMalloc block: IPC handles cover whole allocations
        s->allocs.push_back(p);
        s->mb_block = (uint8_t *) p;
    }
    // a fresh link: counters at zero, and sequence numbers start at 1, so a zeroed inbox holds no message
    B200_CUDA(cudaStreamSynchronize(s->stream));
    B200_CUDA(cudaMemset(s->mb_block, 0, bytes));
    s->use_fold = env_int("B200_PP_FOLD", 1) != 0;
    B200_CUDA(cudaDeviceSynchronize());
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    cudaIpcMemHandle_t h;
    B200_CUDA(cudaIpcGetMemHandle(&h, s->mb_block));
    memcpy(handle64, &h, 64);
    return 0;
}

int b200_pipeline_mailbox_connect(b200_slice_t * s, const void * handles, int nranks) {
    if (!s || !handles) return fail(B200_EINVAL, "null argument");
    std::lock_guard<std::mutex> lk(s->mu);
    if (!s->mb_block) return fail(B200_EINVAL, "export this rank's mailbox first");
    if (nranks != s->pp_world || nranks < 2) return fail(B200_EINVAL, "mailbox_connect: %d handles for a pipeline of %d ranks", nranks, s->pp_world);
    if (env_int("B200_PP_PEER", 1) == 0) { s->mb_on = false; return 0; }       // keep the NCCL send/recv path (tested fallback)
    B200_CUDA(cudaSetDevice(s->device));
    const int next = (s->pp_rank + 1) % nranks, prev = (s->pp_rank + nranks - 1) % nranks;
    cudaIpcMemHandle_t hn, hp;
    memcpy(&hn, (const uint8_t *) handles + (size_t) next * 64, 64);
    memcpy(&hp, (const uint8_t *) handles + (size_t) prev * 64, 64);
    void * pn = nullptr, * pp = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&pn, hn, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(B200_ECUDA, "cudaIpcOpenMemHandle(next rank %d) failed: %s", next, cudaGetErrorString(e)); }
    if (prev == next) pp = pn;
    else {
        e = cudaIpcOpenMemHandle(&pp, hp, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) { cudaGetLastError(); cudaIpcCloseMemHandle(pn); return fail(B200_ECUDA, "cudaIpcOpenMemHandle(previous rank %d) failed: %s", prev, cudaGetErrorString(e)); }
    }
    s->mb_next = (uint8_t *) pn; s->mb_prev = (uint8_t *) pp;
    s->mb_on = true;
    return 0;
}

/* Measurement aid: `iters` bare hand-offs of n_rows rows around the ring with NO layers in between (rank 0: send, recv;
 * others: recv, send), on the active transport; returns the device time per iteration in microseconds in *us_per_iter
 * (one iteration = `world` hops).  Every rank must call it. */
int b200_pipeline_pingpong(b200_slice_t * s, int n_rows, int iters, float * us_per_iter) {
    if (!s || !s->nccl_comm || !us_per_iter) return fail(B200_EINVAL, "pipeline not initialised");
    std::lock_guard<std::mutex> lk(s->mu);
    B200_CUDA(cudaSetDevice(s->device));
    const int r = s->pp_rank, W = s->pp_world;
    const size_t count = (size_t) n_rows * s->E;
    NcclApi & n = nccl();
    MailboxHdr * mine = (MailboxHdr *) s->mb_block;
    auto send = [&]() -> int {
        if (s->mb_on) {
            PeerSendArgs sa{mine, (uint2 *)(s->mb_next + sizeof(MailboxHdr)), s->mb_slot_floats, s->d_out, (int) count};
            return launch_simple(s, k_peer_send, dim3((unsigned) std::min<size_t>(32, (count + 8191) / 8192), 1, 1), dim3(1024, 1, 1), 0, sa);
        }
        int rc = n.Send(s->d_out, count, kNcclFloat32, (r + 1) % W, s->nccl_comm, s->stream);
        return rc ? nccl_fail("ncclSend", rc) : 0;
    };
    auto recv = [&]() -> int {
        if (s->mb_on) {
            PeerRecvArgs ra{mine, (const uint2 *)(s->mb_block + sizeof(MailboxHdr)), s->mb_slot_floats, &((MailboxHdr *) s->mb_prev)->ack, s->d_in, (int) count};
            return launch_simple(s, k_peer_recv, dim3((unsigned) std::min<size_t>(32, (count + 8191) / 8192), 1, 1), dim3(1024, 1, 1), 0, ra);
        }
        int rc = n.Recv(s->d_in, count, kNcclFloat32, (r + W - 1) % W, s->nccl_comm, s->stream);
        return rc ? nccl_fail("ncclRecv", rc) : 0;
    };
    cudaEvent_t e0, e1;
    B200_CUDA(cudaEventCreate(&e0)); B200_CUDA(cudaEventCreate(&e1));
    int rc = 0;
    for (int it = 0; it < iters + 8 && !rc; it++) {
        if (it == 8) cudaEventRecord(e0, s->stream);
        if (r == 0) { rc = send(); if (!rc) rc = recv(); }
        else        { rc = recv(); if (!rc) rc = send(); }
    }
    cudaEventRecord(e1, s->stream);
    cudaStreamSynchronize(s->stream);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    *us_per_iter = 1e3f * ms / (float) iters;
    return rc;
}

/* 1 when steps use the peer-memory mailboxes, 0 when they use ncclSend / ncclRecv. */
int b200_pipeline_transport(b200_slice_t * s) { return s && s->mb_on ? 1 : 0; }

/* Force the transport: 0 = NCCL (every rank must do the same, e.g. when ONE rank failed to map a neighbour),
 * 1 = peer mailboxes (only valid after a successful connect). */
int b200_pipeline_set_transport(b200_slice_t * s, int peer) {
    if (!s) return fail(B200_EINVAL, "null handle");
    std::lock_guard<std::mutex> lk(s->mu);
    if (peer && !(s->mb_next && s->mb_prev)) return fail(B200_EINVAL, "peer transport needs connected mailboxes");
    s->mb_on = peer != 0;
    return 0;
}

/* Non-zero if a mailbox poll timed out on this rank since the pipeline was connected (synchronises the stream). */
int b200_pipeline_error(b200_slice_t * s) {
    if (!s || !s->mb_block) return 0;
    cudaSetDevice(s->device);
    cudaStreamSynchronize(s->stream);
    int err = 0;
    cudaMemcpy(&err, s->mb_block + offsetof(MailboxHdr, err), 4, cudaMemcpyDeviceToHost);
    return err;
}

/* Rank 0: receive one final activation ([n_rows][n_embd]) that a step issued with ring = 2 left in flight, into d_dst
 * (NULL: the buffer b200_pipeline_result() returns).  Results arrive in the order the steps were issued.  Other ranks: no-op.
 * This is what keeps every slice busy in throughput mode: rank 0 issues steps for sessions k, k+1, ... back to back and
 * collects session k's result only when it needs it (rank r then works on session k while rank r+1 works on k-1). */
int b200_pipeline_collect(b200_slice_t * s, int n_rows, float * d_dst) {
    if (!s || !s->nccl_comm) return fail(B200_EINVAL, "pipeline not initialised");
    std::lock_guard<std::mutex> lk(s->mu);
    if (s->pp_rank != 0 || s->pp_world < 2) return 0;
    if (n_rows <= 0 || n_rows > s->n_ctx) return fail(B200_EINVAL, "n_rows %d outside [1, n_ctx]", n_rows);
    B200_CUDA(cudaSetDevice(s->device));
    float * dst = d_dst ? d_dst : s->d_final;
    const size_t count = (size_t) n_rows * s->E;
    if (s->mb_on) {
        PeerRecvArgs rf{(MailboxHdr *) s->mb_block, (const uint2 *)(s->mb_block + sizeof(MailboxHdr)), s->mb_slot_floats,
                        &((MailboxHdr *) s->mb_prev)->ack, dst, (int) count};
        s->cur_class = 6;
        int rc = launch_simple(s, k_peer_recv, dim3((unsigned) std::min<size_t>(32, (count + 8191) / 8192), 1, 1), dim3(1024, 1, 1), 0, rf);
        if (rc) return rc;
    } else {
        NcclApi & n = nccl();
        int rc = n.Recv(dst, count, kNcclFloat32, s->pp_world - 1, s->nccl_comm, s->stream);
        if (rc) return nccl_fail("ncclRecv", rc);
        s->launches++;
    }
    return 0;
}

/* Device pointer of the pipeline's final activation on rank 0 (valid after a `ring` step), else dev_out. */
float * b200_pipeline_result(b200_slice_t * s) { return s ? (s->pp_world > 1 && s->pp_rank == 0 && s->d_final ? s->d_final : s->d_out) : nullptr; }

int b200_pipeline_destroy(b200_slice_t * s) {
    if (!s) return fail(B200_EINVAL, "null handle");
    std::lock_guard<std::mutex> lk(s->mu);
    if (s->nccl_comm) {
        cudaSetDevice(s->device);
        cudaStreamSynchronize(s->stream);
        NcclApi & n = nccl();
        if (n.CommDestroy) n.CommDestroy(s->nccl_comm);
        s->nccl_comm = nullptr; s->pp_world = 1; s->pp_rank = 0;
        for (auto & kv : s->pp_graphs) cudaGraphExecDestroy(kv.second);
        s->pp_graphs.clear();
        if (s->mb_next) cudaIpcCloseMemHandle(s->mb_next);
        if (s->mb_prev && s->mb_prev != s->mb_next) cudaIpcCloseMemHandle(s->mb_prev);
        s->mb_next = s->mb_prev = nullptr; s->mb_on = false;
    }
    return 0;
}

}  // extern "C"

// ============================================================================ client-side extra layers (N1)
// tok_embeddings lookup, final RMSNorm + lm_head, argmax, tokenizer -- resident, instead of the reference
// re-opening and re-reading the extra-layers file on every call (tensor_processor.cpp:1717-1908, 2033-2057,
// 2219-2235).  The lm_head is the same exact-mode weight matmul as the slice layers (RMSNorm prologue fused).
#include <queue>
#include <unordered_map>

struct b200_extra {
    b200_slice ctx;                       // device / stream / launch plumbing shared with the slice kernels
    int n_vocab = 0, E = 0, emb_type = 0, out_type = 0;
    uint8_t * emb_raw = nullptr;          // tok_embeddings as stored (row = token)
    float * norm_w = nullptr;
    PackedW out{}; uint16_t * out_f16 = nullptr; uint8_t * out_q6k = nullptr;
    float * d_x = nullptr, * d_logits = nullptr; int32_t * d_tok = nullptr, * d_best = nullptr; int cap_tokens = 0;
    std::vector<std::pair<std::string, float>> vocab;
    std::unordered_map<std::string, int> token_to_id;
    std::mutex mu;
};

namespace b200 {

__global__ void k_embed_rows(const uint8_t * emb, int type, int E, const int32_t * tok, int n_vocab, float * out) {
    const int n = blockIdx.y, t = tok[n];
    float * dst = out + (size_t) n * E;
    if (t < 0 || t >= n_vocab) { for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < E; i += gridDim.x * blockDim.x) dst[i] = 0.f; return; }
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < E; i += gridDim.x * blockDim.x) {
        float v;
        if (type == kWT_Q4_0) {                      // dequantize_row_q4_0, ggml.c:1523-1541
            const uint8_t * blk = emb + ((size_t) t * (E / 32) + i / 32) * 18;
            const float d = h2f(*(const uint16_t *) blk);
            const int j = i & 31, q = blk[2 + (j & 15)];
            v = fmul((float)((j < 16 ? (q & 0x0F) : (q >> 4)) - 8), d);
        } else if (type == kWT_Q4_1) {               // dequantize_row_q4_1, ggml.c:1543-1562: nibble * d, then + m (two roundings)
            const uint8_t * blk = emb + ((size_t) t * (E / 32) + i / 32) * 20;
            const float d = h2f(*(const uint16_t *) blk), m = h2f(*(const uint16_t *)(blk + 2));
            const int j = i & 31, q = blk[4 + (j & 15)];
            v = fadd(fmul((float)(j < 16 ? (q & 0x0F) : (q >> 4)), d), m);
        } else if (type == kWT_Q8_0) {
            const uint8_t * blk = emb + ((size_t) t * (E / 32) + i / 32) * 34;
            v = fmul((float)((const int8_t *)(blk + 2))[i & 31], h2f(*(const uint16_t *) blk));
        } else if (type == kWT_F16) v = h2f(((const uint16_t *) emb)[(size_t) t * E + i]);
        else v = ((const float *) emb)[(size_t) t * E + i];
        dst[i] = v;
    }
}

static int extra_reserve(b200_extra * e, int n) {
    if (n <= e->cap_tokens) return 0;
    b200_slice * s = &e->ctx;
    // growth: release the old staging buffers first (they are tracked in `allocs` for unload)
    cudaStreamSynchronize(s->stream);
    for (void * old : {(void *) e->d_x, (void *) e->d_logits, (void *) e->d_tok, (void *) e->d_best}) {
        if (!old) continue;
        s->allocs.erase(std::remove(s->allocs.begin(), s->allocs.end(), old), s->allocs.end());
        cudaFree(old);
    }
    e->d_x = nullptr; e->d_logits = nullptr; e->d_tok = nullptr; e->d_best = nullptr; e->cap_tokens = 0;
    int rc;
    if ((rc = dev_alloc(s, &e->d_x, (size_t) n * e->E)) || (rc = dev_alloc(s, &e->d_logits, (size_t) n * e->n_vocab)) ||
        (rc = dev_alloc(s, &e->d_tok, (size_t) n)) || (rc = dev_alloc(s, &e->d_best, (size_t) 1))) return rc;
    e->cap_tokens = n;
    return 0;
}

// sample_next_token (tensor_processor.cpp:1894-1908): best = -1e12, id = 0; `if (logit > best)` in index order, i.e. the
// FIRST maximum wins, NaNs never win, and a row that never exceeds -1e12 yields id 0.  One block over the row.
__global__ void __launch_bounds__(1024) k_argmax_first(const float * logits, int n, int32_t * out) {
    __shared__ float sv[32]; __shared__ int si[32];
    float bv = -(1000000000000.0f); int bi = 0x7fffffff;
    for (int i = threadIdx.x; i < n; i += blockDim.x) { const float v = logits[i]; if (v > bv) { bv = v; bi = i; } }
    auto better = [](float v, int i, float bv, int bi) { return v > bv || (v == bv && i < bi); };
    for (int o = 16; o > 0; o >>= 1) {
        const float v = __shfl_xor_sync(0xffffffffu, bv, o); const int i = __shfl_xor_sync(0xffffffffu, bi, o);
        if (better(v, i, bv, bi)) { bv = v; bi = i; }
    }
    if ((threadIdx.x & 31) == 0) { sv[threadIdx.x >> 5] = bv; si[threadIdx.x >> 5] = bi; }
    __syncthreads();
    if (threadIdx.x < 32) {
        bv = threadIdx.x < (blockDim.x >> 5) ? sv[threadIdx.x] : -(1000000000000.0f);
        bi = threadIdx.x < (blockDim.x >> 5) ? si[threadIdx.x] : 0x7fffffff;
        for (int o = 16; o > 0; o >>= 1) {
            const float v = __shfl_xor_sync(0xffffffffu, bv, o); const int i = __shfl_xor_sync(0xffffffffu, bi, o);
            if (better(v, i, bv, bi)) { bv = v; bi = i; }
        }
        if (threadIdx.x == 0) *out = bi == 0x7fffffff ? 0 : bi;
    }
}

// sentencepiece-style greedy bigram merging, as tensor_processor.cpp:1596-1714 specifies it:
// start from UTF-8 characters, repeatedly merge the adjacent pair whose concatenation is the vocabulary
// entry with the highest score (ties: leftmost), then map pieces to ids, unknown pieces to byte ids (+3).
static void tokenize_pieces(const b200_extra & e, const std::string & text, std::vector<int32_t> & out) {
    struct Piece { int prev, next; size_t off, len; };
    struct Cand { float score; int left, right; size_t len; };
    struct Worse { bool operator()(const Cand & a, const Cand & b) const { return a.score < b.score || (a.score == b.score && a.left > b.left); } };
    std::vector<Piece> ps;
    for (size_t off = 0; off < text.size();) {
        static const size_t lens[16] = {1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 2, 2, 3, 4};
        size_t n = std::min(text.size() - off, lens[(uint8_t) text[off] >> 4]);
        const int idx = (int) ps.size();
        ps.push_back({idx - 1, off + n == text.size() ? -1 : idx + 1, off, n});
        off += n;
    }
    std::priority_queue<Cand, std::vector<Cand>, Worse> heap;
    auto offer = [&](int l, int r) {
        if (l < 0 || r < 0) return;
        const std::string joined = text.substr(ps[l].off, ps[l].len + ps[r].len);
        auto it = e.token_to_id.find(joined);
        if (it == e.token_to_id.end() || (size_t) it->second >= e.vocab.size()) return;
        heap.push({e.vocab[it->second].second, l, r, joined.size()});
    };
    for (int i = 1; i < (int) ps.size(); i++) offer(i - 1, i);
    while (!heap.empty()) {
        const Cand c = heap.top(); heap.pop();
        Piece & L = ps[c.left]; Piece & R = ps[c.right];
        if (L.len == 0 || R.len == 0 || L.len + R.len != c.len) continue;      // stale candidate
        L.len += R.len; R.len = 0;
        L.next = R.next;
        if (R.next >= 0) ps[R.next].prev = c.left;
        offer(L.prev, c.left);
        offer(c.left, L.next);
    }
    for (int i = ps.empty() ? -1 : 0; i != -1; i = ps[i].next) {
        auto it = e.token_to_id.find(text.substr(ps[i].off, ps[i].len));
        if (it != e.token_to_id.end()) out.push_back(it->second);
        else for (size_t j = 0; j < ps[i].len; j++) out.push_back((int32_t)(uint8_t) text[ps[i].off + j] + 3);
    }
}

}  // namespace b200

extern "C" {

int b200_extra_load(const char * path, int device, b200_extra_t ** out) {
    if (!path || !out) return fail(B200_EINVAL, "b200_extra_load: null argument");
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(B200_ENODEV, "no CUDA device visible: no CPU fallback");
    if (device < 0 || device >= ndev) return fail(B200_ENODEV, "device %d out of range", device);
    cudaDeviceProp prop;
    B200_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail(B200_ENODEV, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
    B200_CUDA(cudaSetDevice(device));
    std::unique_ptr<GgjtFile> fp;
    try { fp.reset(new GgjtFile(path, true)); }
    catch (const std::exception & ex) { return fail(B200_EFILE, "error loading extra layers: %s", ex.what()); }
    GgjtFile & f = *fp;
    // frees the stream and every device allocation if the load fails half-way (a node keeps running after a bad extra-layers file)
    struct ExtraGuard {
        b200_extra * p;
        ~ExtraGuard() {
            if (!p) return;
            b200_slice * c = &p->ctx;
            if (c->stream) cudaStreamSynchronize(c->stream);
            for (void * q : c->allocs) cudaFree(q);
            if (c->ev0) cudaEventDestroy(c->ev0);
            if (c->ev1) cudaEventDestroy(c->ev1);
            if (c->stream) cudaStreamDestroy(c->stream);
            delete p;
        }
    };
    ExtraGuard e_guard{new b200_extra()};
    b200_extra * e = e_guard.p;
    b200_slice * s = &e->ctx;
    s->device = device; s->n_sm = prop.multiProcessorCount;
    s->use_pdl = false; s->use_graph = false;
    B200_CUDA(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
    e->n_vocab = (int) f.n_vocab; e->E = (int) f.n_embd;
    const uint32_t E = f.n_embd, V = f.n_vocab;
    int rc;
    try {
        const GgjtTensor & te = f.get("tok_embeddings.weight", {E, V});
        const GgjtTensor & tn = f.get("norm.weight", {E});
        const GgjtTensor & to = f.get("output.weight", {E, V});
        e->emb_type = (int) te.type; e->out_type = (int) to.type;
        if (te.type != GT_Q4_0 && te.type != GT_Q4_1 && te.type != GT_Q8_0 && te.type != GT_F16 && te.type != GT_F32)
            return fail(B200_EFILE, "tok_embeddings type %u unsupported", te.type);
        if (to.type != GT_Q4_0 && to.type != GT_Q4_1 && to.type != GT_Q8_0 && to.type != GT_F16 && to.type != GT_Q6_K)
            return fail(B200_EFILE, "output.weight type %u unsupported (Q4_0, Q4_1, Q8_0, F16, Q6_K)", to.type);
        if (to.type == GT_Q6_K && E % 256) return fail(B200_EFILE, "Q6_K output.weight needs n_embd %% 256 == 0");
        if (tn.type != GT_F32) return fail(B200_EFILE, "norm.weight must be F32");
        if ((rc = dev_alloc(s, &e->emb_raw, te.nbytes)) || (rc = dev_alloc(s, &e->norm_w, (size_t) E))) return rc;
        B200_CUDA(cudaMemcpyAsync(e->norm_w, f.data(tn), (size_t) E * 4, cudaMemcpyHostToDevice, s->stream));
        std::vector<LoadJob> jobs;
        LoadJob je; je.kind = 2; je.nsrc = 1; je.src[0] = &te; je.raw_dst = e->emb_raw; jobs.push_back(je);
        LoadJob jo; jo.nsrc = 1; jo.src[0] = &to;
        if (to.type == GT_Q6_K) {
            if ((rc = dev_alloc(s, &e->out_q6k, (size_t) V * (E / 256) * kQ6Packed))) return rc;
            jo.kind = 3; jo.raw_dst = e->out_q6k;
        } else if (to.type == GT_F16) { jo.kind = 1; jo.outf = &e->out_f16; }
        else { jo.kind = 0; jo.mode = 0; jo.G = 1; jo.out = &e->out; }
        jobs.push_back(jo);
        if ((rc = run_load_jobs(s, f, jobs))) return rc;
    } catch (const std::exception & ex) { return fail(B200_EFILE, "error loading extra layers: %s", ex.what()); }
    // fp16 SiLU table is not needed here, but the launch helper wants events
    B200_CUDA(cudaEventCreate(&s->ev0));
    B200_CUDA(cudaEventCreate(&s->ev1));
    e->vocab = std::move(f.vocab);
    for (int i = 0; i < (int) e->vocab.size(); i++) e->token_to_id[e->vocab[i].first] = i;
    *out = e;
    e_guard.p = nullptr;
    return 0;
}

int b200_extra_unload(b200_extra_t * e) {
    if (!e) return fail(B200_EINVAL, "null handle");
    b200_slice * s = &e->ctx;
    cudaSetDevice(s->device);
    if (s->stream) cudaStreamSynchronize(s->stream);
    for (void * p : s->allocs) cudaFree(p);
    if (s->ev0) cudaEventDestroy(s->ev0);
    if (s->ev1) cudaEventDestroy(s->ev1);
    for (cudaEvent_t ev : s->prof_ev) cudaEventDestroy(ev);
    if (s->stream) cudaStreamDestroy(s->stream);
    delete e;
    return 0;
}

int b200_extra_dims(b200_extra_t * e, int * n_vocab, int * n_embd) {
    if (!e) return fail(B200_EINVAL, "null handle");
    if (n_vocab) *n_vocab = e->n_vocab;
    if (n_embd) *n_embd = e->E;
    return 0;
}

int b200_extra_embed(b200_extra_t * e, const int32_t * tokens, int n_tokens, float * out) {
    if (!e || !tokens || !out || n_tokens <= 0) return fail(B200_EINVAL, "bad argument");
    std::lock_guard<std::mutex> lk(e->mu);
    b200_slice * s = &e->ctx;
    B200_CUDA(cudaSetDevice(s->device));
    int rc = extra_reserve(e, n_tokens);
    if (rc) return rc;
    B200_CUDA(cudaMemcpyAsync(e->d_tok, tokens, (size_t) n_tokens * 4, cudaMemcpyHostToDevice, s->stream));
    k_embed_rows<<<dim3((e->E + 255) / 256, n_tokens), 256, 0, s->stream>>>(e->emb_raw, e->emb_type, e->E, e->d_tok, e->n_vocab, e->d_x);
    B200_CUDA(cudaGetLastError());
    s->launches++;
    B200_CUDA(cudaMemcpyAsync(out, e->d_x, (size_t) n_tokens * e->E * 4, cudaMemcpyDeviceToHost, s->stream));
    B200_CUDA(cudaStreamSynchronize(s->stream));
    return 0;
}

static int extra_logits_device(b200_extra * e, const float * emb, int n_tokens) {
    b200_slice * s = &e->ctx;
    int rc = extra_reserve(e, n_tokens);
    if (rc) return rc;
    B200_CUDA(cudaMemcpyAsync(e->d_x, emb, (size_t) n_tokens * e->E * 4, cudaMemcpyHostToDevice, s->stream));
    if (e->out_type == kWT_Q6_K) {
        LmHeadQ6Args q{e->out_q6k, e->n_vocab, e->E, e->d_x, e->E, e->norm_w, e->d_logits, e->n_vocab, n_tokens};
        const size_t smem = (size_t)(e->E / 256) * (64 * 4 + 4) + (size_t) e->E * 4 + 64;
        static bool attr_set[16] = {false};
        if (!attr_set[s->device & 15]) {
            B200_CUDA(cudaFuncSetAttribute(k_lmhead_q6k, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
            attr_set[s->device & 15] = true;
        }
        return launch_simple(s, k_lmhead_q6k, dim3((e->n_vocab + 31) / 32, n_tokens, 1), dim3(256, 1, 1), smem, q);
    }
    if (e->out_type == kWT_F16) {
        GemvF16Args f{}; f.K = e->E; f.x = e->d_x; f.ldx = e->E; f.norm_w = e->norm_w; f.N = n_tokens;
        f.rows = e->n_vocab; f.W = e->out_f16; f.y = e->d_logits; f.ldy = e->n_vocab;
        return launch_f16<PRO_NORM, EPI_STORE>(s, f);
    }
    GemvArgs g{}; g.W = e->out; g.x = e->d_x; g.ldx = e->E; g.norm_w = e->norm_w; g.y = e->d_logits; g.ldy = e->n_vocab;
    g.N = n_tokens; g.out_rows = e->n_vocab;
    return launch_gemv<1, PRO_NORM, EPI_STORE>(s, g);
}

int b200_extra_logits(b200_extra_t * e, const float * emb, int n_tokens, int all_logits, float * out) {
    if (!e || !emb || !out || n_tokens <= 0) return fail(B200_EINVAL, "bad argument");
    std::lock_guard<std::mutex> lk(e->mu);
    b200_slice * s = &e->ctx;
    B200_CUDA(cudaSetDevice(s->device));
    int rc = extra_logits_device(e, emb, n_tokens);
    if (rc) return rc;
    const size_t V = (size_t) e->n_vocab;
    if (all_logits) B200_CUDA(cudaMemcpyAsync(out, e->d_logits, (size_t) n_tokens * V * 4, cudaMemcpyDeviceToHost, s->stream));
    else B200_CUDA(cudaMemcpyAsync(out, e->d_logits + (size_t)(n_tokens - 1) * V, V * 4, cudaMemcpyDeviceToHost, s->stream));
    B200_CUDA(cudaStreamSynchronize(s->stream));
    return 0;
}

int b200_extra_next_token(b200_extra_t * e, const float * emb, int n_tokens, int32_t * token) {
    if (!e || !emb || !token || n_tokens <= 0) return fail(B200_EINVAL, "bad argument");
    std::lock_guard<std::mutex> lk(e->mu);
    b200_slice * s = &e->ctx;
    B200_CUDA(cudaSetDevice(s->device));
    // only the LAST token's logits decide (get_llm_output + sample_next_token, tensor_processor.cpp:1787-1908); rows of
    // the lm_head are independent, so computing that row alone is the same arithmetic.  The argmax runs on the device:
    // 4 bytes come back instead of n_vocab floats.
    int rc = extra_logits_device(e, emb + (size_t)(n_tokens - 1) * e->E, 1);
    if (rc) return rc;
    k_argmax_first<<<1, 1024, 0, s->stream>>>(e->d_logits, e->n_vocab, e->d_best);
    B200_CUDA(cudaGetLastError());
    s->launches++;
    B200_CUDA(cudaMemcpyAsync(token, e->d_best, 4, cudaMemcpyDeviceToHost, s->stream));
    B200_CUDA(cudaStreamSynchronize(s->stream));
    return 0;
}

int b200_extra_tokenize(b200_extra_t * e, const char * prompt, int32_t * out, int cap) {
    if (!e || !prompt) return -B200_EINVAL;
    const std::string text(prompt);
    std::vector<int32_t> ids;
    if (!text.empty()) { ids.push_back(1); tokenize_pieces(*e, text, ids); }      // BOS = 1 (llama_token_bos)
    for (int i = 0; i < (int) ids.size() && i < cap && out; i++) out[i] = ids[i];
    return (int) ids.size();
}

const char * b200_extra_token_text(b200_extra_t * e, int32_t id, int * len) {
    if (!e || id < 0 || id >= (int32_t) e->vocab.size()) { if (len) *len = 0; return nullptr; }
    if (len) *len = (int) e->vocab[id].first.size();
    return e->vocab[id].first.data();
}

}  // extern "C"
