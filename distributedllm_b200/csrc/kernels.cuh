// kernels.cuh -- the sm_100a kernels of the slice forward (exact mode).
//
// "Exact mode" = every rounding point and accumulation order of the reference's CPU path
// (ggml's AVX2+FMA+F16C build) is reproduced, so hidden states are bit-identical:
//   weight matmul   ggml_vec_dot_q4_0_q8_0 / q8_0_q8_0   ggml.c:2432-2455, 3313-3335, hsum 614-620
//   act-quant       quantize_row_q8_0 (AVX branch)        ggml.c:1215-1252
//   RMSNorm         ggml_compute_forward_rms_norm_f32     ggml.c:10309-10352 (+ ggml_mul 9062)
//   RoPE            ggml_compute_forward_rope_f32 mode 0  ggml.c:11956-12055
//   K.q / V.p       ggml_vec_dot_f16 + GGML_F32x8_REDUCE  ggml.c:2323-2357, 1895-1913
//   softmax         ggml_compute_forward_soft_max_f32     ggml.c:11524-11590
//   SiLU            ggml_vec_silu_f32 (GGML_SILU_FP16)    ggml.c:3541-3560
// graph order: tensor_processor.cpp:537-766.
#pragma once
#include "common.cuh"

namespace b200 {

// =============================================================================================
// Packed weight layout (HBM).  A matrix W[rows][K] of 32-wide blocks is cut into
//   row-groups of 8 rows  x  quads of 4 consecutive blocks            -> one CHUNK
//   tiles of TR row-groups (one CTA's rows), all quads of the tile contiguous, q-major:
//       tile t : [q = 0..nbq) [rg = 0..TR) [chunk bytes]
// Q4_0 chunk (576 B = the file's 18 B/block, nothing added):
//       512 B : lane L = 4*r + w (r = row in group, w = 32-bit word of the 16 nibble bytes)
//               holds 16 B = word w of blocks 4q..4q+3 of row r; nibbles stored as two's-complement
//               4-bit (file nibble XOR 8), so `(x<<4)&0xF0F0F0F0` / `x&0xF0F0F0F0` are 16*(nibble-8)
//               as signed bytes, ready for dp4a
//        64 B : fp16 d of row r, blocks 4q..4q+3 at 512 + 8*r
// Q8_0 chunk (1088 B = 34 B/block): 512 B words w of 4 blocks per lane, 512 B words w+4, 64 B scales.
// Q4_1 chunk (640 B = 20 B/block): the Q4_0 shape with the nibbles left UNSIGNED (0..15, no XOR) + 64 B of fp16 minima
//       at 576 + 8*r.  ggml_vec_dot_q4_1_q8_1 (ggml.c:2700-2733): acc_l = fma(d0*d1, float(sum n*a), acc_l) with an
//       f32 (unrounded) activation scale d1, plus a SCALAR chain summs += m * s (s = d1 * sum of the block's quants).
// A warp reads a chunk with one conflict-free LDS.128 (+ one LDS.64) per lane.
// =============================================================================================
constexpr int kWT_F16 = 1, kWT_Q4_0 = 2, kWT_Q4_1 = 3, kWT_Q8_0 = 8;
constexpr int kQ4Chunk = 576, kQ41Chunk = 640, kQ8Chunk = 1088;
constexpr int kWPC = 4;                 // consumer warps per CTA (8 rows x G groups each)
constexpr int kConsumers = kWPC * 32;
constexpr int kQS = 4;                  // quads per ring stage (nbq is padded to a multiple of kQS at pack time)
constexpr float kMagic = 12582912.0f;   // 1.5 * 2^23: int->float through the dp4a accumulator
constexpr int kMagicI = 0x4B400000;

__host__ __device__ constexpr int chunk_bytes(int wt) { return wt == kWT_Q4_0 ? kQ4Chunk : (wt == kWT_Q4_1 ? kQ41Chunk : kQ8Chunk); }
__host__ __device__ constexpr bool wt_nibbles(int wt) { return wt == kWT_Q4_0 || wt == kWT_Q4_1; }

struct PackedW {
    const uint8_t * data;
    int wtype, rows, K, nb, nbq, TR, n_tiles;
    long long tile_bytes;
};

// ---- repack: raw GGJT blocks -> packed layout (one thread per output 32-bit word) -----------
// mode 0: single source; 1: three sources concatenated by rows (wq|wk|wv); 2: two sources with
// row-groups interleaved (even = w1, odd = w3) so one warp owns row r of both for the SiLU gate.
struct RepackArgs {
    const uint8_t * src[3];
    int mode, wtype, rows_per_src, nb, nbq, TR, n_tiles;
    uint8_t * dst;
};

__global__ void k_repack(RepackArgs a) {
    const int cb = chunk_bytes(a.wtype), words = cb / 4;
    const long long total = (long long) a.n_tiles * a.nbq * a.TR * words;
    for (long long i = blockIdx.x * (long long) blockDim.x + threadIdx.x; i < total; i += (long long) gridDim.x * blockDim.x) {
        const int wi = (int)(i % words);
        long long c = i / words;
        const int rg = (int)(c % a.TR); c /= a.TR;
        const int q = (int)(c % a.nbq);
        const int tile = (int)(c / a.nbq);
        const int gi = tile * a.TR + rg;                    // global row-group index
        int s, sg;
        if (a.mode == 1)      { const int gps = a.rows_per_src / 8; s = gi / gps; sg = gi % gps; }
        else if (a.mode == 2) { s = gi & 1; sg = gi >> 1; }
        else                  { s = 0; sg = gi; }
        const int bsz = a.wtype == kWT_Q4_0 ? 18 : (a.wtype == kWT_Q4_1 ? 20 : 34);
        uint32_t out = 0;
        const bool src_ok = s < 3 && a.src[s] != nullptr;
        if (wt_nibbles(a.wtype)) {
            const bool q41 = a.wtype == kWT_Q4_1;
            if (wi < 128) {                                  // nibble words
                const int lane = wi >> 2, bq = wi & 3, r = lane >> 2, w = lane & 3;
                const int row = sg * 8 + r, b = q * 4 + bq;
                if (src_ok && row < a.rows_per_src && b < a.nb) {
                    const uint8_t * blk = a.src[s] + ((long long) row * a.nb + b) * bsz;
                    const uint16_t * p = (const uint16_t *)(blk + (q41 ? 4 : 2) + 4 * w);
                    out = ((uint32_t) p[0] | ((uint32_t) p[1] << 16)) ^ (q41 ? 0u : 0x88888888u);
                }
            } else {                                         // scales (then Q4_1 minima): 16 words = 8 rows x 4 halves
                const int sel = (wi - 128) >> 4;             // 0: d at +0, 1: m at +2
                const int h0 = ((wi - 128) & 15) * 2;
                uint32_t v[2] = {0, 0};
                for (int k = 0; k < 2; k++) {
                    const int r = (h0 + k) >> 2, bq = (h0 + k) & 3, row = sg * 8 + r, b = q * 4 + bq;
                    if (src_ok && row < a.rows_per_src && b < a.nb)
                        v[k] = *(const uint16_t *)(a.src[s] + ((long long) row * a.nb + b) * bsz + 2 * sel);
                }
                out = v[0] | (v[1] << 16);
            }
        } else {                                             // Q8_0
            if (wi < 256) {
                const int half = wi >> 7, lw = wi & 127, lane = lw >> 2, bq = lw & 3, r = lane >> 2, w = (lane & 3) + 4 * half;
                const int row = sg * 8 + r, b = q * 4 + bq;
                if (src_ok && row < a.rows_per_src && b < a.nb) {
                    const uint8_t * blk = a.src[s] + ((long long) row * a.nb + b) * bsz;
                    const uint16_t * p = (const uint16_t *)(blk + 2 + 4 * w);
                    out = (uint32_t) p[0] | ((uint32_t) p[1] << 16);
                }
            } else {
                const int h0 = (wi - 256) * 2;
                uint32_t v[2] = {0, 0};
                for (int k = 0; k < 2; k++) {
                    const int r = (h0 + k) >> 2, bq = (h0 + k) & 3, row = sg * 8 + r, b = q * 4 + bq;
                    if (src_ok && row < a.rows_per_src && b < a.nb)
                        v[k] = *(const uint16_t *)(a.src[s] + ((long long) row * a.nb + b) * bsz);
                }
                out = v[0] | (v[1] << 16);
            }
        }
        ((uint32_t *) a.dst)[i] = out;
    }
}

// =============================================================================================
// K1: block-quantised weight matmul, exact mode (decode GEMV and NC-column prefill).
//
//   y[n][row] = hsum_l( fma_b( D_b, (float) sum_j w_j a_j, acc_l ) )      (ggml.c:2431-2455)
//
// Thread (r, w) of a consumer warp owns AVX lanes l = w and l = w+4 of row r: for every block it
// takes ONE 32-bit word of nibbles, splits it into the two lanes' signed bytes, and runs two
// dp4a -> fadd -> fma chains strictly in block order.  Parallelism comes from rows, never from K.
//   * warp  = 8 rows x G row-groups; CTA = 4 consumer warps (+1 producer warp)
//   * producer lane streams the tile's chunks with 1-D bulk async copies (UBLKCP) into a ring of
//     NS stages guarded by full/empty mbarriers; it starts BEFORE griddepcontrol.wait because the
//     weights never depend on the previous kernel -- the HBM stream runs across kernel boundaries
//   * prologue (fused, per CTA): [RMSNorm * weight ->] Q8_0 act-quant of the input column(s) into
//     shared memory in dp4a word order
//   * epilogue (fused): store | + residual | SiLU(w1 x) * (w3 x)
// =============================================================================================
// =============================================================================================
// Inter-slice hand-off through PEER MEMORY (NVLink / NVSwitch), no host and no NCCL kernel in the path.
// Every rank owns a MAILBOX in its own HBM, mapped into its ring neighbours (cudaIpc):
//     ack                    written by the NEXT rank: highest sequence number it has consumed from OUR sends
//     inbox[kMbSlots][n_ctx * n_embd] of 8-byte ELEMENTS {f32 bits, sequence number}
// The payload carries its own flag ("LL" style: a 64-bit store is single-copy atomic, so a reader that sees the sequence
// number in the high word has the value in the low word): the sender needs NO fence and NO separate flag write, the
// latency of a hop is one NVLink store plus a poll.
//   * sender = the slice's LAST matmul itself for single-token steps (EPI_RESID_SEND: every output row is stored to the
//     local buffer and, as {value, seq}, into the next rank's inbox the moment it is computed), or k_peer_send for
//     multi-row steps;
//   * receiver = k_peer_recv, first kernel of the next slice's step: every thread polls ITS elements until they carry
//     the expected sequence number, compacts them into the slice's input buffer and acknowledges the slot.  It sits
//     inside the step's captured graph with programmatic dependent launch: while it polls, the slice's first weight
//     matmul is already resident and streaming weights into shared memory.
// Sequence counters are per link and live in device memory, so a graph replay needs no host-side argument.  The sender
// reuses a slot only after the receiver acknowledged message seq - kMbSlots.  A poll that exceeds kMbTimeoutNs sets
// *err and falls through (the host reports it) instead of hanging the GPU.
// =============================================================================================
constexpr int kMbSlots = 2;
constexpr unsigned long long kMbTimeoutNs = 8000000000ull;

struct MailboxHdr {              // first 256 bytes of a mailbox block
    int pad0[16];
    int ack;                     // remote-written (next rank)
    int pad1[15];
    int seq_in, seq_out;         // local counters: messages consumed / produced on my inbound / outbound link
    int err;                     // local: a poll timed out
    int cnt_send, cnt_recv;      // local: last-CTA election of multi-CTA sends / receives
    int pad2[27];
};
static_assert(sizeof(MailboxHdr) == 256, "mailbox header layout");

__device__ __forceinline__ int ld_relaxed_sys(const int * p) {
    int v; asm volatile("ld.relaxed.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v;
}
__device__ __forceinline__ void st_relaxed_sys(int * p, int v) {
    asm volatile("st.relaxed.sys.global.s32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint2 ld_ll(const uint2 * p) {
    uint2 v; asm volatile("ld.relaxed.sys.global.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory"); return v;
}
__device__ __forceinline__ void st_ll(uint2 * p, float val, int seq) {
    asm volatile("st.relaxed.sys.global.v2.u32 [%0], {%1, %2};" :: "l"(p), "r"(__float_as_uint(val)), "r"((uint32_t) seq) : "memory");
}
// wait until the receiver has consumed message seq - kMbSlots (the slot message `seq` is about to overwrite)
__device__ __forceinline__ void mb_wait_slot_free(MailboxHdr * mine, int seq) {
    const unsigned long long t0 = gtime();
    while (ld_relaxed_sys(&mine->ack) < seq - kMbSlots)
        if (gtime() - t0 > kMbTimeoutNs) { mine->err = 1; break; }
}

enum { PRO_PLAIN = 0, PRO_NORM = 1, PRO_PREQ = 2 };
enum { EPI_STORE = 0, EPI_RESID = 1, EPI_GATE = 2, EPI_GATEQ = 3, EPI_RESID_NQ = 4, EPI_RESID_SEND = 5 };

struct GemvArgs {
    PackedW W;
    const float * x;      int ldx;       // PRO_PLAIN / PRO_NORM: input [N][ldx], K valid per row
    const float * norm_w;                // PRO_NORM: weight [K]
    const int * aq_in; const float * da_in;   // PRO_PREQ: pre-quantised input, [N][nbq*32] words + [N][nbq*4] scales
    int in_soff, out_soff;               // Q4_1 weights (Q8_1 activations): the block sums s live in a second plane, this many
                                         // floats behind the scales (da_in / da_out); 0 for Q8_0 activations
    const float * resid;  int ldr;       // EPI_RESID
    float * y;            int ldy;       // output [N][ldy]
    int * aq_out; float * da_out; int out_nbq; float out_dscale;   // EPI_GATEQ / EPI_RESID_NQ: quantised output for the next matmul
    const float * nq_norm_w; int * nq_counter; double * nq_partial;   // EPI_RESID_NQ: next RMSNorm weight [out_rows]; 2 counters per column group; per-tile sums of squares
    int N;                               // columns (tokens)
    int out_rows;                        // valid output rows (E, 3E, or FF for the gate)
    const uint16_t * tsilu;              // EPI_GATE*: fp16 SiLU table (65536 entries)
    int NS;                              // ring stages
    unsigned long long * trace;          // debug timeline (B200_TRACE), or null
    int pre_stages;                      // ring stages the producer may request before the prologue loads are issued
    int dbg_nomath;                      // debug: consume ring stages without computing (streaming-rate probe)
    // pipeline hand-off folded into the slice's first / last matmul (single-token steps; see "PEER MEMORY" above)
    MailboxHdr * mb_mine;                // EPI_RESID_SEND: this rank's mailbox (ack, seq_out)
    uint2 * mb_peer_inbox; size_t mb_slot_elems;   // EPI_RESID_SEND: next rank's inbox (mapped peer memory), elements per slot
};

__host__ __device__ inline size_t act_bytes_per_col(int nbq, int wt) { return (size_t) nbq * (128 + 16 + (wt == kWT_Q4_1 ? 16 : 0)); }


// (double) of a NON-NEGATIVE float, bit-exact, on the integer pipes: F2F.F64.F32 runs on the quarter-rate XU pipe and
// the RMSNorm prologue needs 32 of them per thread.  Zero and subnormal inputs take the slow path.
__device__ __forceinline__ double widen_nonneg(float f) {
    const uint32_t u = __float_as_uint(f);
    if (u - 0x00800000u < 0x7F000000u) return __hiloint2double((int)((u >> 3) + 0x38000000u), (int)(u << 29));
    return (double) f;
}
// rint() of |x| <= 2^22 through the FMA pipe (round-half-even, as F2I.RN / _mm256_round_ps(NEAREST)) instead of XU
__device__ __forceinline__ int rint_small(float x) { return __float_as_int(fadd(x, kMagic)) - kMagicI; }

// unsigned bytes x signed bytes (Q4_1's nibbles are 0..15: `(x<<4)&0xF0` is 16*nibble as an UNSIGNED byte)
__device__ __forceinline__ int dp4a_us(uint32_t a, int b, int c) {
    int d; asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c)); return d;
}

// Q8_0 act-quant (ggml.c:1215-1252) of the 32 values held one per lane, written straight into the
// dp4a word layout the matmul consumers read: words [Q][w&3][bq][w>>2], scale [b] (x dscale).
// soff != 0: Q8_1 instead (quantize_row_q8_1, ggml.c:1426-1472): the scale is NOT rounded to fp16 and
// s = d * (sum of the quants) is stored soff floats behind the scale.
__device__ __forceinline__ void warp_quant_block(float v, int lane, int * aq_col, float * da_col, int b, float dscale, int soff = 0) {
    float amax = fabsf(v);
    #pragma unroll
    for (int o = 16; o > 0; o >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, o));
    const float dq = __fdiv_rn(amax, 127.f);
    const float d = soff ? dq : h2f(f2h(dq));
    const float id = amax != 0.f ? __fdiv_rn(127.f, amax) : 0.f;
    const int qv = rint_small(fmul(v, id));
    uint32_t pk = ((uint32_t)(qv & 0xFF)) << (8 * (lane & 3));
    pk |= __shfl_xor_sync(0xffffffffu, pk, 1);
    pk |= __shfl_xor_sync(0xffffffffu, pk, 2);
    if ((lane & 3) == 0) {
        const int w = lane >> 2;
        aq_col[(b >> 2) * 32 + (w & 3) * 8 + (b & 3) * 2 + (w >> 2)] = (int) pk;
    }
    if (lane == 0) da_col[b] = fmul(d, dscale);
    if (soff) {
        int qs = qv;
        #pragma unroll
        for (int o = 16; o > 0; o >>= 1) qs += __shfl_xor_sync(0xffffffffu, qs, o);
        if (lane == 0) da_col[soff + b] = fmul(d, (float) qs);
    }
}

// quantise one 32-float block held in registers by ONE thread into shared memory
// `rot`: v[4*w8 .. 4*w8+3] holds 16-byte chunk (w8 + rot) & 7 of the block (bank-conflict-free rotated smem reads)
// WT == Q4_1: Q8_1 (f32 scale, block sum s into sn[b]); otherwise Q8_0.
template <int WT>
__device__ __forceinline__ void thread_quant_block(const float (&v)[32], int * an, float * dn, int b, int rot = 0, float * sn = nullptr) {
    float m[8];
    #pragma unroll
    for (int j = 0; j < 8; j++) m[j] = fmaxf(fmaxf(fabsf(v[j]), fabsf(v[j + 8])), fmaxf(fabsf(v[j + 16]), fabsf(v[j + 24])));
    const float amax = fmaxf(fmaxf(fmaxf(m[0], m[1]), fmaxf(m[2], m[3])), fmaxf(fmaxf(m[4], m[5]), fmaxf(m[6], m[7])));
    const float dq = __fdiv_rn(amax, 127.f);
    const float d = (WT == kWT_Q4_1) ? dq : h2f(f2h(dq));
    const float id = amax != 0.f ? __fdiv_rn(127.f, amax) : 0.f;
    dn[b] = wt_nibbles(WT) ? fmul(d, 0.0625f) : d;          // the 1/16 of the nibble placement, folded (exact)
    int * dst = an + (b >> 2) * 32 + (b & 3) * 2;
    int qsum = 0;
    #pragma unroll
    for (int w = 0; w < 8; w++) {
        uint32_t pk = 0;
        #pragma unroll
        for (int j = 0; j < 4; j++) {
            const int qv = rint_small(fmul(v[w*4 + j], id));
            if (WT == kWT_Q4_1) qsum += qv;
            pk |= ((uint32_t)(qv & 0xFF)) << (8 * j);
        }
        const int ww = (w + rot) & 7;
        dst[(ww & 3) * 8 + (ww >> 2)] = (int) pk;
    }
    if (WT == kWT_Q4_1) sn[b] = fmul(d, (float) qsum);
}

template <int WT, int G, int NC, int PRO, int EPI, bool RING>
__global__ void __launch_bounds__(kConsumers + 32) k_gemv(const GemvArgs a) {
    constexpr int CB = chunk_bytes(WT);
    constexpr bool Q41 = WT == kWT_Q4_1;
    constexpr int TR = kWPC * G;
    extern __shared__ __align__(128) uint8_t smem[];
    const int nbq = a.W.nbq, K = a.W.K, nb = a.W.nb;
    const int NS = a.NS;
    constexpr int stage_bytes = kQS * TR * CB;
    // smem: [ring NS*stage][act words NC*nbq*128][act scales NC*nbq*16][Q4_1: act block sums NC*nbq*16][full 16][empty 16][act bar][red 4][gq NC*32]
    uint8_t * ring = smem;
    int * a_s = (int *)(smem + (RING ? (size_t) NS * stage_bytes : 0));
    float * da_s = (float *)((uint8_t *) a_s + (size_t) NC * nbq * 128);
    float * sa_s = da_s + (size_t) NC * nbq * 4;                         // Q4_1 only
    uint64_t * full = (uint64_t *)((uint8_t *) da_s + (size_t) NC * nbq * (Q41 ? 32 : 16));
    uint64_t * empty = full + 16;
    uint64_t * actbar = empty + 16;
    double * red = (double *)(actbar + 2);           // [kWPC]
    float * gq = (float *)(red + kWPC);              // [NC][32] gate values of one tile (EPI_GATEQ)
    float * xs = gq + NC * 32;                       // [K] input row staged by one bulk copy (PRO_NORM, NC == 1)

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int col0 = blockIdx.y * NC;
    const int n_stage = nbq / kQS;

    if (tid == 0) {
        B200_TRACE(a.trace, 0);
        if (RING) for (int s = 0; s < NS; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], kWPC); }
        mbar_init(actbar, 1);
        mbar_init(actbar + 1, kWPC);        // gate: consumers have issued their prologue loads
        mbar_fence_init();
    }
    __syncthreads();

    if (RING && warp == kWPC) {
        // ------------------------------------------------------------------ producer warp
        if (lane == 0) {
            int slot = 0, use = 0, issued = 0;
            for (int tile = blockIdx.x; tile < a.W.n_tiles; tile += gridDim.x) {
                const uint8_t * src = a.W.data + (long long) tile * a.W.tile_bytes;
                for (int s = 0; s < n_stage; s++) {
                    // Only `pre_stages` of weights may be requested before the consumers have put their (tiny, latency-
                    // critical) prologue loads on the wire: a prologue load queued behind ~20 MB of bulk-copy requests
                    // waits ~5 us (profiles/r01_timeline_*.txt); behind 2 stages per CTA it waits < 1 us.
                    if (issued == a.pre_stages) mbar_wait(actbar + 1, 0);
                    issued++;
                    if (use > 0) mbar_wait(&empty[slot], (use - 1) & 1);
                    mbar_arrive_expect_tx(&full[slot], (uint32_t) stage_bytes);
                    bulk_g2s(ring + (size_t) slot * stage_bytes, src + (size_t) s * stage_bytes, (uint32_t) stage_bytes, &full[slot]);
                    if (++slot == NS) { slot = 0; use++; }
                }
            }
            // This CTA has requested its last weight byte: let the NEXT kernel's CTAs become resident and
            // start THEIR weight stream now, so HBM never idles across the kernel boundary (depth-1 hand-off).
            // ORDERING GUARANTEE other kernels rely on (k_attn128's pre-wait KV prefetch): the trigger is never
            // fired before this CTA's consumers have returned from griddepcontrol.wait (the gate below), i.e. not
            // before the kernel BEFORE this one has completed.  By induction, whatever runs ahead of its own wait
            // in the next kernel sees every kernel up to this one's predecessor finished.
            if (issued <= a.pre_stages) mbar_wait(actbar + 1, 0);
            grid_dep_launch();
            B200_TRACE(a.trace, 4);
        }
        return;
    }

    // ---------------------------------------------------------------------- consumer warps
    // static data first: the norm weights do not depend on the previous kernel, so their (possibly HBM) round trip
    // is issued before the dependency wait and kept in L2 for the next token
    float wn[32];
    if (PRO == PRO_NORM && nb <= kConsumers) {
        #pragma unroll
        for (int j = 0; j < 8; j++) {
            const float4 u = tid < nb ? ldg_keep(a.norm_w + tid * 32 + (((NC == 1 ? tid : 0) + j) & 7) * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
            wn[j*4] = u.x; wn[j*4+1] = u.y; wn[j*4+2] = u.z; wn[j*4+3] = u.w;
        }
    }
    grid_dep_wait();                                   // the input comes from the previous kernel
    if (!RING && tid == 0) grid_dep_launch();          // (after the wait: same ordering guarantee as the ring producer)
    if (tid == 0) B200_TRACE(a.trace, 1);

    const int ncols = min(NC, a.N - col0);
    bool gate_done = false;
    if (PRO == PRO_PREQ) {
        gate_done = true;
        // the producer of the activation already quantised it (attention / gate epilogue): two bulk copies
        if (tid == 0) {
            const uint32_t b1 = (uint32_t) ncols * nbq * 128, b2 = (uint32_t) ncols * nbq * 16;
            mbar_arrive_expect_tx(actbar, b1 + b2 + (Q41 ? b2 : 0u));
            bulk_g2s(a_s, a.aq_in + (size_t) col0 * nbq * 32, b1, actbar);
            bulk_g2s(da_s, a.da_in + (size_t) col0 * nbq * 4, b2, actbar);
            if (Q41) bulk_g2s(sa_s, a.da_in + a.in_soff + (size_t) col0 * nbq * 4, b2, actbar);
        }
        if (RING && lane == 0) mbar_arrive(actbar + 1);
        for (int n = ncols; n < NC; n++) {
            for (int i = tid; i < nbq * 32; i += kConsumers) a_s[(size_t) n * nbq * 32 + i] = 0;
            for (int i = tid; i < nbq * 4; i += kConsumers) { da_s[(size_t) n * nbq * 4 + i] = 0.f; if (Q41) sa_s[(size_t) n * nbq * 4 + i] = 0.f; }
        }
        mbar_wait(actbar, 0);
    } else {
        for (int n = 0; n < NC; n++) {
            int * an = a_s + (size_t) n * nbq * 32;
            float * dn = da_s + (size_t) n * nbq * 4;
            float * sn = sa_s + (size_t) n * nbq * 4;
            if (n >= ncols) {                              // padded column: zeros
                for (int i = tid; i < nbq * 32; i += kConsumers) an[i] = 0;
                for (int i = tid; i < nbq * 4; i += kConsumers) { dn[i] = 0.f; if (Q41) sn[i] = 0.f; }
                continue;
            }
            const float * x = a.x + (size_t)(col0 + n) * a.ldx;
            for (int b = nb + tid; b < nbq * 4; b += kConsumers) {       // padding blocks
                int * dst = an + (b >> 2) * 32 + (b & 3) * 2;
                for (int w = 0; w < 4; w++) { dst[w * 8] = 0; dst[w * 8 + 1] = 0; }
                dn[b] = 0.f;
                if (Q41) sn[b] = 0.f;
            }
            if (PRO == PRO_NORM && nb <= kConsumers) {
                // one global round trip: x block and norm weights in flight together, x kept in registers
                float v[32];
                const bool own = tid < nb;
                const int rot = NC == 1 ? (tid & 7) : 0;
                if (NC == 1) {
                    // one TMA bulk copy of the row instead of 1024 LDG.128 per CTA: under a saturated memory system the
                    // LDGs took ~2.9 us (in-kernel timeline), the bulk copy of a same-sized activation ~0.5 us.  Each
                    // thread then reads its block with 16-byte chunks rotated by its lane so the quarter-warps never
                    // collide on a bank; chunk (j + rot) & 7 lands in v[4j..4j+3].
                    if (tid == 0) { mbar_arrive_expect_tx(actbar, (uint32_t) K * 4); bulk_g2s(xs, x, (uint32_t) K * 4, actbar); }
                    if (RING && lane == 0) { gate_done = true; mbar_arrive(actbar + 1); }
                    mbar_wait(actbar, 0);
                    #pragma unroll
                    for (int j = 0; j < 8; j++) {
                        const float4 t = own ? *(const float4 *)(xs + tid * 32 + ((j + rot) & 7) * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
                        v[j*4] = t.x; v[j*4+1] = t.y; v[j*4+2] = t.z; v[j*4+3] = t.w;
                    }
                } else {
                    #pragma unroll
                    for (int j = 0; j < 8; j++) {
                        const float4 t = own ? *(const float4 *)(x + tid * 32 + j * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
                        v[j*4] = t.x; v[j*4+1] = t.y; v[j*4+2] = t.z; v[j*4+3] = t.w;
                    }
                    if (RING && n == ncols - 1 && lane == 0) { gate_done = true; mbar_arrive(actbar + 1); }
                }
                double s4[4] = {0.0, 0.0, 0.0, 0.0};
                #pragma unroll
                for (int j = 0; j < 32; j++) s4[j & 3] += widen_nonneg(fmul(v[j], v[j]));
                double s = (s4[0] + s4[1]) + (s4[2] + s4[3]);
                if (tid == 0) B200_TRACE(a.trace, 5);
                for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
                if (lane == 0) red[warp] = s;
                named_bar_sync(1, kConsumers);
                const double tot = (red[0] + red[1]) + (red[2] + red[3]);
                named_bar_sync(1, kConsumers);
                const float scale = __fdiv_rn(1.0f, __fsqrt_rn(fadd((float)(tot / (double) K), 1e-6f)));
                if (tid == 0) B200_TRACE(a.trace, 6);
                if (own) {
                    #pragma unroll
                    for (int j = 0; j < 32; j++) v[j] = fmul(fmul(v[j], scale), wn[j]);
                    thread_quant_block<WT>(v, an, dn, tid, rot, sn);
                }
            } else {
                float scale = 1.0f;
                if (PRO == PRO_NORM) {
                    double s = 0.0;
                    for (int i = tid * 4; i < K; i += kConsumers * 4) {
                        const float4 v = *(const float4 *)(x + i);
                        s += (double) fmul(v.x, v.x); s += (double) fmul(v.y, v.y);
                        s += (double) fmul(v.z, v.z); s += (double) fmul(v.w, v.w);
                    }
                    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
                    if (lane == 0) red[warp] = s;
                    named_bar_sync(1, kConsumers);
                    const double tot = (red[0] + red[1]) + (red[2] + red[3]);
                    named_bar_sync(1, kConsumers);
                    scale = __fdiv_rn(1.0f, __fsqrt_rn(fadd((float)(tot / (double) K), 1e-6f)));
                }
                for (int b = tid; b < nb; b += kConsumers) {
                    float v[32];
                    #pragma unroll
                    for (int j = 0; j < 8; j++) {
                        float4 t = *(const float4 *)(x + b * 32 + j * 4);
                        if (PRO == PRO_NORM) {
                            const float4 wv = *(const float4 *)(a.norm_w + b * 32 + j * 4);
                            t.x = fmul(fmul(t.x, scale), wv.x); t.y = fmul(fmul(t.y, scale), wv.y);
                            t.z = fmul(fmul(t.z, scale), wv.z); t.w = fmul(fmul(t.w, scale), wv.w);
                        }
                        v[j*4] = t.x; v[j*4+1] = t.y; v[j*4+2] = t.z; v[j*4+3] = t.w;
                    }
                    thread_quant_block<WT>(v, an, dn, b, 0, sn);
                }
            }
        }
    }
    if (RING && lane == 0 && !gate_done) mbar_arrive(actbar + 1);     // slow-path prologues open the gate late
    named_bar_sync(1, kConsumers);
    if (tid == 0) B200_TRACE(a.trace, 2);

    const int r = lane >> 2, w = lane & 3;
    int slot = 0, phase = 0;
#ifdef B200_TRACE_WAITS                                                // special build (costs ~5 % of the step even when idle)
    long long dbg_wait = 0, dbg_t0 = a.trace ? clock64() : 0;      // B200_TRACE: cycles warp 0 waits for weight stages
#endif
    uint2 * send_slot = nullptr; int send_seq = 0;
    if (EPI == EPI_RESID_SEND) {
        // last matmul of a pipelined slice (N = 1): every output row also goes, as {value, seq}, into the next rank's inbox
        // slot the moment it is computed -- no fence, no flag, no extra kernel.  seq_out is advanced by k_advance_pp.
        send_seq = a.mb_mine->seq_out + 1;
        if (lane == 0) mb_wait_slot_free(a.mb_mine, send_seq);
        __syncwarp();
        send_slot = a.mb_peer_inbox + (size_t)(send_seq & (kMbSlots - 1)) * a.mb_slot_elems;
    }
    for (int tile = blockIdx.x; tile < a.W.n_tiles; tile += gridDim.x) {
        float acc[G][NC][2];
        float summ[G][NC];                  // Q4_1: the scalar chain summs += m * s of row r (every w-thread of the row keeps a copy)
        #pragma unroll
        for (int g = 0; g < G; g++)
            #pragma unroll
            for (int n = 0; n < NC; n++) { acc[g][n][0] = 0.f; acc[g][n][1] = 0.f; summ[g][n] = 0.f; }
        const uint8_t * gsrc = a.W.data + (long long) tile * a.W.tile_bytes;

        for (int s = 0; s < n_stage; s++) {
            const uint8_t * base;
            if (RING) {
#ifdef B200_TRACE_WAITS
                if (a.trace) { const long long c0 = clock64(); mbar_wait(&full[slot], phase); dbg_wait += clock64() - c0; }
                else
#endif
                mbar_wait(&full[slot], phase);
                base = ring + (size_t) slot * stage_bytes;
            } else {
                base = gsrc + (size_t) s * stage_bytes;
            }
            base += (size_t)(warp * G) * CB;
            if (!a.dbg_nomath)
            #pragma unroll
            for (int qi = 0; qi < kQS; qi++) {
                const int Q = s * kQS + qi;
                uint4 wv[G], wv2[G]; uint2 sc[G], mc[G];
                #pragma unroll
                for (int g = 0; g < G; g++) {
                    const uint8_t * ch = base + (size_t)(qi * TR + g) * CB;
                    wv[g] = *(const uint4 *)(ch + lane * 16);
                    if (WT == kWT_Q8_0) { wv2[g] = *(const uint4 *)(ch + 512 + lane * 16); sc[g] = *(const uint2 *)(ch + 1024 + r * 8); }
                    else sc[g] = *(const uint2 *)(ch + 512 + r * 8);
                    mc[g] = Q41 ? *(const uint2 *)(ch + 576 + r * 8) : make_uint2(0u, 0u);
                }
                #pragma unroll
                for (int n = 0; n < NC; n++) {
                    const int4 * ap = (const int4 *)(a_s + (size_t) n * nbq * 32 + Q * 32 + w * 8);
                    const int4 a01 = ap[0], a23 = ap[1];           // {lo0,hi0,lo1,hi1}, {lo2,hi2,lo3,hi3}
                    const float4 dav = *(const float4 *)(da_s + (size_t) n * nbq * 4 + Q * 4);
                    const int alo[4] = {a01.x, a01.z, a23.x, a23.z};
                    const int ahi[4] = {a01.y, a01.w, a23.y, a23.w};
                    const float da[4] = {dav.x, dav.y, dav.z, dav.w};
                    float sa[4] = {0.f, 0.f, 0.f, 0.f};
                    if (Q41) { const float4 sav = *(const float4 *)(sa_s + (size_t) n * nbq * 4 + Q * 4); sa[0] = sav.x; sa[1] = sav.y; sa[2] = sav.z; sa[3] = sav.w; }
                    #pragma unroll
                    for (int g = 0; g < G; g++) {
                        const uint32_t ww[4] = {wv[g].x, wv[g].y, wv[g].z, wv[g].w};
                        const uint32_t ww2[4] = {wv2[g].x, wv2[g].y, wv2[g].z, wv2[g].w};
                        const uint32_t sw[2] = {sc[g].x, sc[g].y};
                        const uint32_t mw[2] = {mc[g].x, mc[g].y};
                        #pragma unroll
                        for (int bq = 0; bq < 4; bq++) {
                            const uint16_t dh = (uint16_t)(sw[bq >> 1] >> (16 * (bq & 1)));
                            const float D = fmul(h2f(dh), da[bq]);
                            float f0, f1;
                            if (Q41) {
                                // summs += fp16->f32(m) * s first (ggml.c:2712), then the lane fma: two independent chains
                                const uint16_t mh = (uint16_t)(mw[bq >> 1] >> (16 * (bq & 1)));
                                summ[g][n] = fadd(summ[g][n], fmul(h2f(mh), sa[bq]));
                                const uint32_t lo = (ww[bq] << 4) & 0xF0F0F0F0u, hi = ww[bq] & 0xF0F0F0F0u;
                                f0 = fadd(__int_as_float(dp4a_us(lo, alo[bq], kMagicI)), -kMagic);
                                f1 = fadd(__int_as_float(dp4a_us(hi, ahi[bq], kMagicI)), -kMagic);
                            } else {
                                int lo, hi;
                                if (WT == kWT_Q4_0) { lo = (int)((ww[bq] << 4) & 0xF0F0F0F0u); hi = (int)(ww[bq] & 0xF0F0F0F0u); }
                                else                { lo = (int) ww[bq]; hi = (int) ww2[bq]; }
                                f0 = fadd(__int_as_float(__dp4a(lo, alo[bq], kMagicI)), -kMagic);
                                f1 = fadd(__int_as_float(__dp4a(hi, ahi[bq], kMagicI)), -kMagic);
                            }
                            acc[g][n][0] = ffma(D, f0, acc[g][n][0]);
                            acc[g][n][1] = ffma(D, f1, acc[g][n][1]);
                        }
                    }
                }
            }
            if (RING) {
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty[slot]);
                if (++slot == NS) { slot = 0; phase ^= 1; }
            }
        }

        // epilogue: hsum_float_8 order ((a0+a4)+(a2+a6)) + ((a1+a5)+(a3+a7))
        float res[G][NC];
        #pragma unroll
        for (int g = 0; g < G; g++)
            #pragma unroll
            for (int n = 0; n < NC; n++) {
                float t = fadd(acc[g][n][0], acc[g][n][1]);
                t = fadd(t, __shfl_xor_sync(0xffffffffu, t, 2));
                t = fadd(t, __shfl_xor_sync(0xffffffffu, t, 1));
                res[g][n] = Q41 ? fadd(t, summ[g][n]) : t;          // hsum_float_8(acc) + summs
            }
        if (EPI == EPI_GATE || EPI == EPI_GATEQ) {
            const int row = (tile * kWPC + warp) * 8 + r;
            if (w == 0) {
                #pragma unroll
                for (int n = 0; n < NC; n++) {
                    const float gv = fmul(h2f(a.tsilu[f2h(res[0][n])]), res[G - 1][n]);
                    if (EPI == EPI_GATEQ) gq[n * 32 + warp * 8 + r] = row < a.out_rows ? gv : 0.f;
                    else if (row < a.out_rows && n < ncols) a.y[(size_t)(col0 + n) * a.ldy + row] = gv;
                }
            }
            if (EPI == EPI_GATEQ) {
                // the tile's 32 gate rows are exactly one Q8_0 block of w2's input: quantise it here
                named_bar_sync(1, kConsumers);
                for (int n = warp; n < ncols; n += kWPC)
                    warp_quant_block(gq[n * 32 + lane], lane, a.aq_out + (size_t)(col0 + n) * a.out_nbq * 32,
                                     a.da_out + (size_t)(col0 + n) * a.out_nbq * 4, tile, a.out_dscale, a.out_soff);
                named_bar_sync(1, kConsumers);
            }
        } else if (w == 0) {
            #pragma unroll
            for (int g = 0; g < G; g++) {
                const int row = ((tile * kWPC + warp) * G + g) * 8 + r;
                if (row < a.out_rows) {
                    #pragma unroll
                    for (int n = 0; n < NC; n++) {
                        if (n < ncols) {
                            float v = res[g][n];
                            if (EPI == EPI_RESID || EPI == EPI_RESID_NQ || EPI == EPI_RESID_SEND) v = fadd(v, a.resid[(size_t)(col0 + n) * a.ldr + row]);
                            a.y[(size_t)(col0 + n) * a.ldy + row] = v;
                            if (EPI == EPI_RESID_SEND) st_ll(send_slot + row, v, send_seq);   // {value, seq} straight into the next rank's inbox (NVLink)
                            if (EPI == EPI_RESID_NQ) gq[n * 32 + warp * 8 + r] = v;
                        }
                    }
                }
            }
        }
    }
    if (EPI == EPI_RESID_NQ) {
        // The output row feeds an RMSNorm + weight matmul next.  Instead of every CTA of that matmul re-reading and
        // re-normalising the whole row (16 KB of LDGs that queue behind its own weight stream: ~3 us per kernel, and
        // 20 % extra L2 traffic), THIS kernel finishes the job while the values are still on chip:
        //   every CTA owns exactly one 32-row tile = one Q8_0 block (the host guarantees gridDim.x == n_tiles);
        //   1. partial sum of squares of its block -> global;  2. grid-wide arrive + spin on a counter;
        //   3. every CTA adds the n_tiles partials in the same fixed order -> identical RMS scale everywhere;
        //   4. normalise, multiply by the norm weight, Q8_0-quantise its own block into the consumer's word layout.
        // All CTAs are co-resident (grid <= SM count x CTAs/SM, and dependents are launched only after every CTA of
        // this grid has started), so the spin cannot deadlock.
        named_bar_sync(1, kConsumers);
        if (warp == 0) {
            const int tile = blockIdx.x, nt = (int) gridDim.x;
            for (int n = 0; n < ncols; n++) {
                const float val = gq[n * 32 + lane];
                double s = widen_nonneg(fmul(val, val));
                for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
                double * part = a.nq_partial + ((size_t) blockIdx.y * NC + n) * nt;
                if (lane == 0) part[tile] = s;
            }
            int * cnt = a.nq_counter + 2 * blockIdx.y;
            if (lane == 0) {
                __threadfence();
                atomicAdd(cnt, 1);
                while (*(volatile int *) cnt < nt) { }
                __threadfence();
            }
            __syncwarp();
            const int row = tile * 32 + lane;
            for (int n = 0; n < ncols; n++) {
                const double * part = a.nq_partial + ((size_t) blockIdx.y * NC + n) * nt;
                double s = 0.0;
                for (int i = lane; i < nt; i += 32) s += __ldcg(part + i);
                for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
                const float scale = __fdiv_rn(1.0f, __fsqrt_rn(fadd((float)(s / (double) a.out_rows), 1e-6f)));
                const float val = gq[n * 32 + lane];
                const float wv = row < a.out_rows ? a.nq_norm_w[row] : 0.f;
                warp_quant_block(fmul(fmul(val, scale), wv), lane, a.aq_out + (size_t)(col0 + n) * a.out_nbq * 32,
                                 a.da_out + (size_t)(col0 + n) * a.out_nbq * 4, tile, a.out_dscale, a.out_soff);
            }
            if (lane == 0) {                                   // the last CTA through re-arms the counters
                if (atomicAdd(cnt + 1, 1) == nt - 1) { cnt[0] = 0; cnt[1] = 0; }
            }
        }
    }
    if (tid == 0) B200_TRACE(a.trace, 3);
#ifdef B200_TRACE_WAITS
    if (tid == 0 && a.trace)                           // slot 7: (cycles spent waiting for weight stages) << 32 | main-loop cycles
        a.trace[((size_t) blockIdx.y * gridDim.x + blockIdx.x) * 8 + 7] = ((unsigned long long) dbg_wait << 32) | (unsigned long long)((clock64() - dbg_t0) & 0xFFFFFFFFll);
#endif
}

// =============================================================================================
// K1n: the NARROW matrices of a single-token step (wo, w2: 128 tiles of 32 rows for 7B = at most one CTA per SM).
// With k_gemv's mapping (4 threads per row) such a CTA is 4 consumer warps = ONE warp per scheduler, and a lone warp
// cannot hide its own latencies: measured IPC 0.39, ~19 cycles per block step, wo 2.6 us / w2 6.1 us of main loop for
// 9.4 / 25.4 MB (1.5 / 3.9 us at the HBM rate).  The parallelism exact mode allows is rows x 8 AVX lanes (each lane's fma
// chain is sequential in K), so this variant spends ALL of it: 8 threads per row, thread (r, l) owns AVX lane l alone.
//   * 8 consumer warps per CTA, warp = 4 rows x 8 lanes, same 32-row tile, same packed layout, same TMA ring;
//   * per block and thread: one shift+mask (lanes 0..3 take the low nibbles of word l, lanes 4..7 the high nibbles of
//     word l-4), one dp4a, the magic-number int->float, one fma -- 8 instead of 15 instructions on the warp's critical path;
//   * the scale product D = d_w * d_a is now computed by 8 threads instead of 4 (+27 % instructions in total), which is
//     why the wide matrices (qkv, w1|w3: >= 2.3 warps per scheduler already) keep k_gemv.
// Pre-quantised input only (PRO_PREQ: the attention / gate epilogue already produced Q8_0), one column, epilogues
// + residual and + residual + send (EPI_RESID, EPI_RESID_SEND).  Arithmetic per lane chain is k_gemv's, operand for operand.
// MEASURED (7B Q4_0, 64 steps, same box): 806 tok/s with this kernel against 823 with k_gemv -- twice the warps and half the
// instructions per warp did NOT shorten wo / w2, so their main loops are not bound by the lone warp's issue rate after all;
// opt-in (B200_N8=1), bit-exact (tests/test_gpu_parity.py::test_narrow_matrix_kernel_is_a_scheduling_choice).
// =============================================================================================
constexpr int kN8Warps = 8;
constexpr int kN8Consumers = kN8Warps * 32;

template <int WT, int EPI>
__global__ void __launch_bounds__(kN8Consumers + 32) k_gemv_n8(const GemvArgs a) {
    static_assert(WT == kWT_Q4_0 || WT == kWT_Q8_0, "narrow variant: Q4_0 / Q8_0");
    constexpr int CB = chunk_bytes(WT);
    constexpr int TR = 4;                                   // row-groups of 8 rows per tile (= k_gemv with G = 1)
    constexpr int stage_bytes = kQS * TR * CB;
    extern __shared__ __align__(128) uint8_t smem[];
    const int nbq = a.W.nbq, NS = a.NS;
    // smem: [ring NS*stage][act words nbq*128][act scales nbq*16][full 16][empty 16][act bar 2]
    uint8_t * ring = smem;
    int * a_s = (int *)(smem + (size_t) NS * stage_bytes);
    float * da_s = (float *)((uint8_t *) a_s + (size_t) nbq * 128);
    uint64_t * full = (uint64_t *)((uint8_t *) da_s + (size_t) nbq * 16);
    uint64_t * empty = full + 16;
    uint64_t * actbar = empty + 16;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n_stage = nbq / kQS;

    if (tid == 0) {
        B200_TRACE(a.trace, 0);
        for (int s = 0; s < NS; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], kN8Warps); }
        mbar_init(actbar, 1);
        mbar_init(actbar + 1, kN8Warps);
        mbar_fence_init();
    }
    __syncthreads();

    if (warp == kN8Warps) {
        // producer warp: k_gemv's, including the gate on the consumers' prologue copies and the late dependent trigger
        if (lane == 0) {
            int slot = 0, use = 0, issued = 0;
            for (int tile = blockIdx.x; tile < a.W.n_tiles; tile += gridDim.x) {
                const uint8_t * src = a.W.data + (long long) tile * a.W.tile_bytes;
                for (int s = 0; s < n_stage; s++) {
                    if (issued == a.pre_stages) mbar_wait(actbar + 1, 0);
                    issued++;
                    if (use > 0) mbar_wait(&empty[slot], (use - 1) & 1);
                    mbar_arrive_expect_tx(&full[slot], (uint32_t) stage_bytes);
                    bulk_g2s(ring + (size_t) slot * stage_bytes, src + (size_t) s * stage_bytes, (uint32_t) stage_bytes, &full[slot]);
                    if (++slot == NS) { slot = 0; use++; }
                }
            }
            if (issued <= a.pre_stages) mbar_wait(actbar + 1, 0);
            grid_dep_launch();
            B200_TRACE(a.trace, 4);
        }
        return;
    }

    grid_dep_wait();                                        // the quantised activation comes from the previous kernel
    if (tid == 0) {
        B200_TRACE(a.trace, 1);
        const uint32_t b1 = (uint32_t) nbq * 128, b2 = (uint32_t) nbq * 16;
        mbar_arrive_expect_tx(actbar, b1 + b2);
        bulk_g2s(a_s, a.aq_in, b1, actbar);
        bulk_g2s(da_s, a.da_in, b2, actbar);
    }
    if (lane == 0) mbar_arrive(actbar + 1);
    mbar_wait(actbar, 0);
    if (tid == 0) B200_TRACE(a.trace, 2);

    const int rg = warp >> 1;                               // row-group of the tile
    const int r = (warp & 1) * 4 + (lane >> 3), l = lane & 7;   // row in the group, AVX lane
    const int sh = (WT == kWT_Q4_0 && l < 4) ? 4 : 0;
    const uint32_t w_off = (uint32_t)((WT == kWT_Q8_0 ? (l >> 2) * 512 : 0) + (4 * r + (l & 3)) * 16);
    const uint32_t s_off = (uint32_t)((WT == kWT_Q8_0 ? 1024 : 512) + r * 8);
    const int * a_l = a_s + (l & 3) * 8 + (l >> 2);         // words [Q][l&3][bq][l>>2]
    uint2 * send_slot = nullptr; int send_seq = 0;
    if (EPI == EPI_RESID_SEND) {
        send_seq = a.mb_mine->seq_out + 1;
        if (lane == 0) mb_wait_slot_free(a.mb_mine, send_seq);
        __syncwarp();
        send_slot = a.mb_peer_inbox + (size_t)(send_seq & (kMbSlots - 1)) * a.mb_slot_elems;
    }
    int slot = 0, phase = 0;
#ifdef B200_TRACE_WAITS
    long long dbg_wait = 0, dbg_t0 = a.trace ? clock64() : 0;
#endif
    for (int tile = blockIdx.x; tile < a.W.n_tiles; tile += gridDim.x) {
        float acc = 0.f;
        for (int s = 0; s < n_stage; s++) {
#ifdef B200_TRACE_WAITS
            if (a.trace) { const long long c0 = clock64(); mbar_wait(&full[slot], phase); dbg_wait += clock64() - c0; }
            else
#endif
            mbar_wait(&full[slot], phase);
            const uint8_t * base = ring + (size_t) slot * stage_bytes + (size_t) rg * CB;
            if (!a.dbg_nomath)
            #pragma unroll
            for (int qi = 0; qi < kQS; qi++) {
                const int Q = s * kQS + qi;
                const uint8_t * ch = base + (size_t) qi * TR * CB;
                const uint4 wv = *(const uint4 *)(ch + w_off);
                const uint2 sc = *(const uint2 *)(ch + s_off);
                const float4 dav = *(const float4 *)(da_s + Q * 4);
                const int av[4] = {a_l[Q * 32], a_l[Q * 32 + 2], a_l[Q * 32 + 4], a_l[Q * 32 + 6]};
                const uint32_t ww[4] = {wv.x, wv.y, wv.z, wv.w};
                const uint32_t sw[2] = {sc.x, sc.y};
                const float da[4] = {dav.x, dav.y, dav.z, dav.w};
                #pragma unroll
                for (int bq = 0; bq < 4; bq++) {
                    const uint16_t dh = (uint16_t)(sw[bq >> 1] >> (16 * (bq & 1)));
                    const float D = fmul(h2f(dh), da[bq]);
                    const int v = WT == kWT_Q4_0 ? (int)((ww[bq] << sh) & 0xF0F0F0F0u) : (int) ww[bq];
                    const float f = fadd(__int_as_float(__dp4a(v, av[bq], kMagicI)), -kMagic);
                    acc = ffma(D, f, acc);
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[slot]);
            if (++slot == NS) { slot = 0; phase ^= 1; }
        }
        // hsum_float_8: (a_l + a_l+4), then + lane^2, then + lane^1
        float t = fadd(acc, __shfl_xor_sync(0xffffffffu, acc, 4));
        t = fadd(t, __shfl_xor_sync(0xffffffffu, t, 2));
        t = fadd(t, __shfl_xor_sync(0xffffffffu, t, 1));
        const int row = (tile * TR + rg) * 8 + r;
        if (l == 0 && row < a.out_rows) {
            const float v = fadd(t, a.resid[row]);
            a.y[row] = v;
            if (EPI == EPI_RESID_SEND) st_ll(send_slot + row, v, send_seq);
        }
    }
    if (tid == 0) B200_TRACE(a.trace, 3);
#ifdef B200_TRACE_WAITS
    if (tid == 0 && a.trace)
        a.trace[(size_t) blockIdx.x * 8 + 7] = ((unsigned long long) dbg_wait << 32) | (unsigned long long)((clock64() - dbg_t0) & 0xFFFFFFFFll);
#endif
}

// =============================================================================================
// K3: RMSNorm * weight -> Q8_0 act-quant of whole rows, once per token, for MULTI-token calls (prefill chunks, batched
// steps).  With several columns per CTA the fused PRO_NORM prologue would repeat this for every 32-row tile (480x for
// qkv) behind one dependent global round trip per column; here it is done once and the matmul CTAs fetch the quantised
// columns with a bulk copy (PRO_PREQ).  Same per-block arithmetic as the fused prologue (thread_quant_block).
// Single-token steps keep the fused prologue: there the extra launch would cost more than the redundancy.
// =============================================================================================
struct NormQuantArgs {
    const float * x; int ldx; const float * norm_w; int K;
    int * aq; float * da; int nbq;            // [N][nbq*32] words, [N][nbq*4] scales (x 1/16 for Q4_0 / Q4_1 weights)
    int soff;                                 // Q4_1: block sums s at da + soff
};

template <int WT>
__global__ void __launch_bounds__(256) k_norm_quant(const NormQuantArgs a) {
    __shared__ double red[8];
    const int n = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nb = a.K / 32;
    if (tid == 0) grid_dep_launch();
    grid_dep_wait();
    const float * x = a.x + (size_t) n * a.ldx;
    double s = 0.0;
    for (int b = tid; b < nb; b += 256) {
        #pragma unroll
        for (int j = 0; j < 8; j++) {
            const float4 t = *(const float4 *)(x + b * 32 + j * 4);
            s += widen_nonneg(fmul(t.x, t.x)); s += widen_nonneg(fmul(t.y, t.y));
            s += widen_nonneg(fmul(t.z, t.z)); s += widen_nonneg(fmul(t.w, t.w));
        }
    }
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) red[warp] = s;
    __syncthreads();
    double tot = 0.0;
    #pragma unroll
    for (int i = 0; i < 8; i++) tot += red[i];
    const float scale = __fdiv_rn(1.0f, __fsqrt_rn(fadd((float)(tot / (double) a.K), 1e-6f)));
    int * an = a.aq + (size_t) n * a.nbq * 32;
    float * dn = a.da + (size_t) n * a.nbq * 4;
    for (int b = tid; b < nb; b += 256) {
        float v[32];
        #pragma unroll
        for (int j = 0; j < 8; j++) {
            const float4 t = *(const float4 *)(x + b * 32 + j * 4);
            const float4 wv = *(const float4 *)(a.norm_w + b * 32 + j * 4);
            v[j*4]   = fmul(fmul(t.x, scale), wv.x); v[j*4+1] = fmul(fmul(t.y, scale), wv.y);
            v[j*4+2] = fmul(fmul(t.z, scale), wv.z); v[j*4+3] = fmul(fmul(t.w, scale), wv.w);
        }
        thread_quant_block<WT>(v, an, dn, b, 0, dn + a.soff);
    }
}

// =============================================================================================
// K1f: F16-weight matmul, exact mode: ggml_vec_dot_f16 (32 f32 slots, chunks of 32 in order,
// fixed reduce tree, n%32 tail in double).  One warp per output row, lane = slot; weights are
// re-laid at load as [row][c8 = chunk/8][lane][8 chunks] so each lane issues one 16 B load per
// 8 chunks.  The activation row is rounded to fp16 (ggml_fp32_to_fp16_row, ggml.c:495-512).
// =============================================================================================
struct GemvF16Args {
    const uint16_t * W;   // packed [rows][nc8][32][8]  (+ tail [rows][K%32] after, see tail)
    const uint16_t * tail;
    int rows, K;
    const float * x; int ldx; const float * norm_w;
    const float * resid; int ldr;
    float * y; int ldy; int N;
    const uint16_t * tsilu;
    const uint16_t * W2; const uint16_t * tail2;   // EPI_GATE: second matrix (w3)
};

template <int PRO, int EPI>
__global__ void __launch_bounds__(256) k_gemv_f16(const GemvF16Args a) {
    extern __shared__ __align__(16) uint8_t smem[];
    uint16_t * xh = (uint16_t *) smem;               // [K] fp16 activation
    __shared__ double red[8];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, K = a.K;
    const int col = blockIdx.y;
    grid_dep_wait();
    const float * x = a.x + (size_t) col * a.ldx;
    float scale = 1.0f;
    if (PRO == PRO_NORM) {
        double s = 0.0;
        for (int i = tid; i < K; i += 256) s += (double) fmul(x[i], x[i]);
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) red[warp] = s;
        __syncthreads();
        double tot = 0.0;
        for (int i = 0; i < 8; i++) tot += red[i];
        scale = __fdiv_rn(1.0f, __fsqrt_rn(fadd((float)(tot / (double) K), 1e-6f)));
    }
    for (int i = tid; i < K; i += 256) {
        float v = x[i];
        if (PRO == PRO_NORM) v = fmul(fmul(v, scale), a.norm_w[i]);
        xh[i] = f2h(v);
    }
    __syncthreads();
    const int nchunk = K / 32, nc8 = (nchunk + 7) / 8, ntail = K & 31;
    for (int row = blockIdx.x * 8 + warp; row < a.rows; row += gridDim.x * 8) {
        float res[2] = {0.f, 0.f};
        #pragma unroll
        for (int m = 0; m < (EPI == EPI_GATE ? 2 : 1); m++) {
            const uint16_t * Wm = m ? a.W2 : a.W;
            const uint16_t * tl = m ? a.tail2 : a.tail;
            float acc = 0.f;
            const uint4 * wp = (const uint4 *)(Wm + ((size_t) row * nc8 * 32 + lane) * 8);
            // 4 x 16 B per lane in flight (2 KB per warp): the FMA chain stays in chunk order, the loads run ahead
            constexpr int U = 4;
            for (int c8 = 0; c8 < nc8; c8 += U) {
                uint4 v[U];
                #pragma unroll
                for (int q = 0; q < U; q++) v[q] = c8 + q < nc8 ? __ldcs(wp + (size_t)(c8 + q) * 32) : make_uint4(0, 0, 0, 0);
                #pragma unroll
                for (int q = 0; q < U; q++) {
                    const uint32_t u[4] = {v[q].x, v[q].y, v[q].z, v[q].w};
                    #pragma unroll
                    for (int j = 0; j < 8; j++) {
                        const int c = (c8 + q) * 8 + j;
                        if (c < nchunk) {
                            const uint16_t wh = (uint16_t)(u[j >> 1] >> (16 * (j & 1)));
                            acc = ffma(h2f(wh), h2f(xh[c * 32 + lane]), acc);
                        }
                    }
                }
            }
            // slots s = 8*j + l: (x0+x2)+(x1+x3) -> xor 16, xor 8; lo128+hi128 -> xor 4; hadd, hadd -> xor 1, xor 2
            acc = fadd(acc, __shfl_xor_sync(0xffffffffu, acc, 16));
            acc = fadd(acc, __shfl_xor_sync(0xffffffffu, acc, 8));
            acc = fadd(acc, __shfl_xor_sync(0xffffffffu, acc, 4));
            acc = fadd(acc, __shfl_xor_sync(0xffffffffu, acc, 1));
            acc = fadd(acc, __shfl_xor_sync(0xffffffffu, acc, 2));
            double sumf = (double) acc;
            for (int i = 0; i < ntail; i++)
                sumf += (double) fmul(h2f(tl[(size_t) row * ntail + i]), h2f(xh[nchunk * 32 + i]));
            res[m] = (float) sumf;
        }
        if (lane == 0) {
            float v = res[0];
            if (EPI == EPI_RESID) v = fadd(v, a.resid[(size_t) col * a.ldr + row]);
            if (EPI == EPI_GATE)  v = fmul(h2f(a.tsilu[f2h(res[0])]), res[1]);
            a.y[(size_t) col * a.ldy + row] = v;
        }
    }
}

// K1f-mc: the same F16 matmul for MULTI-token calls (prompt chunks, batched steps).  k_gemv_f16 takes one column per CTA, so
// every token re-reads the whole matrix from L2 (405 MB per 7B layer and token: a 1024-token prompt ran at the L2 rate, 66 us per
// token and layer, barely faster than decoding).  Here a CTA carries NC columns: the activations sit in shared memory as f32
// (the fp16-rounded value widened, what h2f() would produce per use) interleaved [k][NC], so one 16-byte weight load and one
// conversion per weight feed NC fma chains (LDS.128 = 4 columns).  Per column the chain is k_gemv_f16's, chunk for chunk.
template <int PRO, int EPI, int NC>
__global__ void __launch_bounds__(256) k_gemv_f16_mc(const GemvF16Args a) {
    static_assert(NC == 4 || NC == 8, "columns per CTA");
    extern __shared__ __align__(16) uint8_t smem[];
    float * xf = (float *) smem;                     // [K][NC]
    __shared__ double red[8];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, K = a.K;
    const int col0 = blockIdx.y * NC, ncols = min(NC, a.N - col0);
    grid_dep_wait();
    for (int n = 0; n < NC; n++) {
        if (n >= ncols) { for (int i = tid; i < K; i += 256) xf[(size_t) i * NC + n] = 0.f; continue; }
        const float * x = a.x + (size_t)(col0 + n) * a.ldx;
        float scale = 1.0f;
        if (PRO == PRO_NORM) {
            double s = 0.0;
            for (int i = tid; i < K; i += 256) s += (double) fmul(x[i], x[i]);
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            __syncthreads();                         // red[] of the previous column has been read
            if (lane == 0) red[warp] = s;
            __syncthreads();
            double tot = 0.0;
            for (int i = 0; i < 8; i++) tot += red[i];
            scale = __fdiv_rn(1.0f, __fsqrt_rn(fadd((float)(tot / (double) K), 1e-6f)));
        }
        for (int i = tid; i < K; i += 256) {
            float v = x[i];
            if (PRO == PRO_NORM) v = fmul(fmul(v, scale), a.norm_w[i]);
            xf[(size_t) i * NC + n] = h2f(f2h(v));
        }
    }
    __syncthreads();
    const int nchunk = K / 32, nc8 = (nchunk + 7) / 8, ntail = K & 31;
    // a warp owns TWO rows: every activation value read from shared memory feeds both (the LDS.128 stream, 4 bytes per
    // weight and column, is what bounds this kernel once the weights are shared by NC columns)
    for (int row0 = (blockIdx.x * 8 + warp) * 2; row0 < a.rows; row0 += gridDim.x * 16) {
        const bool two = row0 + 1 < a.rows;
        float res[2][2][NC];                                   // [matrix][row][column]
        #pragma unroll
        for (int m = 0; m < (EPI == EPI_GATE ? 2 : 1); m++) {
            const uint16_t * Wm = m ? a.W2 : a.W;
            const uint16_t * tl = m ? a.tail2 : a.tail;
            float acc[2][NC];
            #pragma unroll
            for (int n = 0; n < NC; n++) { acc[0][n] = 0.f; acc[1][n] = 0.f; }
            const uint4 * wp0 = (const uint4 *)(Wm + ((size_t) row0 * nc8 * 32 + lane) * 8);
            const uint4 * wp1 = (const uint4 *)(Wm + ((size_t)(two ? row0 + 1 : row0) * nc8 * 32 + lane) * 8);
            constexpr int U = 2;
            uint4 v0[U], v1[U];
            #pragma unroll
            for (int q = 0; q < U; q++) {
                v0[q] = q < nc8 ? __ldg(wp0 + (size_t) q * 32) : make_uint4(0, 0, 0, 0);
                v1[q] = q < nc8 ? __ldg(wp1 + (size_t) q * 32) : make_uint4(0, 0, 0, 0);
            }
            for (int c8 = 0; c8 < nc8; c8 += U) {
                uint4 n0[U], n1[U];                            // the next block's weights are on their way while this one is multiplied
                #pragma unroll
                for (int q = 0; q < U; q++) {
                    n0[q] = c8 + U + q < nc8 ? __ldg(wp0 + (size_t)(c8 + U + q) * 32) : make_uint4(0, 0, 0, 0);
                    n1[q] = c8 + U + q < nc8 ? __ldg(wp1 + (size_t)(c8 + U + q) * 32) : make_uint4(0, 0, 0, 0);
                }
                #pragma unroll
                for (int q = 0; q < U; q++) {
                    const uint32_t u0[4] = {v0[q].x, v0[q].y, v0[q].z, v0[q].w};
                    const uint32_t u1[4] = {v1[q].x, v1[q].y, v1[q].z, v1[q].w};
                    #pragma unroll
                    for (int j = 0; j < 8; j++) {
                        const int c = (c8 + q) * 8 + j;
                        if (c < nchunk) {
                            const float w0 = h2f((uint16_t)(u0[j >> 1] >> (16 * (j & 1))));
                            const float w1 = h2f((uint16_t)(u1[j >> 1] >> (16 * (j & 1))));
                            const float4 * xp = (const float4 *)(xf + (size_t)(c * 32 + lane) * NC);
                            #pragma unroll
                            for (int n4 = 0; n4 < NC / 4; n4++) {
                                const float4 xv = xp[n4];
                                acc[0][n4*4]   = ffma(w0, xv.x, acc[0][n4*4]);   acc[0][n4*4+1] = ffma(w0, xv.y, acc[0][n4*4+1]);
                                acc[0][n4*4+2] = ffma(w0, xv.z, acc[0][n4*4+2]); acc[0][n4*4+3] = ffma(w0, xv.w, acc[0][n4*4+3]);
                                acc[1][n4*4]   = ffma(w1, xv.x, acc[1][n4*4]);   acc[1][n4*4+1] = ffma(w1, xv.y, acc[1][n4*4+1]);
                                acc[1][n4*4+2] = ffma(w1, xv.z, acc[1][n4*4+2]); acc[1][n4*4+3] = ffma(w1, xv.w, acc[1][n4*4+3]);
                            }
                        }
                    }
                }
                #pragma unroll
                for (int q = 0; q < U; q++) { v0[q] = n0[q]; v1[q] = n1[q]; }
            }
            #pragma unroll
            for (int rr = 0; rr < 2; rr++)
                #pragma unroll
                for (int n = 0; n < NC; n++) {
                    float t = acc[rr][n];
                    t = fadd(t, __shfl_xor_sync(0xffffffffu, t, 16));
                    t = fadd(t, __shfl_xor_sync(0xffffffffu, t, 8));
                    t = fadd(t, __shfl_xor_sync(0xffffffffu, t, 4));
                    t = fadd(t, __shfl_xor_sync(0xffffffffu, t, 1));
                    t = fadd(t, __shfl_xor_sync(0xffffffffu, t, 2));
                    double sumf = (double) t;
                    const int row = (rr && two) ? row0 + 1 : row0;
                    for (int i = 0; i < ntail; i++)
                        sumf += (double) fmul(h2f(tl[(size_t) row * ntail + i]), xf[(size_t)(nchunk * 32 + i) * NC + n]);
                    res[m][rr][n] = (float) sumf;
                }
        }
        if (lane == 0) {
            #pragma unroll
            for (int rr = 0; rr < 2; rr++) {
                if (rr && !two) break;
                const int row = row0 + rr;
                #pragma unroll
                for (int n = 0; n < NC; n++) {
                    if (n < ncols) {
                        float v = res[0][rr][n];
                        if (EPI == EPI_RESID) v = fadd(v, a.resid[(size_t)(col0 + n) * a.ldr + row]);
                        if (EPI == EPI_GATE)  v = fmul(h2f(a.tsilu[f2h(res[0][rr][n])]), res[1][rr][n]);
                        a.y[(size_t)(col0 + n) * a.ldy + row] = v;
                    }
                }
            }
        }
    }
}

// K1f-ring: the same F16 matmul fed by 1-D TMA bulk copies (single-token steps).  The warp-per-row kernel above starts
// its weight stream only after its RMSNorm prologue and keeps at most a few KB per warp in flight; here
//   * a producer warp streams every consumer warp's rows through that warp's OWN ring of shared-memory stages
//     (kF16Stage bytes = kF16Stage / 512 groups of 8 chunks, contiguous in the packed row), starting BEFORE
//     griddepcontrol.wait -- weights never depend on the previous kernel -- so the stream runs through the prologue and
//     across the kernel boundary (programmatic dependent launch, trigger after the last copy is issued);
//   * the activation row is normalised once per CTA, rounded to fp16 (ggml_fp32_to_fp16_row) and stored WIDENED BACK to f32
//     in the weights' [c8][lane] permutation (two conflict-free planes of 4 chunks), so the 8 activations of a 16-byte
//     weight word are two LDS.128 and the inner loop is one F16->F32 conversion + one FFMA per weight (the ncu capture
//     of the warp-per-row kernel showed ~8 instructions per weight and 45-57 % issue utilisation: it was issue-bound);
//   * rows are whole groups of 8 chunks (K % 256 == 0: every LLaMA shape); other K use the kernel above;
//   * arithmetic unchanged: lane = slot, FMA chain in chunk order, fixed reduce tree, double tail (ggml.c:2323-2357).
constexpr int kF16Stage = 2048;                  // bytes per ring stage: 4 groups of 8 chunks of one row
constexpr int kF16Warps = 8;

template <int PRO, int EPI>
__global__ void __launch_bounds__(kF16Warps * 32 + 32) k_gemv_f16_ring(const GemvF16Args a, int NS) {
    extern __shared__ __align__(128) uint8_t smem[];
    const int K = a.K, nchunk = K / 32, nc8 = (nchunk + 7) / 8;
    const int row_bytes = nc8 * 512;
    const int n_stage = (row_bytes + kF16Stage - 1) / kF16Stage;         // stages per row (the last one may be short)
    constexpr int NM = (EPI == EPI_GATE) ? 2 : 1;
    // smem: [ring kF16Warps * NS * kF16Stage][xf: 2 planes x nc8 * 32 lanes x 4 f32][full kF16Warps*NS][empty kF16Warps*NS][red 8 doubles]
    uint8_t * ring = smem;
    float * xf = (float *)(smem + (size_t) kF16Warps * NS * kF16Stage);
    uint64_t * full = (uint64_t *)((uint8_t *) xf + (size_t) nc8 * 1024);
    uint64_t * empty = full + kF16Warps * NS;
    double * red = (double *)(empty + kF16Warps * NS);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int col = blockIdx.y;
    const int n_tiles = (a.rows + kF16Warps - 1) / kF16Warps;
    if (tid == 0) {
        for (int i = 0; i < kF16Warps * NS; i++) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        mbar_fence_init();
    }
    __syncthreads();

    if (warp == kF16Warps) {
        // ------------------------------------------------------------------ producer: lane w feeds consumer warp w
        if (lane < kF16Warps) {
            uint8_t * ring_w = ring + (size_t) lane * NS * kF16Stage;
            uint64_t * full_w = full + lane * NS, * empty_w = empty + lane * NS;
            int slot = 0, use = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                const int row = tile * kF16Warps + lane;
                if (row >= a.rows) continue;
                #pragma unroll 1
                for (int m = 0; m < NM; m++) {
                    const uint8_t * src = (const uint8_t *)((m ? a.W2 : a.W) + (size_t) row * nc8 * 256);
                    for (int st = 0; st < n_stage; st++) {
                        const uint32_t bytes = (uint32_t) min(kF16Stage, row_bytes - st * kF16Stage);
                        if (use > 0) mbar_wait(&empty_w[slot], (use - 1) & 1);
                        mbar_arrive_expect_tx(&full_w[slot], bytes);
                        bulk_g2s(ring_w + (size_t) slot * kF16Stage, src + (size_t) st * kF16Stage, bytes, &full_w[slot]);
                        if (++slot == NS) { slot = 0; use++; }
                    }
                }
            }
        }
        return;
    }

    // ---------------------------------------------------------------------- consumers
    grid_dep_wait();
    // after the wait (the ordering guarantee k_attn128's pre-wait prefetch relies on, see k_gemv): the next kernel's CTAs may
    // become resident as this kernel's CTAs drain and start THEIR weight stream
    if (tid == 0) grid_dep_launch();
    const float * x = a.x + (size_t) col * a.ldx;
    float scale = 1.0f;
    if (PRO == PRO_NORM) {
        double s = 0.0;
        for (int i = tid; i < K; i += kF16Warps * 32) s += (double) fmul(x[i], x[i]);
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) red[warp] = s;
        named_bar_sync(1, kF16Warps * 32);
        double tot = 0.0;
        for (int i = 0; i < kF16Warps; i++) tot += red[i];
        scale = __fdiv_rn(1.0f, __fsqrt_rn(fadd((float)(tot / (double) K), 1e-6f)));
    }
    for (int i = tid; i < nc8 * 256; i += kF16Warps * 32) {
        // chunk c = 8 * c8 + j of slot l (element x[c * 32 + l]) -> plane j >> 2, [c8][l][j & 3]
        const int c8 = i >> 8, l = (i >> 3) & 31, j = i & 7, c = c8 * 8 + j;
        float v = x[c * 32 + l];
        if (PRO == PRO_NORM) v = fmul(fmul(v, scale), a.norm_w[c * 32 + l]);
        xf[(size_t)(j >> 2) * nc8 * 128 + (c8 * 32 + l) * 4 + (j & 3)] = h2f(f2h(v));
    }
    named_bar_sync(1, kF16Warps * 32);

    const uint8_t * ring_w = ring + (size_t) warp * NS * kF16Stage;
    uint64_t * full_w = full + warp * NS, * empty_w = empty + warp * NS;
    int slot = 0, phase = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int row = tile * kF16Warps + warp;
        if (row >= a.rows) continue;
        float res[2] = {0.f, 0.f};
        #pragma unroll 1
        for (int m = 0; m < NM; m++) {
            float acc = 0.f;
            for (int st = 0; st < n_stage; st++) {
                mbar_wait(&full_w[slot], phase);
                const uint4 * wp = (const uint4 *)(ring_w + (size_t) slot * kF16Stage) + lane;
                const float4 * xa = (const float4 *) xf + (size_t) st * (kF16Stage / 512) * 32 + lane;
                const float4 * xb = xa + (size_t) nc8 * 32;
                const int g_n = min(kF16Stage / 512, nc8 - st * (kF16Stage / 512));
                #pragma unroll
                for (int g = 0; g < kF16Stage / 512; g++) {
                    if (g < g_n) {
                        const uint4 wv = wp[g * 32];
                        const float4 x0 = xa[g * 32], x1 = xb[g * 32];
                        const float2 w01 = __half22float2(*(const __half2 *) &wv.x), w23 = __half22float2(*(const __half2 *) &wv.y);
                        const float2 w45 = __half22float2(*(const __half2 *) &wv.z), w67 = __half22float2(*(const __half2 *) &wv.w);
                        acc = ffma(w01.x, x0.x, acc); acc = ffma(w01.y, x0.y, acc);
                        acc = ffma(w23.x, x0.z, acc); acc = ffma(w23.y, x0.w, acc);
                        acc = ffma(w45.x, x1.x, acc); acc = ffma(w45.y, x1.y, acc);
                        acc = ffma(w67.x, x1.z, acc); acc = ffma(w67.y, x1.w, acc);
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty_w[slot]);
                if (++slot == NS) { slot = 0; phase ^= 1; }
            }
            // slots s = 8*j + l: (x0+x2)+(x1+x3) -> xor 16, xor 8; lo128+hi128 -> xor 4; hadd, hadd -> xor 1, xor 2
            acc = fadd(acc, __shfl_xor_sync(0xffffffffu, acc, 16));
            acc = fadd(acc, __shfl_xor_sync(0xffffffffu, acc, 8));
            acc = fadd(acc, __shfl_xor_sync(0xffffffffu, acc, 4));
            acc = fadd(acc, __shfl_xor_sync(0xffffffffu, acc, 1));
            acc = fadd(acc, __shfl_xor_sync(0xffffffffu, acc, 2));
            res[m] = (float)(double) acc;                       // K % 32 == 0 on this path: no double-precision tail
        }
        if (lane == 0) {
            float v = res[0];
            if (EPI == EPI_RESID) v = fadd(v, a.resid[(size_t) col * a.ldr + row]);
            if (EPI == EPI_GATE)  v = fmul(h2f(a.tsilu[f2h(res[0])]), res[1]);
            a.y[(size_t) col * a.ldy + row] = v;
        }
    }
}

// repack F16 weights [rows][K] -> [rows][nc8][32 lanes][8 chunks] (+ tail [rows][K%32])
__global__ void k_repack_f16(const uint16_t * src, uint16_t * dst, uint16_t * tail, int rows, int K) {
    const int nchunk = K / 32, nc8 = (nchunk + 7) / 8, ntail = K & 31;
    const long long total = (long long) rows * nc8 * 256;
    for (long long i = blockIdx.x * (long long) blockDim.x + threadIdx.x; i < total; i += (long long) gridDim.x * blockDim.x) {
        const int j = (int)(i & 7), lane = (int)((i >> 3) & 31);
        const long long rc = i >> 8; const int c8 = (int)(rc % nc8); const long long row = rc / nc8;
        const int c = c8 * 8 + j;
        dst[i] = c < nchunk ? src[row * K + c * 32 + lane] : (uint16_t) 0;
    }
    const long long tt = (long long) rows * ntail;
    for (long long i = blockIdx.x * (long long) blockDim.x + threadIdx.x; i < tt; i += (long long) gridDim.x * blockDim.x)
        tail[i] = src[(i / ntail) * K + nchunk * 32 + (i % ntail)];
}

// =============================================================================================
// K4: RoPE (q, k) + KV append.  qkv [N][3E] f32 -> q16 [N][E] (fp16, the rounding mul_mat applies
// to src1), K cache [pos][E] fp16 (post-RoPE), V cache [pos][E] fp16.  cos/sin come from a host
// table built with the host libm, theta iterated in f32 exactly as ggml.c:12000-12044.
// =============================================================================================
struct RopeArgs {
    const float * qkv; int E, H, D, N;
    const int * n_past;
    const float2 * cs;            // [n_ctx][D/2] (cos, sin)
    uint16_t * q16; uint16_t * kc; uint16_t * vc;   // kc/vc: this layer's cache base
    const int4 * cols; size_t sess_stride;          // multi-session step: column n = (session, position, T, 0); cache base += session * stride
};

__global__ void k_rope_append(const RopeArgs a) {
    grid_dep_launch();
    grid_dep_wait();
    const int n = blockIdx.y, half = a.D / 2;
    int pos; uint16_t * kcb = a.kc, * vcb = a.vc;
    if (a.cols) { const int4 c = a.cols[n]; pos = c.y; kcb += (size_t) c.x * a.sess_stride; vcb += (size_t) c.x * a.sess_stride; }
    else pos = *a.n_past + n;
    const float * row = a.qkv + (size_t) n * 3 * a.E;
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < a.E / 2; p += gridDim.x * blockDim.x) {
        const int j = p % half;
        const float2 cs = a.cs[(size_t) pos * half + j];
        const float2 q = *(const float2 *)(row + 2 * p);
        const float2 k = *(const float2 *)(row + a.E + 2 * p);
        const float2 v = *(const float2 *)(row + 2 * a.E + 2 * p);
        const float q0 = fsub(fmul(q.x, cs.x), fmul(q.y, cs.y)), q1 = fadd(fmul(q.x, cs.y), fmul(q.y, cs.x));
        const float k0 = fsub(fmul(k.x, cs.x), fmul(k.y, cs.y)), k1 = fadd(fmul(k.x, cs.y), fmul(k.y, cs.x));
        *(uint32_t *)(a.q16 + (size_t) n * a.E + 2 * p) = (uint32_t) f2h(q0) | ((uint32_t) f2h(q1) << 16);
        *(uint32_t *)(kcb + (size_t) pos * a.E + 2 * p) = (uint32_t) f2h(k0) | ((uint32_t) f2h(k1) << 16);
        *(uint32_t *)(vcb + (size_t) pos * a.E + 2 * p) = (uint32_t) f2h(v.x) | ((uint32_t) f2h(v.y) << 16);
    }
}

// =============================================================================================
// K5: attention for one (head, query token), exact mode.
//   scores  s_t = f32( dot_f16(K[t], q16) * 1/sqrt(d) ),  t <= n_past + n      (mask, ggml.c:11476)
//   softmax e_t = EXP_TABLE[fp16(s_t - max)], S in double, p_t = e_t * (float)(1/S), rounded to fp16
//   out_c   = dot_f16(V[0..T)[c], p16[0..T)),  T = n_past + N  (the split into 32-slot body and
//             double tail follows the FULL row length T, masked entries contribute exact zeros)
// One warp = one K.q dot (lane = slot); V.p: thread (g, c) owns slots 8g..8g+7 of channel c.
// =============================================================================================
struct AttnArgs {
    const uint16_t * q16; const uint16_t * kc; const uint16_t * vc;
    const int * n_past; int E, H, D, N;
    const uint16_t * texp;
    float * out;                  // [N][E]
    float kq_scale;
    const int4 * cols; size_t sess_stride;   // multi-session step: column n = (session, position, T, 0), tcount = position + 1
};

__global__ void __launch_bounds__(512) k_attention(const AttnArgs a) {
    extern __shared__ __align__(16) uint8_t smem[];
    grid_dep_launch();
    grid_dep_wait();
    const int h = blockIdx.x, n = blockIdx.y, D = a.D, E = a.E;
    int T, tcount; const uint16_t * kcb = a.kc, * vcb = a.vc;
    if (a.cols) { const int4 c = a.cols[n]; T = c.z; tcount = c.y + 1; kcb += (size_t) c.x * a.sess_stride; vcb += (size_t) c.x * a.sess_stride; }
    else { const int n_past = *a.n_past; T = n_past + a.N; tcount = n_past + n + 1; }
    float * sc = (float *) smem;                                   // [T]
    uint16_t * p16 = (uint16_t *)(sc + ((T + 3) & ~3));            // [T]
    float * part = (float *)(p16 + ((T + 7) & ~7));                // [4][D][8]
    __shared__ double redd[16]; __shared__ float redf[16];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nwarp = blockDim.x >> 5;

    // ---- scores
    const int np = D & ~31, nch = np >> 5;
    const uint16_t * q = a.q16 + (size_t) n * E + h * D;
    float qf[8];
    #pragma unroll
    for (int c = 0; c < 8; c++) qf[c] = c < nch ? h2f(q[c * 32 + lane]) : 0.f;
    for (int t = warp; t < tcount; t += nwarp) {
        const uint16_t * k = kcb + (size_t) t * E + h * D;
        float acc = 0.f;
        #pragma unroll
        for (int c = 0; c < 8; c++) if (c < nch) acc = ffma(h2f(k[c * 32 + lane]), qf[c], acc);
        acc = fadd(acc, __shfl_xor_sync(0xffffffffu, acc, 16));
        acc = fadd(acc, __shfl_xor_sync(0xffffffffu, acc, 8));
        acc = fadd(acc, __shfl_xor_sync(0xffffffffu, acc, 4));
        acc = fadd(acc, __shfl_xor_sync(0xffffffffu, acc, 1));
        acc = fadd(acc, __shfl_xor_sync(0xffffffffu, acc, 2));
        if (lane == 0) {
            double sumf = (double) acc;
            for (int i = np; i < D; i++) sumf += (double) fmul(h2f(k[i]), h2f(q[i]));
            sc[t] = fmul((float) sumf, a.kq_scale);
        }
    }
    __syncthreads();

    // ---- softmax over t < tcount
    float mx = -INFINITY;
    for (int t = tid; t < tcount; t += blockDim.x) mx = fmaxf(mx, sc[t]);
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if (lane == 0) redf[warp] = mx;
    __syncthreads();
    mx = redf[0];
    for (int i = 1; i < nwarp; i++) mx = fmaxf(mx, redf[i]);
    double s = 0.0;
    for (int t = tid; t < tcount; t += blockDim.x) {
        const float e = h2f(a.texp[f2h(fsub(sc[t], mx))]);
        sc[t] = e; s += (double) e;
    }
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) redd[warp] = s;
    __syncthreads();
    double S = 0.0;
    for (int i = 0; i < nwarp; i++) S += redd[i];                 // fp16-valued terms: exact in any order
    const float inv = (float)(1.0 / S);
    for (int t = tid; t < tcount; t += blockDim.x) p16[t] = f2h(fmul(sc[t], inv));
    __syncthreads();

    // ---- V . p
    const int npT = T & ~31;
    const int g = tid / D, c = tid - g * D;
    if (g < 4) {
        float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        const uint16_t * v = vcb + h * D + c;
        const int lim = min(npT, tcount);
        for (int base = 8 * g; base < lim; base += 32) {
            #pragma unroll
            for (int l = 0; l < 8; l++) {
                const int t = base + l;
                if (t < lim) acc[l] = ffma(h2f(v[(size_t) t * E]), h2f(p16[t]), acc[l]);
            }
        }
        #pragma unroll
        for (int l = 0; l < 8; l++) part[(g * D + c) * 8 + l] = acc[l];
    }
    __syncthreads();
    if (tid < D) {
        float vv[8];
        #pragma unroll
        for (int l = 0; l < 8; l++) {
            const float a0 = fadd(part[(0 * D + tid) * 8 + l], part[(2 * D + tid) * 8 + l]);
            const float a1 = fadd(part[(1 * D + tid) * 8 + l], part[(3 * D + tid) * 8 + l]);
            vv[l] = fadd(a0, a1);
        }
        const float t0 = fadd(vv[0], vv[4]), t1 = fadd(vv[1], vv[5]), t2 = fadd(vv[2], vv[6]), t3 = fadd(vv[3], vv[7]);
        double sumf = (double) fadd(fadd(t0, t1), fadd(t2, t3));
        const uint16_t * v = vcb + h * D + tid;
        for (int t = npT; t < tcount; t++) sumf += (double) fmul(h2f(v[(size_t) t * E]), h2f(p16[t]));
        a.out[(size_t) n * E + h * D + tid] = (float) sumf;
    }
}

// =============================================================================================
// K5c: attention for head size 128, one thread-block CLUSTER of 4 CTAs per (head, query token).
// Same arithmetic as k_attention; the work is cut along the structure ggml_vec_dot_f16 already has:
//   * V.p keeps 32 f32 slots per channel, slot = t mod 32, and the AVX reduce first adds the four
//     8-lane vectors j = slot/8.  CTA g of the cluster owns vector j = g, i.e. positions
//     t = 32k + 8g + l (l = 0..7): it computes THOSE scores and accumulates THOSE slots, so K and V
//     are each read exactly once per step and 4x as many SMs pull on HBM/L2 per head.
//   * scores and slot partials meet in the CTAs' shared memory (distributed shared memory stores, ordered by
//     barrier.cluster release/acquire); every CTA then runs the (cheap) softmax redundantly and CTA g
//     finishes channels [32g, 32g+32) with the fixed reduce tree and the double-precision tail.
// FUSE (decode, N = 1): RoPE of q and k, fp16 rounding and the KV append of the new position are
// done in the prologue from the f32 qkv row, removing the separate rope/append launch.
// K.q: 4 lanes per position, lane ql loads the four 16 B vectors m = ql + 4c (c = chunk) and owns
// slots 8*ql + e, so each 256 B key row is one coalesced 64 B segment per chunk.
// =============================================================================================
struct Attn128Args {
    const float * qkv;            // FUSE: [N][3E] f32 (q | k | v), pre-RoPE
    const uint16_t * q16;         // !FUSE: [N][E] fp16 bits, post-RoPE
    uint16_t * kc; uint16_t * vc; // this layer's cache [n_ctx][E]
    const int * n_past; int E, H, N, n0;   // n0: first query token of this launch (chunked prefill launches)
    const float2 * cs; const uint16_t * texp;
    float * out;                  // [N][E]
    int * aq_out; float * da_out; int out_nbq; float out_dscale;   // optional: Q8_0-quantised output for the wo matmul
    int out_soff;                                                    // Q4_1 weights: Q8_1 instead, block sums at da_out + out_soff
    int n_ctx; float kq_scale;
    unsigned long long * trace;
    // multi-session step: column n = (session, position, T, 0).  FUSE: every column is an N = 1 step (T = position + 1);
    // !FUSE: launch column ny is colmap[n0 + ny], the columns of a mixed step that are not on the tiled kernel
    const int4 * cols; size_t sess_stride; const int * colmap;
    int pf_rows;                  // FUSE: rows of this CTA's K / V share staged in shared memory ahead of the dependency wait
    int lut_smem;                 // FUSE: also stage the negative half of the exp table (64 KB) -- softmax arguments are <= 0
};

constexpr int kAttnRow = 272;     // 256 B fp16 row + 16 B pad: the 8-thread phases of an LDS.128 never share a bank

__device__ __forceinline__ void cp_async16(void * dst_smem, const void * src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(smem_u32(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
}

__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void cluster_arrive_relaxed() { asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait()           { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
// address of the same shared-memory location in CTA `rank` of this cluster (distributed shared memory)
__device__ __forceinline__ uint32_t dsmem_addr(const void * local, int rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(local)), "r"(rank));
    return r;
}
__device__ __forceinline__ void dsmem_st(uint32_t addr, float v) {
    asm volatile("st.shared::cluster.f32 [%0], %1;" :: "r"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ void dsmem_st4(uint32_t addr, float4 v) {
    asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" :: "r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

template <bool FUSE>
__global__ void __cluster_dims__(4, 1, 1) __launch_bounds__(256) k_attn128(const Attn128Args a) {
    extern __shared__ __align__(16) uint8_t smem[];
    __shared__ __align__(16) uint16_t q16s[128], k16s[128], v16s[128];
    __shared__ double redd[8]; __shared__ float redf[8];
    __shared__ __align__(16) float partl[4 * 8 * 32];             // [source CTA j][slot l][channel of THIS CTA's 32]
    __shared__ __align__(8) uint64_t lutbar;
    if (threadIdx.x == 0) { B200_TRACE(a.trace, 0); grid_dep_launch(); }
    cluster_arrive_relaxed();                                      // "I am running": peers may write my shared memory after the matching wait
    // FUSE (single-token steps): the kernel before this one is the qkv matmul, whose CTAs release their dependents only
    // after their own dependency wait (see k_gemv).  So when this code runs, every kernel up to the one before qkv has
    // finished: the position counter is final and all cache rows < pos are final.  Only the qkv row itself needs the wait.
    if (!FUSE) grid_dep_wait();
    const int h = blockIdx.x >> 2, g = blockIdx.x & 3, ny = blockIdx.y, n = a.colmap ? a.colmap[a.n0 + ny] : a.n0 + ny, E = a.E;
    int T, tcount, pos;
    uint16_t * kc = a.kc, * vc = a.vc;
    if (a.cols) { const int4 c = a.cols[n]; pos = c.y; T = c.z; tcount = pos + 1; kc += (size_t) c.x * a.sess_stride; vc += (size_t) c.x * a.sess_stride; }
    else { const int n_past = *a.n_past; T = n_past + a.N; tcount = n_past + n + 1; pos = n_past + n; }
    float * sc = (float *) smem;                                   // [T]
    uint16_t * p16 = (uint16_t *)(sc + ((T + 3) & ~3));            // [T]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // staged rows: local row i <-> position 32 (i >> 3) + 8 g + (i & 7), the positions this CTA scores and accumulates
    uint8_t * Ks = smem + ((((size_t)((a.n_ctx + 3) & ~3) * 4 + (size_t)((a.n_ctx + 7) & ~7) * 2) + 15) & ~(size_t) 15);
    uint8_t * Vs = Ks + (size_t) a.pf_rows * kAttnRow;
    uint8_t * Vt = Vs + (size_t) a.pf_rows * kAttnRow;            // [32][64 B]: V rows of the double-precision tail, channels [32g, 32g+32)
    const int npf = FUSE ? min(a.pf_rows, 8 * ((pos + 31) >> 5)) : 0;
    uint16_t * luts = (uint16_t *)(Vt + 32 * 64);                 // [32768] exp table entries 0x8000..0xFFFF
    float2 cs_pre = make_float2(0.f, 0.f);
    if (FUSE) {
        if (a.lut_smem && tid == 0) {
            mbar_init(&lutbar, 1);
            mbar_fence_init();
            mbar_arrive_expect_tx(&lutbar, 65536u);
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         :: "r"(smem_u32(luts)), "l"(a.texp + 32768), "r"(65536u), "r"(smem_u32(&lutbar)) : "memory");
        }
        if (tid < 64) cs_pre = a.cs[(size_t) pos * 64 + tid];      // host-built table: no dependency on the previous kernel
        for (int idx = tid; idx < npf * 16; idx += 256) {
            const int i = idx >> 4, ch = idx & 15, t = 32 * (i >> 3) + 8 * g + (i & 7);
            if (t < pos) {
                cp_async16(Ks + (size_t) i * kAttnRow + ch * 16, kc + (size_t) t * E + h * 128 + ch * 8);
                cp_async16(Vs + (size_t) i * kAttnRow + ch * 16, vc + (size_t) t * E + h * 128 + ch * 8);
            }
        }
        if (tid < 128) {
            const int t = (T & ~31) + (tid >> 2), ch = tid & 3;
            if (t < pos) cp_async16(Vt + (size_t)(tid >> 2) * 64 + ch * 16, vc + (size_t) t * E + h * 128 + 32 * g + ch * 8);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        grid_dep_wait();
    }
    if (threadIdx.x == 0) B200_TRACE(a.trace, 1);

    // ---- phase 0: q (and, fused, the new k / v row) into shared memory
    if (FUSE) {
        if (tid < 64) {
            const float * row = a.qkv + (size_t) n * 3 * E + h * 128;
            const float2 cs = cs_pre;
            const float2 q = *(const float2 *)(row + 2 * tid);
            const float2 k = *(const float2 *)(row + E + 2 * tid);
            const float2 v = *(const float2 *)(row + 2 * E + 2 * tid);
            const float q0 = fsub(fmul(q.x, cs.x), fmul(q.y, cs.y)), q1 = fadd(fmul(q.x, cs.y), fmul(q.y, cs.x));
            const float k0 = fsub(fmul(k.x, cs.x), fmul(k.y, cs.y)), k1 = fadd(fmul(k.x, cs.y), fmul(k.y, cs.x));
            const uint32_t qq = (uint32_t) f2h(q0) | ((uint32_t) f2h(q1) << 16);
            const uint32_t kk = (uint32_t) f2h(k0) | ((uint32_t) f2h(k1) << 16);
            const uint32_t vv = (uint32_t) f2h(v.x) | ((uint32_t) f2h(v.y) << 16);
            ((uint32_t *) q16s)[tid] = qq; ((uint32_t *) k16s)[tid] = kk; ((uint32_t *) v16s)[tid] = vv;
            if (g == 0) {
                *(uint32_t *)(kc + (size_t) pos * E + h * 128 + 2 * tid) = kk;
                *(uint32_t *)(vc + (size_t) pos * E + h * 128 + 2 * tid) = vv;
            }
        }
    } else {
        if (tid < 64) ((uint32_t *) q16s)[tid] = *(const uint32_t *)(a.q16 + (size_t) n * E + h * 128 + 2 * tid);
    }
    if (FUSE) asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();

    if (threadIdx.x == 0) B200_TRACE(a.trace, 2);
    cluster_wait();                                                // every CTA of the cluster has started
    // ---- phase 1: scores of the positions this CTA owns
    {
        const int sub = tid >> 2, ql = tid & 3;
        float qf[4][8];
        #pragma unroll
        for (int c = 0; c < 4; c++)
            #pragma unroll
            for (int e = 0; e < 8; e++) qf[c][e] = h2f(q16s[32 * c + 8 * ql + e]);
        const int nloc = 8 * ((tcount + 31) >> 5);
        // two positions per thread per iteration: 8 x 16-byte loads in flight (rows past the staged window are L2 / HBM reads)
        for (int i0 = sub; i0 < nloc; i0 += 128) {
            uint4 kv[2][4];
            bool valid[2];
            int tt[2];
            #pragma unroll
            for (int u = 0; u < 2; u++) {
                const int i = i0 + 64 * u;
                const int t = 32 * (i >> 3) + 8 * g + (i & 7);
                tt[u] = t;
                valid[u] = i < nloc && t < tcount;
                const uint16_t * krow = (FUSE && t == pos) ? k16s : (i < npf ? (const uint16_t *)(Ks + (size_t) i * kAttnRow)
                                                                              : kc + (size_t) t * E + h * 128);
                #pragma unroll
                for (int c = 0; c < 4; c++) kv[u][c] = valid[u] ? *(const uint4 *)(krow + 32 * c + 8 * ql) : make_uint4(0, 0, 0, 0);
            }
            #pragma unroll
            for (int u = 0; u < 2; u++) {
                if (i0 + 64 * u >= nloc) break;                      // uniform across the warp: i0 + 64 u is < nloc for all lanes or none
                float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                if (valid[u]) {
                    #pragma unroll
                    for (int c = 0; c < 4; c++) {
                        const uint32_t w4[4] = {kv[u][c].x, kv[u][c].y, kv[u][c].z, kv[u][c].w};
                        #pragma unroll
                        for (int e = 0; e < 8; e++) {
                            const uint16_t kh = (uint16_t)(w4[e >> 1] >> (16 * (e & 1)));
                            acc[e] = ffma(h2f(kh), qf[c][e], acc[e]);
                        }
                    }
                }
                float v8[8];
                #pragma unroll
                for (int e = 0; e < 8; e++) {                            // (x0 + x2) + (x1 + x3)
                    float x = fadd(acc[e], __shfl_xor_sync(0xffffffffu, acc[e], 2));
                    v8[e] = fadd(x, __shfl_xor_sync(0xffffffffu, x, 1));
                }
                const float t0 = fadd(v8[0], v8[4]), t1 = fadd(v8[1], v8[5]), t2 = fadd(v8[2], v8[6]), t3 = fadd(v8[3], v8[7]);
                const float dot = fadd(fadd(t0, t1), fadd(t2, t3));
                if (valid[u] && ql == 0) {
                    // scores meet in every CTA's shared memory (distributed shared memory), not in an L2 scratch
                    const float sv = fmul(dot, a.kq_scale);
                    #pragma unroll
                    for (int rnk = 0; rnk < 4; rnk++) dsmem_st(dsmem_addr(sc + tt[u], rnk), sv);
                }
            }
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) B200_TRACE(a.trace, 4);
    cluster_sync_all();
    if (threadIdx.x == 0) B200_TRACE(a.trace, 5);
    if (FUSE && a.lut_smem) mbar_wait(&lutbar, 0);

    // ---- phase 2: softmax over all t < tcount (every CTA, identical results)
    float mx = -INFINITY;
    for (int t = tid; t < tcount; t += 256) mx = fmaxf(mx, sc[t]);
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if (lane == 0) redf[warp] = mx;
    __syncthreads();
    mx = redf[0];
    #pragma unroll
    for (int i = 1; i < 8; i++) mx = fmaxf(mx, redf[i]);
    double s = 0.0;
    for (int t = tid; t < tcount; t += 256) {
        const uint16_t xi = f2h(fsub(sc[t], mx));
        const float e = h2f((FUSE && a.lut_smem && xi >= 0x8000) ? luts[xi - 0x8000] : a.texp[xi]);
        sc[t] = e; s += (double) e;
    }
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) redd[warp] = s;
    __syncthreads();
    double S = 0.0;
    #pragma unroll
    for (int i = 0; i < 8; i++) S += redd[i];
    const float inv = (float)(1.0 / S);
    for (int t = tid; t < tcount; t += 256) p16[t] = f2h(fmul(sc[t], inv));
    __syncthreads();

    if (threadIdx.x == 0) B200_TRACE(a.trace, 6);
    // ---- phase 3: V.p partial sums of slots 8g..8g+7
    const int npT = T & ~31, lim = min(npT, tcount);
    if (tid < 128) {
        const int l = tid >> 4, cg = tid & 15;
        float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        // four value rows in flight per thread (rows past the staged window come from L2 / HBM: one dependent-looking load
        // per iteration made this loop 13 us at T ~ 1000); the FMAs stay in position order
        for (int tb = 8 * g + l; tb < lim; tb += 128) {
            uint4 vv4[4];
            #pragma unroll
            for (int u = 0; u < 4; u++) {
                const int t = tb + 32 * u;
                const int i = ((t >> 5) << 3) + l;
                const uint16_t * vrow = (FUSE && t == pos) ? v16s : (i < npf ? (const uint16_t *)(Vs + (size_t) i * kAttnRow)
                                                                              : vc + (size_t) t * E + h * 128);
                vv4[u] = t < lim ? *(const uint4 *)(vrow + 8 * cg) : make_uint4(0, 0, 0, 0);
            }
            #pragma unroll
            for (int u = 0; u < 4; u++) {
                const int t = tb + 32 * u;
                if (t < lim) {
                    const uint32_t u4[4] = {vv4[u].x, vv4[u].y, vv4[u].z, vv4[u].w};
                    const float p = h2f(p16[t]);
                    #pragma unroll
                    for (int e = 0; e < 8; e++) {
                        const uint16_t vh = (uint16_t)(u4[e >> 1] >> (16 * (e & 1)));
                        acc[e] = ffma(h2f(vh), p, acc[e]);
                    }
                }
            }
        }
        // channels 8cg..8cg+7 are finished by CTA cg >> 2: drop the slot partials straight into its shared memory
        const uint32_t dst = dsmem_addr(partl + (g * 8 + l) * 32 + 8 * (cg & 3), cg >> 2);
        dsmem_st4(dst, make_float4(acc[0], acc[1], acc[2], acc[3]));
        dsmem_st4(dst + 16, make_float4(acc[4], acc[5], acc[6], acc[7]));
    }
    __syncthreads();
    cluster_sync_all();
    if (threadIdx.x == 0) B200_TRACE(a.trace, 7);

    // ---- phase 4: CTA g finishes channels [32g, 32g+32)
    if (tid < 32) {
        const int c = 32 * g + tid;
        float vv[8];
        #pragma unroll
        for (int l = 0; l < 8; l++) {
            const float p0 = partl[(0 * 8 + l) * 32 + tid], p1 = partl[(1 * 8 + l) * 32 + tid];
            const float p2 = partl[(2 * 8 + l) * 32 + tid], p3 = partl[(3 * 8 + l) * 32 + tid];
            vv[l] = fadd(fadd(p0, p2), fadd(p1, p3));
        }
        const float t0 = fadd(vv[0], vv[4]), t1 = fadd(vv[1], vv[5]), t2 = fadd(vv[2], vv[6]), t3 = fadd(vv[3], vv[7]);
        double sumf = (double) fadd(fadd(t0, t1), fadd(t2, t3));
        for (int t = npT; t < tcount; t++) {
            const uint16_t vh = (FUSE && t == pos) ? v16s[c] : (FUSE ? ((const uint16_t *)(Vt + (size_t)(t - npT) * 64))[tid]
                                                                     : vc[(size_t) t * E + h * 128 + c]);
            sumf += (double) fmul(h2f(vh), h2f(p16[t]));
        }
        const float ov = (float) sumf;
        a.out[(size_t) n * E + h * 128 + c] = ov;
        // channels [32g, 32g+32) of head h are Q8_0 block 4h+g of the wo matmul's input: quantise here
        if (a.aq_out) warp_quant_block(ov, lane, a.aq_out + (size_t) n * a.out_nbq * 32, a.da_out + (size_t) n * a.out_nbq * 4,
                                       4 * h + g, a.out_dscale, a.out_soff);
    }
    if (threadIdx.x == 0) B200_TRACE(a.trace, 3);
}

struct PeerRecvArgs {
    MailboxHdr * mine;           // local mailbox
    const uint2 * inbox;         // local inbox base
    size_t slot_elems;
    int * peer_ack;              // &previous rank's mailbox->ack (remote)
    float * dst; int count;      // floats to deliver into the slice's input buffer
};

__global__ void __launch_bounds__(1024) k_peer_recv(const PeerRecvArgs a) {
    if (threadIdx.x == 0) grid_dep_launch();          // the slice's first matmul may start streaming its weights now
    grid_dep_wait();                                  // everything before this step on the stream is done (dst is free)
    const int s = a.mine->seq_in + 1;
    const uint2 * src = a.inbox + (size_t)(s & (kMbSlots - 1)) * a.slot_elems;
    const unsigned long long t0 = gtime();
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < a.count; i += gridDim.x * blockDim.x) {
        uint2 v = ld_ll(src + i);
        while ((int) v.y != s) {
            if (gtime() - t0 > kMbTimeoutNs) { a.mine->err = 1; break; }
            v = ld_ll(src + i);
        }
        a.dst[i] = __uint_as_float(v.x);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        // the LAST CTA to finish has seen every element: count the message, free the slot for the sender
        if (gridDim.x == 1 || atomicAdd(&a.mine->cnt_recv, 1) == (int) gridDim.x - 1) {
            a.mine->cnt_recv = 0;
            a.mine->seq_in = s;
            st_relaxed_sys(a.peer_ack, s);
        }
    }
}

struct PeerSendArgs {
    MailboxHdr * mine;           // local mailbox (ack, seq_out)
    uint2 * peer_inbox;          // next rank's inbox base (remote)
    size_t slot_elems;
    const float * src; int count;
};

__global__ void __launch_bounds__(1024) k_peer_send(const PeerSendArgs a) {
    if (threadIdx.x == 0) grid_dep_launch();
    grid_dep_wait();                                  // src is the previous kernel's output
    const int s = a.mine->seq_out + 1;
    if (threadIdx.x == 0) mb_wait_slot_free(a.mine, s);
    __syncthreads();
    uint2 * dst = a.peer_inbox + (size_t)(s & (kMbSlots - 1)) * a.slot_elems;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < a.count; i += gridDim.x * blockDim.x) st_ll(dst + i, a.src[i], s);
    __syncthreads();
    if (threadIdx.x == 0) {
        // every CTA read seq_out before the last one finishes, so the last one may advance it
        if (gridDim.x == 1 || atomicAdd(&a.mine->cnt_send, 1) == (int) gridDim.x - 1) { a.mine->cnt_send = 0; a.mine->seq_out = s; }
    }
}

// =============================================================================================
// K5t: attention for MULTI-token calls (prompt chunks), head size 128, query-TILED ("flash-style" staging, exact arithmetic).
// k_attn128<false> launches one cluster per (head, query): every query re-reads its head's K and V rows from L2 --
// 4.3 GB per layer for a 512-token prompt, 1.27 ms per layer, 70 % of a tensor-core prefill.  Here one CTA owns a head and
// kAttnQB = 16 consecutive queries: the head's K rows are staged in shared memory ONCE, all 16 queries score against them,
// one warp per query runs the softmax, then the V rows replace the K rows and every query accumulates against them.
// Per query the arithmetic is k_attn128's, operand for operand:
//   scores   4 lanes per position, lane ql owns the 16-byte vectors m = ql + 4c; (x0+x2)+(x1+x3), fixed 8-slot tree
//   softmax  max, fp16 exp table, sum in double (exact in any order), p = fp16(e * (float)(1/S))
//   V.p      32 f32 slots per channel (slot = t mod 32, vector j = slot / 8 -> warp-quad g), positions in ascending order,
//            ((p0+p2)+(p1+p3)) per slot, the 8-slot tree, the (T mod 32) tail in double -- T = n_past + N of the CALL
// Needs T = n_past + N <= kAttnTMax staged rows (139 KB); longer contexts keep the per-query cluster kernel.
// A mixed step (prompt chunks of several sessions in one pass) hands the kernel a table of query blocks: block y holds nq
// consecutive columns of ONE segment, and carries that segment's session (whose cache the CTA stages) and T.  A prompt chunk
// of one sequence is the one-segment case: no table, blocks of kAttnQB columns at the device-side position *n_past.
// =============================================================================================
constexpr int kAttnQB = 16;
constexpr int kAttnTMax = 512;

struct AttnBlock { int col0, nq, session, pos0, T; };   // first column, queries, session, position of the first query, T

struct AttnTiledArgs {
    const uint16_t * q16; const uint16_t * kc; const uint16_t * vc;
    const int * n_past; int E, H, N;
    const uint16_t * texp;
    float * out;                                   // [N][E]
    int * aq_out; float * da_out; int out_nbq; float out_dscale; int out_soff;
    float kq_scale;
    int t_rows, t_pad;                             // staged rows (>= the largest T) and the padded score row length
    const AttnBlock * blocks; size_t sess_stride;  // mixed step: block table (grid.y entries); cache base += session * stride
};

__global__ void __launch_bounds__(512) k_attn128_tiled(const AttnTiledArgs a) {
    extern __shared__ __align__(16) uint8_t smem[];
    if (threadIdx.x == 0) grid_dep_launch();
    grid_dep_wait();
    const int h = blockIdx.x, E = a.E;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    int col0, nq, pos0, T;                                               // first column, queries, first query's position, T
    const uint16_t * kc = a.kc, * vc = a.vc;
    if (a.blocks) {
        const AttnBlock b = a.blocks[blockIdx.y];
        col0 = b.col0; nq = b.nq; pos0 = b.pos0; T = b.T;
        kc += (size_t) b.session * a.sess_stride; vc += (size_t) b.session * a.sess_stride;
    } else {
        const int n_past = *a.n_past;
        col0 = blockIdx.y * kAttnQB; nq = min(kAttnQB, a.N - col0); pos0 = n_past + col0; T = n_past + a.N;
    }
    const int tmax = pos0 + nq;                                          // positions the block's last query sees
    uint8_t * KV = smem;                                                 // [t_rows][kAttnRow]
    float * sc = (float *)(smem + (size_t) a.t_rows * kAttnRow);         // [QB][t_pad]
    uint16_t * p16 = (uint16_t *)(sc + (size_t) kAttnQB * a.t_pad);      // [QB][t_pad]
    float * partl = (float *)(p16 + (size_t) kAttnQB * a.t_pad);         // [4 groups][8 slots][128 channels]
    uint16_t * q16s = (uint16_t *)(partl + 4 * 8 * 128);                 // [QB][128]

    // ---- stage the head's key rows t < tmax and the block's query rows
    for (int idx = tid; idx < tmax * 16; idx += 512) {
        const int t = idx >> 4, ch = idx & 15;
        cp_async16(KV + (size_t) t * kAttnRow + ch * 16, kc + (size_t) t * E + h * 128 + ch * 8);
    }
    for (int idx = tid; idx < nq * 16; idx += 512) {
        const int q = idx >> 4, ch = idx & 15;
        cp_async16(q16s + q * 128 + ch * 8, a.q16 + (size_t)(col0 + q) * E + h * 128 + ch * 8);
    }
    cp_async_wait_all();
    __syncthreads();

    // ---- scores: 128 positions per pass, 4 lanes per position
    {
        const int ql = tid & 3;
        for (int q = 0; q < nq; q++) {
            const int tcount = pos0 + q + 1;
            float qf[4][8];
            #pragma unroll
            for (int c = 0; c < 4; c++)
                #pragma unroll
                for (int e = 0; e < 8; e++) qf[c][e] = h2f(q16s[q * 128 + 32 * c + 8 * ql + e]);
            for (int t0 = 0; t0 < tcount; t0 += 128) {
                const int t = t0 + (tid >> 2);
                const bool valid = t < tcount;
                float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                if (valid) {
                    const uint16_t * krow = (const uint16_t *)(KV + (size_t) t * kAttnRow);
                    uint4 kv[4];
                    #pragma unroll
                    for (int c = 0; c < 4; c++) kv[c] = *(const uint4 *)(krow + 32 * c + 8 * ql);
                    #pragma unroll
                    for (int c = 0; c < 4; c++) {
                        const uint32_t u[4] = {kv[c].x, kv[c].y, kv[c].z, kv[c].w};
                        #pragma unroll
                        for (int e = 0; e < 8; e++) {
                            const uint16_t kh = (uint16_t)(u[e >> 1] >> (16 * (e & 1)));
                            acc[e] = ffma(h2f(kh), qf[c][e], acc[e]);
                        }
                    }
                }
                float v8[8];
                #pragma unroll
                for (int e = 0; e < 8; e++) {                            // (x0 + x2) + (x1 + x3)
                    float x = fadd(acc[e], __shfl_xor_sync(0xffffffffu, acc[e], 2));
                    v8[e] = fadd(x, __shfl_xor_sync(0xffffffffu, x, 1));
                }
                const float u0 = fadd(v8[0], v8[4]), u1 = fadd(v8[1], v8[5]), u2 = fadd(v8[2], v8[6]), u3 = fadd(v8[3], v8[7]);
                const float dot = fadd(fadd(u0, u1), fadd(u2, u3));
                if (valid && ql == 0) sc[(size_t) q * a.t_pad + t] = fmul(dot, a.kq_scale);
            }
        }
    }
    __syncthreads();

    // ---- softmax: warp q owns query q; meanwhile the value rows replace the key rows
    for (int idx = tid; idx < tmax * 16; idx += 512) {
        const int t = idx >> 4, ch = idx & 15;
        cp_async16(KV + (size_t) t * kAttnRow + ch * 16, vc + (size_t) t * E + h * 128 + ch * 8);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    if (warp < nq) {
        const int q = warp, tcount = pos0 + q + 1;
        float * s_q = sc + (size_t) q * a.t_pad;
        uint16_t * p_q = p16 + (size_t) q * a.t_pad;
        float mx = -INFINITY;
        for (int t = lane; t < tcount; t += 32) mx = fmaxf(mx, s_q[t]);
        for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        double s = 0.0;
        for (int t = lane; t < tcount; t += 32) {
            const float e = h2f(a.texp[f2h(fsub(s_q[t], mx))]);
            s_q[t] = e; s += (double) e;
        }
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);      // fp16-valued terms: exact in any order
        const float inv = (float)(1.0 / s);
        for (int t = lane; t < tcount; t += 32) p_q[t] = f2h(fmul(s_q[t], inv));
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();

    // ---- V . p: FOUR queries at a time, one per 128-thread group.  Thread (l, cg) of a group walks all four slot vectors
    // j = 0..3 of its slot l (positions 32k + 8j + l, ascending per slot) for channels 8cg..8cg+7, adds them as the AVX reduce
    // does -- (j0 + j2) + (j1 + j3) -- in registers, and only the 8-slot tree crosses threads (group-local shared memory).
    const int npT = T & ~31;
    const int grp = tid >> 7, gt = tid & 127, l = gt >> 4, cg = gt & 15;
    float * part_g = partl + grp * (8 * 128);                            // [8 slots][128 channels] of this group
    for (int q0 = 0; q0 < nq; q0 += 4) {
        const int q = q0 + grp;
        const bool live = q < nq;
        const int n = col0 + q, tcount = pos0 + q + 1, lim = live ? min(npT, tcount) : 0;
        const uint16_t * p_q = p16 + (size_t) q * a.t_pad;
        float acc[4][8];
        #pragma unroll
        for (int j = 0; j < 4; j++)
            #pragma unroll
            for (int e = 0; e < 8; e++) acc[j][e] = 0.f;
        for (int tb = l; tb < lim; tb += 32) {
            #pragma unroll
            for (int j = 0; j < 4; j++) {
                const int t = tb + 8 * j;
                if (t < lim) {
                    const uint4 vv = *(const uint4 *)(KV + (size_t) t * kAttnRow + cg * 16);
                    const uint32_t u[4] = {vv.x, vv.y, vv.z, vv.w};
                    const float p = h2f(p_q[t]);
                    #pragma unroll
                    for (int e = 0; e < 8; e++) {
                        const uint16_t vh = (uint16_t)(u[e >> 1] >> (16 * (e & 1)));
                        acc[j][e] = ffma(h2f(vh), p, acc[j][e]);
                    }
                }
            }
        }
        float4 * dst = (float4 *)(part_g + l * 128 + 8 * cg);
        dst[0] = make_float4(fadd(fadd(acc[0][0], acc[2][0]), fadd(acc[1][0], acc[3][0])), fadd(fadd(acc[0][1], acc[2][1]), fadd(acc[1][1], acc[3][1])),
                             fadd(fadd(acc[0][2], acc[2][2]), fadd(acc[1][2], acc[3][2])), fadd(fadd(acc[0][3], acc[2][3]), fadd(acc[1][3], acc[3][3])));
        dst[1] = make_float4(fadd(fadd(acc[0][4], acc[2][4]), fadd(acc[1][4], acc[3][4])), fadd(fadd(acc[0][5], acc[2][5]), fadd(acc[1][5], acc[3][5])),
                             fadd(fadd(acc[0][6], acc[2][6]), fadd(acc[1][6], acc[3][6])), fadd(fadd(acc[0][7], acc[2][7]), fadd(acc[1][7], acc[3][7])));
        named_bar_sync(1 + grp, 128);
        if (live) {
            const int c = gt;                                            // one channel per thread of the group
            float vv[8];
            #pragma unroll
            for (int k = 0; k < 8; k++) vv[k] = part_g[k * 128 + c];
            const float t0 = fadd(vv[0], vv[4]), t1 = fadd(vv[1], vv[5]), t2 = fadd(vv[2], vv[6]), t3 = fadd(vv[3], vv[7]);
            double sumf = (double) fadd(fadd(t0, t1), fadd(t2, t3));
            for (int t = npT; t < tcount; t++)
                sumf += (double) fmul(h2f(((const uint16_t *)(KV + (size_t) t * kAttnRow))[c]), h2f(p_q[t]));
            const float ov = (float) sumf;
            a.out[(size_t) n * E + h * 128 + c] = ov;
            // channels [32 w, 32 w + 32) of head h are Q8_0 block 4 h + w of the wo matmul's input (w = warp within the group)
            if (a.aq_out) warp_quant_block(ov, lane, a.aq_out + (size_t) n * a.out_nbq * 32, a.da_out + (size_t) n * a.out_nbq * 4,
                                           4 * h + (gt >> 5), a.out_dscale, a.out_soff);
        }
        named_bar_sync(1 + grp, 128);
    }
}

// position counter kept on the device so a captured graph can be replayed for every token
__global__ void k_advance(int * n_past, int by) { grid_dep_wait(); if (threadIdx.x == 0) *n_past += by; }
// the same for a pipelined slice whose LAST matmul stored its rows into the next rank's inbox (EPI_RESID_SEND): the message
// is complete when that kernel is, count it
__global__ void k_advance_sent(int * n_past, int by, MailboxHdr * mine) {
    grid_dep_wait();
    if (threadIdx.x == 0) { *n_past += by; mine->seq_out = mine->seq_out + 1; }
}
// multi-session step: the columns of one session are consecutive, so the last column of each segment sets that session's
// counter to its position + 1 (= n_past + segment length); one writer per session
__global__ void k_advance_segs(int * n_past, const int4 * cols, int n) {
    grid_dep_wait();
    for (int i = threadIdx.x; i < n; i += blockDim.x)
        if (i == n - 1 || cols[i + 1].x != cols[i].x) n_past[cols[i].x] = cols[i].y + 1;
}

}  // namespace b200

namespace b200 {
// =============================================================================================
// lm_head with a Q6_K `output.weight` (what llama.cpp's quantize writes for q4_0 models whose n_embd is a multiple
// of 256, llama.cpp:2523-2528): exact restatement of ggml_vec_dot_q6_K_q8_K's AVX2 branch (k_quants.c:3484-3561)
// on activations quantised like quantize_row_q8_K_reference (k_quants.c:1133-1168).
//   per 256-weight super-block i and AVX lane L (bytes 4L..4L+3 of each 32-byte vector):
//     S_L = sum_{j<2,k<4} scale[8j+2k+(L>=4)] * sum_{e<4} (q6 - 32) * q8        (all integer)
//     acc_L = fma(d_i, (float) S_L, acc_L),  d_i = y.d * fp16->f32(x.d);   result = hsum_float_8(acc)
// Packed layout (k_repack_q6k): per (row, super-block) 288 B = 8 lanes x 8 words of (q6-32) int8x4 in (j,k) order,
// 16 int8 scales, fp16 d, padding.  Thread (row, L); 32 rows per CTA.
// =============================================================================================
constexpr int kWT_Q6_K = 14;
constexpr int kQ6Packed = 288;

__global__ void k_repack_q6k(const uint8_t * src, uint8_t * dst, int rows, int nb256) {
    const long long total = (long long) rows * nb256 * 72;       // 72 words per packed block
    for (long long i = blockIdx.x * (long long) blockDim.x + threadIdx.x; i < total; i += (long long) gridDim.x * blockDim.x) {
        const int wi = (int)(i % 72); const long long rb = i / 72;
        const uint8_t * blk = src + rb * 210;                    // ql[128] qh[64] scales[16] d(2)
        uint32_t out = 0;
        if (wi < 64) {
            const int L = wi >> 3, jk = wi & 7, j = jk >> 2, k = jk & 3;
            for (int e = 0; e < 4; e++) {
                const int l = 4 * L + e;
                const uint8_t qlb = blk[64 * j + l + ((k & 1) ? 32 : 0)];
                const int lo = (k & 2) ? (qlb >> 4) : (qlb & 0xF);
                const int hi = (blk[128 + 32 * j + l] >> (2 * k)) & 3;
                out |= ((uint32_t)(((lo | (hi << 4)) - 32) & 0xFF)) << (8 * e);
            }
        } else if (wi < 68) {
            const uint8_t * sc = blk + 192 + (wi - 64) * 4;
            out = (uint32_t) sc[0] | ((uint32_t) sc[1] << 8) | ((uint32_t) sc[2] << 16) | ((uint32_t) sc[3] << 24);
        } else if (wi == 68) {
            out = (uint32_t) blk[208] | ((uint32_t) blk[209] << 8);
        }
        ((uint32_t *) dst)[i] = out;
    }
}

struct LmHeadQ6Args {
    const uint8_t * W; int rows, K;
    const float * x; int ldx; const float * norm_w;
    float * y; int ldy; int N;
};

__global__ void __launch_bounds__(256) k_lmhead_q6k(const LmHeadQ6Args a) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int nb = a.K / 256, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, n = blockIdx.y;
    int * a8 = (int *) smem;                       // [nb][8 jk][8 L] words
    float * dq = (float *)(a8 + nb * 64);          // [nb]
    float * ys = dq + nb;                          // [K] normalised activations
    __shared__ double red[8];
    __shared__ unsigned long long redk[8];
    const float * x = a.x + (size_t) n * a.ldx;
    // RMSNorm * weight (ggml.c:10309-10352, 9062)
    double s = 0.0;
    for (int i = tid; i < a.K; i += 256) s += (double) fmul(x[i], x[i]);
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) red[warp] = s;
    __syncthreads();
    double tot = 0.0;
    for (int i = 0; i < 8; i++) tot += red[i];
    const float scale = __fdiv_rn(1.0f, __fsqrt_rn(fadd((float)(tot / (double) a.K), 1e-6f)));
    for (int i = tid; i < a.K; i += 256) ys[i] = fmul(fmul(x[i], scale), a.norm_w[i]);
    __syncthreads();
    // quantize_row_q8_K_reference: thread t owns element t of every super-block
    for (int b = 0; b < nb; b++) {
        const float v = ys[b * 256 + tid];
        // first element with the largest magnitude: key = (|v| bits, reversed index)
        unsigned long long key = ((unsigned long long) __float_as_uint(fabsf(v)) << 32) | (unsigned)(255 - tid);
        for (int o = 16; o > 0; o >>= 1) { const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o); key = other > key ? other : key; }
        if (lane == 0) redk[warp] = key;
        __syncthreads();
        unsigned long long best = redk[0];
        for (int i = 1; i < 8; i++) best = redk[i] > best ? redk[i] : best;
        const int arg = 255 - (int)(best & 0xFFFFFFFFu);
        const float mx = ys[b * 256 + arg];
        int q = 0; float d = 0.f;
        if ((best >> 32) != 0) {
            const float iscale = __fdiv_rn(-128.f, mx);
            const float val = fadd(fmul(iscale, v), 12582912.f);                 // nearest_int (k_quants.c:50-55)
            q = min(127, (int)((__float_as_uint(val) & 0x007fffffu) - 0x00400000));
            d = __fdiv_rn(1.0f, iscale);
        }
        // element t = 128 j + 32 k + 4 L + e  ->  byte e of word [jk][L]
        const int j = tid >> 7, k = (tid >> 5) & 3, L = (tid >> 2) & 7, e = tid & 3;
        uint32_t pk = ((uint32_t)(q & 0xFF)) << (8 * e);
        pk |= __shfl_xor_sync(0xffffffffu, pk, 1);
        pk |= __shfl_xor_sync(0xffffffffu, pk, 2);
        if (e == 0) a8[b * 64 + (j * 4 + k) * 8 + L] = (int) pk;
        if (tid == 0) dq[b] = d;
        __syncthreads();
    }
    const int row = blockIdx.x * 32 + (tid >> 3), L = tid & 7;
    float acc = 0.f;
    if (row < a.rows) {
        const uint8_t * wrow = a.W + (size_t) row * nb * kQ6Packed;
        for (int b = 0; b < nb; b++) {
            const uint4 * wp = (const uint4 *)(wrow + (size_t) b * kQ6Packed + L * 32);
            const uint4 w0 = wp[0], w1 = wp[1];
            const uint32_t ww[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
            const int8_t * sc = (const int8_t *)(wrow + (size_t) b * kQ6Packed + 256);
            const float dw = h2f(*(const uint16_t *)(wrow + (size_t) b * kQ6Packed + 272));
            int S = 0;
            #pragma unroll
            for (int jk = 0; jk < 8; jk++)
                S += (int) sc[2 * jk + (L >> 2)] * __dp4a((int) ww[jk], a8[b * 64 + jk * 8 + L], 0);
            acc = ffma(fmul(dq[b], dw), (float) S, acc);
        }
    }
    acc = fadd(acc, __shfl_xor_sync(0xffffffffu, acc, 4));
    acc = fadd(acc, __shfl_xor_sync(0xffffffffu, acc, 2));
    acc = fadd(acc, __shfl_xor_sync(0xffffffffu, acc, 1));
    if (L == 0 && row < a.rows) a.y[(size_t) n * a.ldy + row] = acc;
}
}  // namespace b200
