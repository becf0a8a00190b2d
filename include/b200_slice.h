/*
 * b200_slice.h -- C ABI of libb200slice.so, the B200 (sm_100a) slice runtime.
 *
 * Drop-in boundary: these entry points are what the reference's CPython module `llm`
 * (distllm/tensor_processor.cpp:2238-2260) binds for the per-slice forward path, with Python
 * lists replaced by plain float buffers.  Each function cites the reference interface it
 * replaces.  Conventions:
 *   - return 0 on success, a B200_E* code otherwise; no C++ exception crosses the ABI;
 *     b200_last_error() returns a thread-local, human-readable description of the last failure;
 *   - the caller owns every in/out buffer (they are copied, as the reference copies at
 *     tensor_processor.cpp:523 and 798-799); the library owns weights, KV cache and n_past;
 *   - activations are row-major [n_tokens][n_embd] float32 (ggml ne0 = n_embd);
 *   - one handle = one slice on one GPU; calls on a handle are serialised by an internal mutex;
 *   - there is NO CPU fallback: every call fails with B200_ENODEV when no sm_100 device is present.
 */
#ifndef B200_SLICE_H
#define B200_SLICE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct b200_slice b200_slice_t;
typedef struct b200_extra b200_extra_t;

enum {
    B200_OK       = 0,
    B200_EINVAL   = 1,   /* bad argument (null handle, n_tokens <= 0, ...) */
    B200_EFILE    = 2,   /* slice file missing / malformed / unsupported tensor type */
    B200_ENODEV   = 3,   /* no CUDA device, or device is not sm_100 */
    B200_ECUDA    = 4,   /* a CUDA call or kernel failed */
    B200_ECONTEXT = 5,   /* n_past + n_tokens would exceed n_ctx */
    B200_ENCCL    = 6,   /* pipeline hand-off failed */
};

typedef struct b200_slice_info {
    int32_t n_embd, n_head, n_ff, n_layer, first_layer, n_ctx, n_past, weight_type, device;
    int64_t weight_bytes;       /* bytes of slice weights as stored in the reference file */
    int64_t kv_bytes_per_pos;   /* KV-cache bytes appended per position (all layers) */
} b200_slice_info_t;

/* ---- slice lifetime ------------------------------------------------------------------ */

/* llm.load_slice(path)  (tensor_processor.cpp:1995-2009; TransformerSlice ctor 1497-1510).
 * Parses the reference's slice file (GGJT v3 + first_layer, tensor_processor.cpp:152-248),
 * uploads and repacks the weights into HBM, allocates the f16 KV cache for n_ctx positions.
 * n_ctx <= 0 selects the reference default, 512 (vendor examples/common.h:28). */
int b200_slice_load(const char * path, int device, int n_ctx, b200_slice_t ** out);

/* llm.unload_slice()  (tensor_processor.cpp:2023-2030).  Waits for a call that is already inside the library on this
 * handle; the caller must not START another call on the handle concurrently with (or after) unload -- the `llm` module
 * guarantees that with a reference count (csrc/llm_module.cpp). */
int b200_slice_unload(b200_slice_t * s);

/* Create the CUDA context of `device` ahead of the first load (the first CUDA call of a process takes 0.3 s on a 1-GPU
 * box, seconds on an 8-GPU box); optional, lets a caller time b200_slice_load without it. */
int b200_device_init(int device);

/* llm.clear_context()  (tensor_processor.cpp:2012-2021, TransformerSlice::clear_context 1512-1521):
 * n_past = 0; the cache contents become unreachable. */
int b200_slice_clear(b200_slice_t * s);

int b200_slice_info(b200_slice_t * s, b200_slice_info_t * info);

/* Extension (no reference counterpart): move n_past back to `n_past` (<= current) so a benchmark
 * can re-decode positions without re-running the prefill.  Cache rows below n_past stay valid. */
int b200_slice_rewind(b200_slice_t * s, int n_past);

/* ---- the hot path -------------------------------------------------------------------- */

/* llm.propagate_forward(values)  (tensor_processor.cpp:2127-2163 -> TransformerSlice::forward
 * 1523-1544 -> llama_eval_internal 474-809).  `in` and `out` are HOST buffers of
 * n_tokens*n_embd floats; the call copies in (H2D), runs every layer of the slice on the GPU at
 * positions [n_past, n_past+n_tokens), copies out (D2H), and advances n_past. */
int b200_slice_forward(b200_slice_t * s, const float * in, int n_tokens, float * out);

/* Same, with DEVICE buffers on the slice's GPU; asynchronous on the slice's stream unless
 * `sync` != 0.  Used when the activation already lives in HBM (chained slices, benchmarks). */
int b200_slice_forward_device(b200_slice_t * s, const float * d_in, int n_tokens, float * d_out, int sync);

/* ---- sessions and batched steps (additive: SURVEY 8f N3, BASELINE config 5) --------------------
 * The reference holds ONE context per process (tensor_processor.cpp:1491, 1992), so a node serves one sequence at a
 * time.  Here a slice may hold n_sessions independent contexts (own KV cache + own n_past) over the same weights.
 * Session 0 is the context every b200_slice_* call above uses.  Each session behaves exactly like a reference slice
 * of its own: results are bit-identical to a private slice fed the same tokens. */
int b200_slice_load_ex(const char * path, int device, int n_ctx, int n_sessions, b200_slice_t ** out);
int b200_session_count(b200_slice_t * s);
int b200_session_n_past(b200_slice_t * s, int session);                      /* -1 on a bad argument */
int b200_session_clear(b200_slice_t * s, int session);                       /* session -1 = every session */
int b200_session_rewind(b200_slice_t * s, int session, int n_past);
int b200_session_forward(b200_slice_t * s, int session, const float * in, int n_tokens, float * out);          /* host buffers */
int b200_session_forward_device(b200_slice_t * s, int session, const float * d_in, int n_tokens, float * d_out, int sync);

/* Throughput mode: ONE token for each of n_seq DISTINCT sessions in a single pass.  in / out are [n_seq][n_embd]; row b
 * belongs to sessions[b] and is processed at that session's own position.  The weights are streamed once for the whole
 * batch; every row's arithmetic is that of its own single-token step, so the result is bit-identical to calling
 * b200_session_forward(sessions[b], row b, 1, ...) for each b.  A session listed twice -> B200_EINVAL. */
int b200_batch_forward(b200_slice_t * s, const int * sessions, int n_seq, const float * in, float * out);      /* host buffers */
int b200_batch_forward_device(b200_slice_t * s, const int * sessions, int n_seq, const float * d_in, float * d_out, int sync);

/* Mixed step (continuous batching): for each of n_seg DISTINCT sessions, n_tokens[i] >= 1 consecutive tokens of that session,
 * all in ONE pass -- a new session's prompt chunk rides in the same weight pass as the other sessions' decode tokens.  in / out
 * are [sum n_tokens][n_embd], the segments back to back in the listed order.  Segment i's rows are bit-identical to
 * b200_session_forward(sessions[i], <its rows>, n_tokens[i]) on the state before the call, whatever the other segments are;
 * b200_batch_forward is the case n_tokens[i] = 1.  Always exact mode: the fast-prefill switch is ignored.
 * A session listed twice, n_tokens[i] <= 0, a session out of range, or sum n_tokens > n_ctx -> B200_EINVAL; a session with
 * n_past + n_tokens[i] > n_ctx -> B200_ECONTEXT.  A rejected step advances no session.  No device: B200_ENODEV. */
int b200_mixed_forward(b200_slice_t * s, const int * sessions, const int * n_tokens, int n_seg, const float * in, float * out);   /* host buffers */
int b200_mixed_forward_device(b200_slice_t * s, const int * sessions, const int * n_tokens, int n_seg,
                              const float * d_in, float * d_out, int sync);

/* Fast mode for prefill calls (n_tokens >= min_tokens): the Q4_0 / Q8_0 weight matmuls run on the tcgen05 tensor cores with
 * the dequantisation fused in (csrc/fastgemm2.cuh; Q4_1 and F16 slices ignore the switch and stay exact).  NOT bit-exact: operands are rounded to fp16 after the reference's
 * Q8_0 activation quantisation; deviation from exact mode is bounded in tests/test_gpu_fast_prefill.py and, one matmul at a
 * time, in tests/test_gpu_fast_matmul.py.  The fp16 operands limit the un-normalised inputs of wo and w2 to |x| <= 65504;
 * beyond that fast mode overflows where exact mode stays finite.  Off by default (or B200_FAST_PREFILL=1).  Single-token
 * steps, batched steps (b200_batch_forward*) and mixed steps (b200_mixed_forward*) always run in exact mode, whatever min_tokens is: only a multi-token call of
 * one sequence takes the fast path. */
int b200_slice_set_fast_prefill(b200_slice_t * s, int on, int min_tokens);

/* Block until everything queued on the slice's stream has finished. */
int b200_slice_sync(b200_slice_t * s);

/* Device-side time of the kernels launched by the most recent forward call, in milliseconds
 * (CUDA events on the slice's stream); -1 if none. */
float b200_slice_last_ms(b200_slice_t * s);

/* Record CUDA event `which` (0 = start, 1 = stop) on the slice's stream, and read the time between
 * them: how bench.py times K steps on the stream the kernels are launched on. */
int b200_slice_mark(b200_slice_t * s, int which);
float b200_slice_mark_elapsed_ms(b200_slice_t * s);

/* Per-kernel event timing.  While enabled, forwards run un-graphed with one CUDA-event pair around
 * every launch; _read() returns the summed device time and launch count per kernel class
 * (0 qkv matmul, 1 rope+append, 2 attention, 3 wo matmul, 4 w1/w3 matmul, 5 w2 matmul, 6 advance)
 * since the last read. */
int b200_slice_profile(b200_slice_t * s, int enable);
int b200_slice_profile_read(b200_slice_t * s, float * ms_by_class, int * launches_by_class, int n_class);

/* Number of kernel launches (graph nodes included) issued by this handle so far. */
int64_t b200_slice_launch_count(b200_slice_t * s);

/* Device pointers of the slice's own input / output staging buffers ([n_ctx][n_embd] f32). */
float * b200_slice_dev_in(b200_slice_t * s);
float * b200_slice_dev_out(b200_slice_t * s);

/* Test hook: copy `count` 32-bit words of an internal activation buffer to the host after a forward
 * (0 qkv, 1 att, 2 ffin, 3 gate, 4 xa, 5 xb, 6 q16, 7 k-cache, 8 v-cache).  Not part of the drop-in surface. */
int b200_debug_read(b200_slice_t * s, int which, size_t offset_words, size_t count, void * out);

/* Test hook: run ONE fast-mode weight matmul of `layer` (0-based within the slice) on private buffers, with the launch
 * sequence a fast prefill uses; the KV cache and n_past are untouched.  which: 0 qkv (RMSNorm by attention_norm, x is
 * [n_tokens][n_embd], y has 3 n_embd rows), 1 wo (x [n_tokens][n_embd], y = W x + resid), 2 w1|w3 (RMSNorm by ffn_norm,
 * y = silu(w1 x) * (w3 x), n_ff rows), 3 w2 (x [n_tokens][n_ff], y = W x + resid).  resid is [n_tokens][n_embd] (wo, w2 only).
 * tile: 0 = the token tile a forward would pick, 128 / 256 force one (256 needs the default v2 kernel).
 * y receives [round_up(n_tokens, 256)][rows] floats; rows past n_tokens keep the sentinel 0xFFFFFFFF (a NaN).
 * xh receives the fp16 activation operand [n_tokens][K] (K = n_ff for w2, else n_embd).
 * B200_EINVAL when the slice's weights do not qualify for fast mode. */
int b200_debug_fast_matmul(b200_slice_t * s, int layer, int which, int tile, const float * x, int n_tokens, const float * resid,
                           float * y, uint16_t * xh);

/* Measurement aid (bench.py roofline): while on, a decode step launches only its weight-matmul kernels. */
int b200_debug_skip_attention(b200_slice_t * s, int on);

/* In-kernel %globaltimer timeline of the matmul / attention launches (8 stamps per CTA: [0] entry, [1] dependency
 * resolved, [2] prologue done, [3] exit, [4] last weight copy issued).  _enable(1) re-captures the decode graph with
 * tracing; _read returns the launches recorded so far (class ids as in b200_slice_profile_read). */
int b200_debug_trace_enable(b200_slice_t * s, int on);
int b200_debug_trace_read(b200_slice_t * s, unsigned long long * out, int * cls, int * ctas, int max_launches);

/* Timeline of the persistent single-token step (csrc/persist.cuh; B200_PERSIST=1 and B200_PTRACE=1 at load): 16 stamps per
 * (CTA, layer) of the most recent step; returns the number of (CTA, layer) records written. */
int b200_debug_ptrace_read(b200_slice_t * s, unsigned long long * out, size_t cap_words);

/* ---- layer-slice pipeline over NVLink (one process per GPU) --------------------------- */

/* Join a pipeline of `nranks` slices (rank r holds layer range r of the nodes_map).  `nccl_id`
 * is the 128-byte ncclUniqueId obtained with b200_pipeline_unique_id on rank 0 and distributed
 * by the host (torch.distributed store / TCP).  Replaces the client relaying the activation over
 * TCP between nodes (cli_api/common.py:148-154, control_center.py:224-244) for slices that share
 * one NVSwitch box: the hand-off becomes ONE ncclSend/ncclRecv per hop. */
int b200_pipeline_unique_id(void * id128);
int b200_pipeline_init(b200_slice_t * s, int rank, int nranks, const void * id128);

/* One pipeline step on this rank: rank 0 takes `d_in` (device, may be NULL on other ranks), every
 * rank r>0 receives [n_tokens][n_embd] from r-1, runs its layers, and sends to r+1; the last rank
 * leaves the result in its dev_out buffer and, when `ring` != 0, also sends it to rank 0 (ring = 1: rank 0
 * receives it inside this step into the buffer b200_pipeline_result() returns, closing the token loop; ring = 2: rank 0
 * collects it later, see b200_pipeline_collect). Asynchronous on the slice's stream. */
int b200_pipeline_step(b200_slice_t * s, const float * d_in, int n_tokens, int ring);
/* The same hand-off for one session, and for a batched step (one token for each listed session: [n_seq][n_embd] moves
 * between the slices).  Every rank passes the same session list. */
int b200_pipeline_step_session(b200_slice_t * s, int session, const float * d_in, int n_tokens, int ring);
int b200_pipeline_step_batch(b200_slice_t * s, const int * sessions, int n_seq, const float * d_in, int ring);
/* The same hand-off for a mixed step ([sum n_tokens][n_embd] moves between the slices; see b200_mixed_forward).  Every rank
 * passes the same segment list; a rejected list is rejected on every rank before anything is sent or received. */
int b200_pipeline_step_mixed(b200_slice_t * s, const int * sessions, const int * n_tokens, int n_seg, const float * d_in, int ring);
/* Peer-memory hand-off (the B200-native hop): every rank owns a MAILBOX in its HBM (sequence flags + two inbox slots of
 * [n_ctx][n_embd] f32) that its ring neighbours map over NVLink with cudaIpc.  After b200_pipeline_init, each rank
 * exports its 64-byte handle, the host gathers all of them (torch.distributed all_gather, a file, ...) and every rank
 * connects.  From then on b200_pipeline_step* hands the activation over with a store into the next rank's mailbox + a
 * flag, written by the slice's last kernel and polled by the next slice's first kernel inside the captured step graph:
 * no host code, no NCCL kernel between slices.  B200_PP_PEER=0 (or never connecting) keeps ncclSend / ncclRecv. */
int b200_pipeline_mailbox_export(b200_slice_t * s, void * handle64);
int b200_pipeline_mailbox_connect(b200_slice_t * s, const void * handles /* nranks x 64 bytes, rank order */, int nranks);
int b200_pipeline_transport(b200_slice_t * s);   /* 1 = peer mailboxes, 0 = NCCL */
int b200_pipeline_set_transport(b200_slice_t * s, int peer);   /* all ranks alike; 1 only after a successful connect */
/* Measurement aid: bare hand-offs around the ring, no layers; device microseconds per iteration (= nranks hops). */
int b200_pipeline_pingpong(b200_slice_t * s, int n_rows, int iters, float * us_per_iter);
int b200_pipeline_error(b200_slice_t * s);       /* non-zero: a mailbox poll timed out (8 s) on this rank */

/* Throughput mode (BASELINE config 5): a step issued with ring = 2 sends the last slice's output to rank 0 but rank 0 does
 * not wait for it inside the step; it collects the results later, in issue order, with b200_pipeline_collect (rank 0 only;
 * a no-op elsewhere).  Rank 0 can so issue steps for several sessions back to back and every slice stays busy. */
int b200_pipeline_collect(b200_slice_t * s, int n_rows, float * d_dst /* NULL: the pipeline result buffer */);

/* Device pointer of the pipeline's final activation: on rank 0 after a ring step the last slice's output, else dev_out. */
float * b200_pipeline_result(b200_slice_t * s);
int b200_pipeline_destroy(b200_slice_t * s);

/* ---- client-side extra layers (tok_embeddings / norm / output), next-row N1 ------------ */

/* Replace get_inputs / get_llm_output / sample_next_token (tensor_processor.cpp:1717-1908),
 * which re-read the extra-layers file on every call, with a resident copy. */
int b200_extra_load(const char * path, int device, b200_extra_t ** out);
int b200_extra_unload(b200_extra_t * e);
int b200_extra_dims(b200_extra_t * e, int * n_vocab, int * n_embd);
/* llm.prepare_embeddings(path, tokens) -> [n_tokens][n_embd] (host). */
int b200_extra_embed(b200_extra_t * e, const int32_t * tokens, int n_tokens, float * out);
/* llm.get_logits(path, emb, all_logits) -> [n_tokens or 1][n_vocab] (host). */
int b200_extra_logits(b200_extra_t * e, const float * emb, int n_tokens, int all_logits, float * out);
/* llm.get_next_token(path, emb): argmax of the last token's logits (first maximum wins). */
int b200_extra_next_token(b200_extra_t * e, const float * emb, int n_tokens, int32_t * token);
/* llm.tokenize_prompt(path, prompt): BOS + sentencepiece-style merge (tensor_processor.cpp:1596-1714).
 * Returns the token count (may exceed cap; only cap are written) or a negative error. */
int b200_extra_tokenize(b200_extra_t * e, const char * prompt, int32_t * out, int cap);
/* llm.decode_token(path, id): pointer to the token's bytes (owned by the handle), length in *len. */
const char * b200_extra_token_text(b200_extra_t * e, int32_t id, int * len);

const char * b200_last_error(void);
const char * b200_version(void);

#ifdef __cplusplus
}
#endif
#endif /* B200_SLICE_H */
