"""BASELINE.json's configurations at their FULL sizes, checked bit for bit against the outputs the compiled reference
(oracle/_ref) gave on the same files and inputs, recorded in tests/golden/reference_runs.json by gen_reference_runs.py.

  config 1  OpenLLaMA-3B shapes (n_embd 3200, d_head 100, n_ff 8640), two nodes: layers 0-16 / 17-25, single prompt,
            greedy decode: 16-token prompt + 32 generated tokens -- token ids AND hidden states bit-exact  (SURVEY 8d)
  config 4  LLaMA-7B F16 layer shapes at n_ctx 2048 (the reference is fixed at 512: compared on the positions it has)
  config 5  LLaMA-13B layer shapes, 8 sessions in one batched step vs the reference running each sequence alone
Weights are synthetic (no network); the FILE is the ground truth both sides load."""
import numpy as np
import pytest

from distributedllm_b200 import ggjt
from oracle import goldens, oracle

pytestmark = pytest.mark.gpu


def test_config1_3b_two_nodes_greedy_decode(tmp_path):
    from distributedllm_b200 import capi
    from distributedllm_b200.compute_node.slices import import_llm
    llm = import_llm()
    want = goldens.load("config1")                                 # the reference's own embedding lookup, slices and argmax
    sh = ggjt.SHAPES["3b"]
    pa, pb, extra = str(tmp_path / "a.bin"), str(tmp_path / "b.bin"), str(tmp_path / "extra.bin")
    ggjt.write_fast_q4_slice(pa, sh, 0, 16, seed=3)
    ggjt.write_fast_q4_slice(pb, sh, 17, 25, seed=3)
    ggjt.write_fast_q4_extra(extra, sh, seed=3)
    gpu = [capi.Slice(pa, 0, 512), capi.Slice(pb, 0, 512)]
    tg = [1 + (i * 7919) % 31999 for i in range(16)]              # SURVEY 8d: token-level synthetic prompt
    ids_gpu, bad = [], []
    for step in range(33):
        # everything through the drop-in `llm` module + C ABI
        x = np.array(llm.prepare_embeddings(extra, tg), np.float32).reshape(len(tg), sh.n_embd)
        for s in gpu:
            x = s.forward(x)
        m = goldens.mismatch(x, want["hidden"][step])
        if m:
            bad.append("step %d: %s" % (step, m))
        a = llm.get_next_token(extra, x.ravel().tolist())
        ids_gpu.append(a)
        tg = [a]
    assert ids_gpu == want["ids"]
    assert not bad, bad
    assert len(set(ids_gpu)) > 4                                   # the run is not degenerate
    for s in gpu:
        s.close()


def test_config4_7b_f16_layer_at_n_ctx_2048(tmp_path):
    from distributedllm_b200 import capi
    want = goldens.load("config4")
    sh = ggjt.SHAPES["7b"]
    p = str(tmp_path / "f16.bin")
    ggjt.write_fast_f16_slice(p, sh, 0, 0, seed=4)
    gpu = capi.Slice(p, 0, 2048)
    rng = np.random.default_rng(9)
    for i, n in enumerate((24, 1, 1, 9, 1)):
        x = rng.standard_normal((n, sh.n_embd), dtype=np.float32)
        goldens.check(gpu.forward(x), want[i], "call %d" % i)
    # beyond the reference's 512 positions: the long context still runs and stays finite
    gpu.clear_context()
    x = rng.standard_normal((128, sh.n_embd), dtype=np.float32)
    for _ in range(10):
        y = gpu.forward(x)
    assert gpu.n_past == 1280 and np.isfinite(y).all()
    gpu.close()


def test_config5_13b_batch_of_8_sessions(tmp_path):
    from distributedllm_b200 import capi
    want = goldens.load("config5")                                 # each session run alone on the reference
    sh = ggjt.SHAPES["13b"]
    p = str(tmp_path / "q4.bin")
    ggjt.write_fast_q4_slice(p, sh, 0, 0, seed=5)
    B = 8
    gpu = capi.Slice(p, 0, 512, n_sessions=B)
    rng = np.random.default_rng(10)
    for b in range(B):
        x = rng.standard_normal((3 + 2 * b, sh.n_embd), dtype=np.float32)
        goldens.check(gpu.session_forward(b, x), want["prompts"][b], "session %d prompt" % b)
    for step in range(3):
        x = rng.standard_normal((B, sh.n_embd), dtype=np.float32)
        got = gpu.batch_forward(list(range(B)), x)
        for b in range(B):
            goldens.check(got[b], want["steps"][step][b], "step %d session %d" % (step, b))
    gpu.close()


def test_config2_7b_q4_decode_at_the_end_of_the_sequence(tmp_path):
    """The positions BASELINE's metric is quoted on: a 2-layer LLaMA-7B Q4_0 slice taken to p = 500 in prompt chunks,
    then decoded token by token at p = 500..511 (T up to 512 in attention: every staged-row / tail path of the decode
    kernels) -- hidden states bit-identical to the compiled reference at every step, including the chunked prefill."""
    from distributedllm_b200 import capi
    want = goldens.load("config2")
    sh = ggjt.SHAPES["7b"]
    p = str(tmp_path / "q4_7b_2l.bin")
    ggjt.write_fast_q4_slice(p, sh, 0, 1, seed=6)
    gpu = capi.Slice(p, 0, 512)
    rng = np.random.default_rng(11)
    pos, calls, bad = 0, iter(want), []
    while pos < 500:                                               # the reference's arena caps a call at ~64 tokens
        n = min(oracle.RefSlice.MAX_CHUNK, 500 - pos)
        x = rng.standard_normal((n, sh.n_embd), dtype=np.float32)
        m = goldens.mismatch(gpu.forward(x), next(calls))
        if m:
            bad.append("prompt chunk at position %d: %s" % (pos, m))
        pos += n
    assert not bad, bad
    for pos in range(500, 512):
        x = rng.standard_normal((1, sh.n_embd), dtype=np.float32)
        goldens.check(gpu.forward(x), next(calls), "decode step at position %d" % pos)
    assert gpu.n_past == 512
    with pytest.raises(capi.B200Error):                            # position 512 does not exist at n_ctx 512
        gpu.forward(rng.standard_normal((1, sh.n_embd), dtype=np.float32))
    gpu.close()
