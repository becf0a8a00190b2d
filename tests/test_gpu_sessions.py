"""Sessions and batched steps (SURVEY 8f N3, BASELINE config 5): every session must behave bit-for-bit like a private
reference slice (tensor_processor.cpp:1488-1562 holds ONE context; here there are several over the same weights), and
a batched step must equal stepping its sessions one at a time."""
import numpy as np
import pytest

from distributedllm_b200 import ggjt

pytestmark = pytest.mark.gpu


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


@pytest.mark.parametrize("shape,wtype", [("tiny128", ggjt.T_Q4_0), ("tiny3b", ggjt.T_Q4_0), ("tiny128", ggjt.T_Q8_0),
                                         ("tiny", ggjt.T_F16), ("tiny128", ggjt.T_Q4_1)])
def test_batched_step_equals_private_contexts(tmp_models, shape, wtype):
    from distributedllm_b200 import capi
    from oracle import oracle
    sh = ggjt.SHAPES[shape]
    path = tmp_models(shape, wtype, 0, 1, seed=21)
    B = 5
    gpu = capi.Slice(path, 0, 96, n_sessions=8)
    rng = np.random.default_rng(3)
    prompt_len = [7, 1, 33, 12, 40]                      # ragged prompts -> every session at a different position
    sessions = [6, 0, 3, 7, 2]
    cpu = []
    for b in range(B):
        ref = oracle.PortSlice(path, 96)
        x = rng.standard_normal((prompt_len[b], sh.n_embd), dtype=np.float32)
        assert (_bits(gpu.session_forward(sessions[b], x)) == _bits(ref.forward(x))).all()
        cpu.append(ref)
    for step in range(6):
        x = rng.standard_normal((B, sh.n_embd), dtype=np.float32)
        got = gpu.batch_forward(sessions, x)
        for b in range(B):
            want = cpu[b].forward(x[b:b + 1])
            assert (_bits(got[b]) == _bits(want[0])).all(), (step, b)
    assert [gpu.session_n_past(k) for k in sessions] == [p + 6 for p in prompt_len]
    # sessions that were never touched are still empty; a partial batch works; order inside a batch is free
    assert gpu.session_n_past(1) == 0 and gpu.session_n_past(5) == 0
    x = rng.standard_normal((2, sh.n_embd), dtype=np.float32)
    got = gpu.batch_forward([3, 6], x)
    assert (_bits(got[0]) == _bits(cpu[2].forward(x[0:1])[0])).all()
    assert (_bits(got[1]) == _bits(cpu[0].forward(x[1:2])[0])).all()
    for c in cpu:
        c.close()
    gpu.close()


def test_batched_step_stays_exact_with_fast_prefill_on(tmp_models):
    """A batched step of 40 sessions has more columns than fast mode's min_tokens (32), yet it is 40 single-token steps:
    with fast prefill on it stays bit-identical to the same batch with fast prefill off."""
    from distributedllm_b200 import capi
    sh = ggjt.SHAPES["tiny128b"]
    path = tmp_models("tiny128b", ggjt.T_Q4_0, 0, 1, seed=23)
    B = 40
    fast, exact = capi.Slice(path, 0, 64, n_sessions=B), capi.Slice(path, 0, 64, n_sessions=B)
    rng = np.random.default_rng(5)
    for k in range(B):                                   # prompts shorter than min_tokens: exact on both handles
        x = rng.standard_normal((1 + k % 7, sh.n_embd), dtype=np.float32)
        assert (_bits(fast.session_forward(k, x)) == _bits(exact.session_forward(k, x))).all()
    fast.set_fast_prefill(True, 32)
    sessions = list(rng.permutation(B))
    for step in range(3):
        x = rng.standard_normal((B, sh.n_embd), dtype=np.float32)
        assert (_bits(fast.batch_forward(sessions, x)) == _bits(exact.batch_forward(sessions, x))).all(), step
    fast.close()
    exact.close()


def test_session_zero_is_the_reference_context_and_errors(tmp_models):
    from distributedllm_b200 import capi
    sh = ggjt.SHAPES["tiny128"]
    path = tmp_models("tiny128", ggjt.T_Q4_0, 0, 1, seed=22)
    a, b = capi.Slice(path, 0, 64, n_sessions=3), capi.Slice(path, 0, 64)
    rng = np.random.default_rng(4)
    x = rng.standard_normal((9, sh.n_embd), dtype=np.float32)
    assert (_bits(a.forward(x)) == _bits(b.forward(x))).all()
    assert a.n_past == 9 and a.session_n_past(0) == 9 and a.session_n_past(1) == 0
    y = rng.standard_normal((1, sh.n_embd), dtype=np.float32)
    assert (_bits(a.session_forward(0, y)) == _bits(b.forward(y))).all()      # graph replay, keyed by session
    assert (_bits(a.session_forward(2, x)) == _bits(capi.Slice(path, 0, 64).forward(x))).all()
    with pytest.raises(capi.B200Error) as e:
        a.batch_forward([1, 1], np.zeros((2, sh.n_embd), np.float32))
    assert e.value.code == 1
    with pytest.raises(capi.B200Error):
        a.session_forward(3, y)
    with pytest.raises(capi.B200Error):
        a.batch_forward([0, 1, 2, 0], np.zeros((4, sh.n_embd), np.float32))
    a.session_clear(2)
    assert a.session_n_past(2) == 0 and a.session_n_past(0) == 10
    a.session_clear()
    assert a.n_past == 0
    # context overflow of one member rejects the whole batch and leaves every position unchanged
    a.session_forward(1, np.zeros((64, sh.n_embd), np.float32))
    with pytest.raises(capi.B200Error) as e:
        a.batch_forward([0, 1], np.zeros((2, sh.n_embd), np.float32))
    assert e.value.code == 5 and a.session_n_past(0) == 0 and a.session_n_past(1) == 64
    a.close()
    b.close()
