"""GPU: the reference-facing `llm` module, the resident extra layers, and the whole node/client stack with
the slice forward on the B200 -- checked against goldens dumped from the reference (tests/golden)."""
import gzip
import io
import json
import os
import struct
import threading

import numpy as np
import pytest

from distributedllm_b200 import ggjt

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


@pytest.fixture(scope="module")
def llm():
    from distributedllm_b200.compute_node.slices import import_llm
    return import_llm()


def test_llm_module_slice_functions(llm, tmp_models):
    from oracle import oracle
    sh = ggjt.SHAPES["tiny128"]
    path = tmp_models("tiny128", ggjt.T_Q4_0, 0, 2)
    cpu = oracle.PortSlice(path, 512)
    assert llm.load_slice(path) == 0
    rng = np.random.default_rng(3)
    for n in (6, 1, 1):
        x = rng.standard_normal((n, sh.n_embd), dtype=np.float32)
        out = llm.propagate_forward(x.ravel().tolist())
        assert isinstance(out, list) and len(out) == n * sh.n_embd
        assert (_bits(np.array(out, np.float32)) == _bits(cpu.forward(x)).ravel()).all()
    assert llm.clear_context() == 0
    cpu.clear_context()
    x = rng.standard_normal((2, sh.n_embd), dtype=np.float32)
    raw = llm.propagate_forward_buffer(x)                       # additive zero-copy variant
    assert (np.frombuffer(raw, np.uint32) == _bits(cpu.forward(x)).ravel()).all()
    with pytest.raises(TypeError):
        llm.propagate_forward([1, 2, 3])                        # ints are not floats (tensor_processor.cpp:2115)
    # context overflow: the reference would scribble past its KV cache; here: an int status like a failed eval
    llm.clear_context()
    status = llm.propagate_forward([0.0] * (513 * sh.n_embd))
    assert isinstance(status, int) and status != 0
    assert llm.unload_slice() == 0
    with pytest.raises(RuntimeError):
        llm.load_slice("/no/such/file.bin")


def test_extra_layers_match_reference_goldens(llm, tmp_path):
    g = np.load(os.path.join(GOLD, "extra.npz"))
    sh = ggjt.SHAPES["tiny"]
    extra = str(tmp_path / "extra.bin")
    ggjt.write_synth_extra(extra, sh, ggjt.T_Q4_0, seed=0)
    emb = np.array(llm.prepare_embeddings(extra, g["tokens"].tolist()), np.float32).reshape(-1, sh.n_embd)
    assert (_bits(emb) == _bits(g["emb"])).all()
    hid = g["hidden"]
    la = np.array(llm.get_logits(extra, hid.ravel().tolist(), True), np.float32).reshape(len(hid), -1)
    assert (_bits(la) == _bits(g["logits_all"])).all()
    ll = np.array(llm.get_logits(extra, hid.ravel().tolist(), False), np.float32)
    assert (_bits(ll) == _bits(g["logits_last"]).ravel()).all()
    assert llm.get_next_token(extra, hid.ravel().tolist()) == int(np.argmax(g["logits_last"]))
    assert llm.decode_token(extra, 1) == "<s>"


def test_q4_1_extra_layers_match_reference_goldens(llm, tmp_path):
    """Client side of a `quantize q4_1` model whose n_embd is not a multiple of 256: tok_embeddings rows are nibble * d + m,
    output.weight goes through the Q4_1 x Q8_1 dot."""
    g = np.load(os.path.join(GOLD, "extra_q4_1.npz"))
    sh = ggjt.SHAPES["tiny"]
    extra = str(tmp_path / "extra.bin")
    ggjt.write_synth_extra(extra, sh, ggjt.T_Q4_1, seed=0)
    emb = np.array(llm.prepare_embeddings(extra, g["tokens"].tolist()), np.float32).reshape(-1, sh.n_embd)
    assert (_bits(emb) == _bits(g["emb"])).all()
    hid = g["hidden"]
    la = np.array(llm.get_logits(extra, hid.ravel().tolist(), True), np.float32).reshape(len(hid), -1)
    assert (_bits(la) == _bits(g["logits_all"])).all(), int((_bits(la) != _bits(g["logits_all"])).sum())


def test_q6k_lm_head_matches_reference_goldens(llm):
    """The extra-layers file exactly as the reference's `quantize q4_0` + `slice_model extra_layers` produce it
    (Q6_K output.weight): logits bit-identical to the reference's get_llm_output."""
    g = np.load(os.path.join(GOLD, "extra_q6k.npz"))
    extra = os.path.join(GOLD, "extra_q6k.bin")
    hid = g["hidden"]
    la = np.array(llm.get_logits(extra, hid.ravel().tolist(), True), np.float32).reshape(len(hid), -1)
    assert (_bits(la) == _bits(g["logits_all"])).all(), int((_bits(la) != _bits(g["logits_all"])).sum())
    emb = np.array(llm.prepare_embeddings(extra, g["tokens"].tolist()), np.float32).reshape(len(g["tokens"]), -1)
    assert (_bits(emb) == _bits(g["emb"])).all()


def test_tokenizer_matches_reference_goldens(llm, tmp_path):
    gold = json.load(open(os.path.join(GOLD, "tokenizer.json")))
    raw = gzip.open(os.path.join(GOLD, "llama_vocab.bin.gz")).read()
    vocab, pos = [], 0
    while pos < len(raw):
        (n,) = struct.unpack_from("<I", raw, pos)
        text = raw[pos + 4:pos + 4 + n]
        (score,) = struct.unpack_from("<f", raw, pos + 4 + n)
        vocab.append((text, score))
        pos += 8 + n
    assert len(vocab) == 32000
    sh = ggjt.ModelShape(32000, 64, 32, 2, 1)
    extra = str(tmp_path / "vocab_extra.bin")
    ggjt.write_synth_extra(extra, sh, ggjt.T_Q4_0, seed=0, vocab=vocab)
    for case in gold["cases"]:
        assert llm.tokenize_prompt(extra, case["text"]) == case["ids"], case["text"]


def _serve(tmp_path):
    import distributedllm_b200.compute_node.tcp_handler as th
    from distributedllm_b200.compute_node import serve
    th._PROD = None
    srv = serve.make_server("127.0.0.1", 0, str(tmp_path / "uploads"))
    threading.Thread(target=srv.serve_forever, daemon=True).start()
    return srv


def test_node_end_to_end_greedy_decode_matches_cpu_path(llm, tmp_path):
    """provision -> push_slice -> load_slice -> generate (greedy) through the TCP RPC with the slice on the GPU;
    token ids must equal the CPU oracle's (bit-exact hidden states make this an equality, not a tolerance)."""
    from distributedllm_b200.client import DistributedLLM
    from distributedllm_b200.control_center import Connection
    from oracle import oracle
    sh = ggjt.SHAPES["tiny128"]
    full = str(tmp_path / "full.bin")
    ggjt.write_synth_full(full, sh, ggjt.T_Q4_0, seed=0)
    sl, extra = str(tmp_path / "slice.bin"), str(tmp_path / "extra.bin")
    ggjt.slice_model(full, sl, 0, sh.n_layer - 1)
    ggjt.extract_extra_layers(full, extra)
    srv = _serve(tmp_path)
    try:
        addr = ("127.0.0.1", srv.server_address[1])
        conn = Connection(addr)
        with open(sl, "rb") as f:
            name = conn.push_slice(f, "tiny128", {"layer_from": 0, "layer_to": sh.n_layer - 1})["file_name"]
        conn.load_slice(name)
        assert conn.get_status()["status"] == "up"
        model = DistributedLLM([addr], extra)
        ids = model.generate_greedy("the the a in", max_steps=12)
        # CPU path: same extra layers (GPU lm_head is exact, tested above), slice on the C oracle
        cpu = oracle.PortSlice(sl, 512)
        toks = llm.tokenize_prompt(extra, "the the a in")
        want = []
        for _ in range(12):
            emb = np.array(llm.prepare_embeddings(extra, toks), np.float32).reshape(len(toks), -1)
            hid = cpu.forward(emb)
            t = llm.get_next_token(extra, hid.ravel().tolist())
            want.append(t)
            toks = [t]
        assert ids == want
        # additive binary wire format / chained route (one node here): same ids, tensors never become Python floats
        for wire in ("bytes", "chain"):
            assert DistributedLLM([addr], extra, wire=wire).generate_greedy("the the a in", max_steps=12) == want, wire
        ppl = model.perplexity("the the a in the")
        assert np.isfinite(ppl) and ppl > 1
    finally:
        srv.shutdown()
        srv.server_close()
        llm.unload_slice()


def test_gpu_matches_live_reference(tmp_models):
    """Against the outputs the compiled reference gave on these inputs (reference_runs.json: gpu_live)."""
    from distributedllm_b200 import capi
    from oracle import goldens
    sh = ggjt.SHAPES["tiny128"]
    want = goldens.load("gpu_live")
    path = tmp_models("tiny128", ggjt.T_Q4_0, 0, 2, seed=5)
    gpu = capi.Slice(path, 0, 512)
    rng = np.random.default_rng(8)
    for i, n in enumerate((45, 1, 1, 1)):
        x = rng.standard_normal((n, sh.n_embd), dtype=np.float32)
        goldens.check(gpu.forward(x), want[i], "call %d" % i)
    gpu.close()


def test_goldens_on_gpu(tmp_path):
    """The committed reference goldens, replayed on the GPU."""
    from distributedllm_b200 import capi
    meta = json.load(open(os.path.join(GOLD, "slices.json")))
    meta.update(json.load(open(os.path.join(GOLD, "slices_q4_1.json"))))
    data = dict(np.load(os.path.join(GOLD, "slices.npz")))
    data.update(np.load(os.path.join(GOLD, "slices_q4_1.npz")))
    for name, m in meta.items():
        sh = ggjt.SHAPES[m["shape"]]
        path = str(tmp_path / (name + ".bin"))
        ggjt.write_synth_slice(path, sh, m["layers"][0], m["layers"][1], m["wtype"], seed=0)
        gpu = capi.Slice(path, 0, 512)
        for i in range(len(m["schedule"])):
            got = gpu.forward(data["%s/x%d" % (name, i)])
            assert (_bits(got) == _bits(data["%s/y%d" % (name, i)])).all(), (name, i)
        gpu.close()


def test_llm_module_sessions(llm, tmp_models, monkeypatch):
    """Additive llm functions for several sequences on one node; each session equals a private slice."""
    from distributedllm_b200 import capi
    sh = ggjt.SHAPES["tiny128"]
    path = tmp_models("tiny128", ggjt.T_Q4_0, 0, 1, seed=31)
    monkeypatch.setenv("B200_SESSIONS", "3")
    monkeypatch.setenv("B200_N_CTX", "64")
    llm.load_slice(path)
    try:
        rng = np.random.default_rng(5)
        priv = [capi.Slice(path, 0, 64) for _ in range(3)]
        for k, n in enumerate((4, 9, 1)):
            x = rng.standard_normal((n, sh.n_embd), dtype=np.float32)
            got = np.frombuffer(llm.propagate_forward_session(k, x), np.float32).reshape(n, -1)
            assert (_bits(got) == _bits(priv[k].forward(x))).all()
        x = rng.standard_normal((3, sh.n_embd), dtype=np.float32)
        got = np.frombuffer(llm.propagate_forward_batch([2, 0, 1], x), np.float32).reshape(3, -1)
        for j, k in enumerate((2, 0, 1)):
            assert (_bits(got[j]) == _bits(priv[k].forward(x[j:j + 1])[0])).all()
        # the reference-shaped call is session 0
        y = rng.standard_normal((1, sh.n_embd), dtype=np.float32)
        assert (_bits(np.array(llm.propagate_forward(y.ravel().tolist()), np.float32)) == _bits(priv[0].forward(y)[0])).all()
        with pytest.raises(RuntimeError):
            llm.propagate_forward_batch([0, 0], np.zeros((2, sh.n_embd), np.float32))
        with pytest.raises(ValueError):
            llm.propagate_forward_batch([0, 1], np.zeros((1, sh.n_embd), np.float32))
        assert llm.clear_session(-1) == 0
        for p in priv:
            p.close()
    finally:
        llm.unload_slice()


def test_node_loads_slices_with_different_n_ctx_from_metadata_without_env(llm, tmp_path, monkeypatch):
    """SURVEY 8f N4: n_ctx / n_sessions / device are LOAD METADATA carried by the slice's upload metadata through
    routes.load_slice_request -> SliceContainer.load -> llm.load_slice(path, n_ctx=..., ...); no process environment."""
    from distributedllm_b200.control_center import Connection
    for v in ("B200_N_CTX", "B200_SESSIONS", "B200_DEVICE"):
        monkeypatch.delenv(v, raising=False)
    sh = ggjt.SHAPES["tiny128"]
    p = str(tmp_path / "s.bin")
    ggjt.write_synth_slice(p, sh, 0, 1, ggjt.T_Q4_0, seed=0)
    srv = _serve(tmp_path)
    try:
        conn = Connection(("127.0.0.1", srv.server_address[1]))
        names = []
        for meta in ({"layer_from": 0, "layer_to": 1, "n_ctx": 96, "n_sessions": 3},
                     {"layer_from": 0, "layer_to": 1, "b200": {"n_ctx": 160}}):
            with open(p, "rb") as f:
                names.append(conn.push_slice(f, "tiny128", meta)["file_name"])
        conn.load_slice(names[0])
        info = llm.slice_info()
        assert (info["n_ctx"], info["n_sessions"], info["device"]) == (96, 3, 0)
        x = np.zeros(97 * sh.n_embd, np.float32)
        assert isinstance(llm.propagate_forward(x.tolist()), int)              # 97 tokens overflow n_ctx = 96
        conn.load_slice(names[1])                                              # replaces the first slice (freed first)
        info = llm.slice_info()
        assert (info["n_ctx"], info["n_sessions"]) == (160, 1)
        out = llm.propagate_forward(np.zeros(97 * sh.n_embd, np.float32).tolist())
        assert isinstance(out, list) and len(out) == 97 * sh.n_embd
    finally:
        srv.shutdown()
        srv.server_close()
        llm.unload_slice()
    assert llm.slice_info() is None


def test_load_rejects_a_context_the_attention_kernels_cannot_hold(tmp_models):
    from distributedllm_b200 import capi
    path = tmp_models("tiny128", ggjt.T_Q4_0, 0, 1)
    with pytest.raises(capi.B200Error) as ei:
        capi.Slice(path, 0, 1 << 16)
    assert ei.value.code == 1 and "n_ctx" in str(ei.value)                     # B200_EINVAL at load, not a launch error later
    ok = capi.Slice(path, 0, 4096)
    ok.close()


def test_unload_racing_a_forward_is_safe(llm, tmp_models):
    """ADVICE r1: the node is a ThreadingTCPServer -- an unload / reload arriving while another thread's
    propagate_forward is on the GPU must neither crash nor free the slice under it."""
    sh = ggjt.SHAPES["tiny128"]
    path = tmp_models("tiny128", ggjt.T_Q4_0, 0, 2)
    llm.load_slice(path, n_ctx=512)
    stop, errors, done = threading.Event(), [], [0]

    def hammer():
        x = np.zeros((8, sh.n_embd), np.float32)
        while not stop.is_set():
            try:
                llm.clear_context()
                llm.propagate_forward_buffer(x)
                done[0] += 1
            except RuntimeError:
                pass                                                        # "no slice loaded" between unload and load
            except Exception as e:                                          # noqa: BLE001
                errors.append(repr(e))
                return
    ts = [threading.Thread(target=hammer) for _ in range(3)]
    for t in ts:
        t.start()
    try:
        for i in range(12):
            llm.unload_slice()
            llm.load_slice(path, n_ctx=256 if i % 2 else 512)
    finally:
        stop.set()
        for t in ts:
            t.join()
        llm.unload_slice()
    assert not errors and done[0] > 0
