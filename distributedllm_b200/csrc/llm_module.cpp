// llm_module.cpp -- the CPython module `llm`, drop-in for the reference's module of the same name
// (distllm/tensor_processor.cpp:1992-2275): the same nine functions with the same argument meaning, backed
// by the B200 slice runtime through its C ABI (include/b200_slice.h) instead of llama.cpp on the CPU.
//
//   load_slice(path) -> 0            propagate_forward(list[float]) -> list[float] (int status on eval failure)
//   unload_slice() -> 0              clear_context() -> 0
//   tokenize_prompt(extra, prompt) -> list[int]       prepare_embeddings(extra, tokens) -> list[float]
//   get_logits(extra, emb, all_logits) -> list[float] get_next_token(extra, emb) -> int
//   decode_token(extra, id) -> str
//
// Differences, all additive or stricter: the GIL is released around GPU work; a load failure raises
// RuntimeError instead of printing and leaving a half-built slice (tensor_processor.cpp:1506-1509); a non-float
// list element raises TypeError instead of returning NULL with no exception set (2115-2117, 2137-2139);
// `propagate_forward_buffer(bytes-like f32) -> bytes` avoids the per-float list marshalling; the extra-layers
// file is parsed once per path, not on every call.  Context length, GPU ordinal and session count are LOAD METADATA:
// load_slice(path, n_ctx=0, device=-1, n_sessions=0) -- keyword extras the reference hard-codes
// (tensor_processor.cpp:1997-2006); unset values fall back to B200_N_CTX / B200_DEVICE / B200_SESSIONS, then 512 / 0 / 1.
// The loaded slice is reference-counted: a forward holds its reference for the whole GPU call, load/unload swap the
// pointer and the last user frees it, so an unload racing an in-flight propagate_forward (ThreadingTCPServer) is safe.
#define PY_SSIZE_T_CLEAN
#include <Python.h>

#include <chrono>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "b200_slice.h"

struct SliceRef {                                         // frees the slice when the last user drops it
    b200_slice_t * h;
    explicit SliceRef(b200_slice_t * p) : h(p) {}
    ~SliceRef() { if (h) b200_slice_unload(h); }
};
typedef std::shared_ptr<SliceRef> SlicePtr;
static SlicePtr g_slice;                                  // one slice per process, like the reference (line 1992)
static std::map<std::string, b200_extra_t *> g_extra;
static std::mutex g_mu;
static SlicePtr current_slice() { std::lock_guard<std::mutex> lk(g_mu); return g_slice; }

static int env_int(const char * n, int d) { const char * v = getenv(n); return v ? atoi(v) : d; }

static PyObject * raise_b200(const char * what) {
    PyErr_Format(PyExc_RuntimeError, "%s: %s", what, b200_last_error());
    return nullptr;
}

// list[float] (the reference's argument type) or any C-contiguous buffer of 4-byte floats (bytes / bytearray are taken
// as raw float32; typed buffers must say 'f')
static bool list_to_floats(PyObject * obj, std::vector<float> & out) {
    Py_buffer view;
    if (!PyList_Check(obj) && PyObject_CheckBuffer(obj)) {
        if (PyObject_GetBuffer(obj, &view, PyBUF_C_CONTIGUOUS | PyBUF_FORMAT) != 0) return false;
        const char * f = view.format;
        const bool raw = !f || !strcmp(f, "B") || !strcmp(f, "b") || !strcmp(f, "c");
        const bool f32 = f && (!strcmp(f, "f") || !strcmp(f, "<f") || !strcmp(f, "=f") || !strcmp(f, "@f")) && view.itemsize == 4;
        if ((!raw && !f32) || view.len % 4) {
            PyBuffer_Release(&view);
            PyErr_SetString(PyExc_TypeError, "tensor buffer must hold float32 values (format 'f', or raw bytes of length 4*n)");
            return false;
        }
        out.assign((const float *) view.buf, (const float *) view.buf + view.len / sizeof(float));
        PyBuffer_Release(&view);
        return true;
    }
    PyObject * seq = PySequence_Fast(obj, "expected a list of floats");
    if (!seq) return false;
    const Py_ssize_t n = PySequence_Fast_GET_SIZE(seq);
    out.resize((size_t) n);
    for (Py_ssize_t i = 0; i < n; i++) {
        PyObject * it = PySequence_Fast_GET_ITEM(seq, i);
        if (!PyFloat_Check(it)) { Py_DECREF(seq); PyErr_SetString(PyExc_TypeError, "tensor values must be Python floats"); return false; }
        out[(size_t) i] = (float) PyFloat_AS_DOUBLE(it);
    }
    Py_DECREF(seq);
    return true;
}

static PyObject * floats_to_list(const float * v, size_t n) {
    PyObject * res = PyList_New((Py_ssize_t) n);
    if (!res) return nullptr;
    for (size_t i = 0; i < n; i++) PyList_SET_ITEM(res, (Py_ssize_t) i, PyFloat_FromDouble((double) v[i]));
    return res;
}

static b200_extra_t * extra_for(const char * path) {
    std::lock_guard<std::mutex> lk(g_mu);
    auto it = g_extra.find(path);
    if (it != g_extra.end()) return it->second;
    b200_extra_t * e = nullptr;
    if (b200_extra_load(path, env_int("B200_DEVICE", 0), &e) != 0) return nullptr;
    g_extra[path] = e;
    return e;
}

// Detach the loaded slice and free it once every in-flight call has dropped its reference (GIL released by the caller).
static void retire_slice() {
    SlicePtr old;
    { std::lock_guard<std::mutex> lk(g_mu); old.swap(g_slice); }
    while (old && old.use_count() > 1) std::this_thread::sleep_for(std::chrono::microseconds(200));
    old.reset();                                          // last reference: b200_slice_unload runs here
}

// ---- node side ---------------------------------------------------------------------------------------------
static PyObject * py_load_slice(PyObject *, PyObject * args, PyObject * kwargs) {
    const char * path;
    int n_ctx = 0, device = -1, n_sessions = 0;
    static const char * kw[] = {"path", "n_ctx", "device", "n_sessions", nullptr};
    if (!PyArg_ParseTupleAndKeywords(args, kwargs, "s|iii", (char **) kw, &path, &n_ctx, &device, &n_sessions)) return nullptr;
    if (n_ctx <= 0) n_ctx = env_int("B200_N_CTX", 0);
    if (device < 0) device = env_int("B200_DEVICE", 0);
    if (n_sessions <= 0) n_sessions = env_int("B200_SESSIONS", 1);
    b200_slice_t * s = nullptr;
    int rc;
    Py_BEGIN_ALLOW_THREADS
    // the old slice goes first (the reference leaks it, line 2006): peak HBM is one slice, not two
    retire_slice();
    rc = b200_slice_load_ex(path, device, n_ctx, n_sessions, &s);
    Py_END_ALLOW_THREADS
    if (rc) return raise_b200("load_slice");
    SlicePtr fresh = std::make_shared<SliceRef>(s), old;
    { std::lock_guard<std::mutex> lk(g_mu); old.swap(g_slice); g_slice = fresh; }
    Py_BEGIN_ALLOW_THREADS
    old.reset();                                          // a concurrent load_slice slipped one in: free it too
    Py_END_ALLOW_THREADS
    return PyLong_FromLong(0);
}

static PyObject * py_unload_slice(PyObject *, PyObject *) {
    Py_BEGIN_ALLOW_THREADS
    retire_slice();
    Py_END_ALLOW_THREADS
    return PyLong_FromLong(0);
}

static PyObject * py_clear_context(PyObject *, PyObject *) {
    SlicePtr sp = current_slice();
    int rc = 0;
    Py_BEGIN_ALLOW_THREADS
    if (sp) rc = b200_slice_clear(sp->h);
    sp.reset();
    Py_END_ALLOW_THREADS
    return PyLong_FromLong(rc != 0 ? 1 : 0);
}

// slice_info() -> dict (additive): what the node reports about the slice it serves
static PyObject * py_slice_info(PyObject *, PyObject *) {
    SlicePtr sp = current_slice();
    if (!sp) Py_RETURN_NONE;
    b200_slice_info_t i;
    if (b200_slice_info(sp->h, &i)) return raise_b200("slice_info");
    return Py_BuildValue("{s:i,s:i,s:i,s:i,s:i,s:i,s:i,s:i,s:i,s:L}", "n_embd", i.n_embd, "n_head", i.n_head, "n_ff", i.n_ff,
                         "n_layer", i.n_layer, "first_layer", i.first_layer, "n_ctx", i.n_ctx, "n_past", i.n_past,
                         "device", i.device, "n_sessions", b200_session_count(sp->h), "weight_bytes", (long long) i.weight_bytes);
}

static int forward_vec(const SlicePtr & sp, std::vector<float> & x, std::vector<float> & y) {
    b200_slice_info_t info;
    if (!sp || b200_slice_info(sp->h, &info)) return -1;
    const int n_tokens = (int)(x.size() / (size_t) info.n_embd);       // N = len / n_embd (tensor_processor.cpp:1526)
    y.resize((size_t) n_tokens * info.n_embd);
    return b200_slice_forward(sp->h, x.data(), n_tokens, y.data());
}

static PyObject * py_propagate_forward(PyObject *, PyObject * args) {
    PyObject * values;
    if (!PyArg_ParseTuple(args, "O", &values)) return nullptr;
    SlicePtr sp = current_slice();
    if (!sp) { PyErr_SetString(PyExc_RuntimeError, "propagate_forward: no slice loaded"); return nullptr; }
    std::vector<float> x, y;
    if (!list_to_floats(values, x)) return nullptr;
    int rc;
    Py_BEGIN_ALLOW_THREADS
    rc = forward_vec(sp, x, y);
    sp.reset();
    Py_END_ALLOW_THREADS
    if (rc != 0) return PyLong_FromLong(rc);                            // like the reference: an int status (line 2148-2151)
    return floats_to_list(y.data(), y.size());
}

static PyObject * py_propagate_forward_buffer(PyObject *, PyObject * args) {
    PyObject * values;
    if (!PyArg_ParseTuple(args, "O", &values)) return nullptr;
    SlicePtr sp = current_slice();
    if (!sp) { PyErr_SetString(PyExc_RuntimeError, "propagate_forward: no slice loaded"); return nullptr; }
    std::vector<float> x, y;
    if (!list_to_floats(values, x)) return nullptr;
    int rc; std::string err;
    Py_BEGIN_ALLOW_THREADS
    rc = forward_vec(sp, x, y);
    if (rc) err = b200_last_error();
    sp.reset();
    Py_END_ALLOW_THREADS
    if (rc != 0) { PyErr_Format(PyExc_RuntimeError, "propagate_forward: %s", err.c_str()); return nullptr; }
    return PyBytes_FromStringAndSize((const char *) y.data(), (Py_ssize_t)(y.size() * sizeof(float)));
}

// ---- additive: several sequences on one node (n_sessions contexts over the same weights) ------------------
// propagate_forward_session(session, float32 bytes-like) -> bytes        tokens of ONE session
// propagate_forward_batch([sessions], float32 bytes-like) -> bytes       one token for EACH listed session, one pass
// propagate_forward_mixed([sessions], [n_tokens], float32 bytes-like) -> bytes
//                                                 n_tokens[i] tokens of sessions[i], segments back to back, one pass
// clear_session(session)  (-1 = all)
static PyObject * py_propagate_forward_session(PyObject *, PyObject * args) {
    int session; PyObject * values;
    if (!PyArg_ParseTuple(args, "iO", &session, &values)) return nullptr;
    SlicePtr sp = current_slice();
    if (!sp) { PyErr_SetString(PyExc_RuntimeError, "propagate_forward_session: no slice loaded"); return nullptr; }
    std::vector<float> x, y;
    if (!list_to_floats(values, x)) return nullptr;
    b200_slice_info_t info;
    if (b200_slice_info(sp->h, &info)) return raise_b200("propagate_forward_session");
    const int n_tokens = (int)(x.size() / (size_t) info.n_embd);
    y.resize((size_t) n_tokens * info.n_embd);
    int rc; std::string err;
    Py_BEGIN_ALLOW_THREADS
    rc = b200_session_forward(sp->h, session, x.data(), n_tokens, y.data());
    if (rc) err = b200_last_error();
    sp.reset();
    Py_END_ALLOW_THREADS
    if (rc) { PyErr_Format(PyExc_RuntimeError, "propagate_forward_session: %s", err.c_str()); return nullptr; }
    return PyBytes_FromStringAndSize((const char *) y.data(), (Py_ssize_t)(y.size() * sizeof(float)));
}

static bool list_to_ints(PyObject * list, const char * what, std::vector<int> & out) {
    if (!PyList_Check(list)) { PyErr_Format(PyExc_TypeError, "%s must be a list of int", what); return false; }
    out.resize((size_t) PyList_Size(list));
    for (size_t i = 0; i < out.size(); i++) {
        const long v = PyLong_AsLong(PyList_GetItem(list, (Py_ssize_t) i));
        if (v == -1 && PyErr_Occurred()) return false;
        out[i] = (int) v;
    }
    return true;
}

static PyObject * py_propagate_forward_batch(PyObject *, PyObject * args) {
    PyObject * sessions, * values;
    if (!PyArg_ParseTuple(args, "OO", &sessions, &values)) return nullptr;
    SlicePtr sp = current_slice();
    if (!sp) { PyErr_SetString(PyExc_RuntimeError, "propagate_forward_batch: no slice loaded"); return nullptr; }
    std::vector<int> ids;
    if (!list_to_ints(sessions, "propagate_forward_batch: sessions", ids)) return nullptr;
    std::vector<float> x, y;
    if (!list_to_floats(values, x)) return nullptr;
    b200_slice_info_t info;
    if (b200_slice_info(sp->h, &info)) return raise_b200("propagate_forward_batch");
    if (x.size() != ids.size() * (size_t) info.n_embd) {
        PyErr_SetString(PyExc_ValueError, "propagate_forward_batch: need exactly one n_embd row per listed session");
        return nullptr;
    }
    y.resize(x.size());
    int rc; std::string err;
    Py_BEGIN_ALLOW_THREADS
    rc = b200_batch_forward(sp->h, ids.data(), (int) ids.size(), x.data(), y.data());
    if (rc) err = b200_last_error();
    sp.reset();
    Py_END_ALLOW_THREADS
    if (rc) { PyErr_Format(PyExc_RuntimeError, "propagate_forward_batch: %s", err.c_str()); return nullptr; }
    return PyBytes_FromStringAndSize((const char *) y.data(), (Py_ssize_t)(y.size() * sizeof(float)));
}

static PyObject * py_propagate_forward_mixed(PyObject *, PyObject * args) {
    PyObject * sessions, * counts, * values;
    if (!PyArg_ParseTuple(args, "OOO", &sessions, &counts, &values)) return nullptr;
    SlicePtr sp = current_slice();
    if (!sp) { PyErr_SetString(PyExc_RuntimeError, "propagate_forward_mixed: no slice loaded"); return nullptr; }
    std::vector<int> ids, lens;
    if (!list_to_ints(sessions, "propagate_forward_mixed: sessions", ids) || !list_to_ints(counts, "propagate_forward_mixed: n_tokens", lens))
        return nullptr;
    if (ids.size() != lens.size()) {
        PyErr_SetString(PyExc_ValueError, "propagate_forward_mixed: need one token count per listed session");
        return nullptr;
    }
    std::vector<float> x, y;
    if (!list_to_floats(values, x)) return nullptr;
    b200_slice_info_t info;
    if (b200_slice_info(sp->h, &info)) return raise_b200("propagate_forward_mixed");
    long long rows = 0;
    for (int n : lens) rows += n;
    if (rows < 0 || x.size() != (size_t) rows * info.n_embd) {
        PyErr_SetString(PyExc_ValueError, "propagate_forward_mixed: need exactly sum(n_tokens) rows of n_embd floats");
        return nullptr;
    }
    y.resize(x.size());
    int rc; std::string err;
    Py_BEGIN_ALLOW_THREADS
    rc = b200_mixed_forward(sp->h, ids.data(), lens.data(), (int) ids.size(), x.data(), y.data());
    if (rc) err = b200_last_error();
    sp.reset();
    Py_END_ALLOW_THREADS
    if (rc) { PyErr_Format(PyExc_RuntimeError, "propagate_forward_mixed: %s", err.c_str()); return nullptr; }
    return PyBytes_FromStringAndSize((const char *) y.data(), (Py_ssize_t)(y.size() * sizeof(float)));
}

static PyObject * py_clear_session(PyObject *, PyObject * args) {
    int session;
    if (!PyArg_ParseTuple(args, "i", &session)) return nullptr;
    SlicePtr sp = current_slice();
    if (sp && b200_session_clear(sp->h, session) != 0) return raise_b200("clear_session");
    return PyLong_FromLong(0);
}

// ---- client side ---------------------------------------------------------------------------------------------
static PyObject * py_tokenize_prompt(PyObject *, PyObject * args) {
    const char * path, * prompt;
    if (!PyArg_ParseTuple(args, "ss", &path, &prompt)) return nullptr;
    b200_extra_t * e = extra_for(path);
    if (!e) return raise_b200("tokenize_prompt");
    std::vector<int32_t> ids(4096);
    int n = b200_extra_tokenize(e, prompt, ids.data(), (int) ids.size());
    if (n > (int) ids.size()) { ids.resize((size_t) n); n = b200_extra_tokenize(e, prompt, ids.data(), n); }
    PyObject * res = PyList_New(n);
    for (int i = 0; i < n; i++) PyList_SET_ITEM(res, i, PyLong_FromLong(ids[(size_t) i]));
    return res;
}

static PyObject * py_prepare_embeddings(PyObject *, PyObject * args) {
    const char * path; PyObject * tokens;
    if (!PyArg_ParseTuple(args, "sO", &path, &tokens)) return nullptr;
    b200_extra_t * e = extra_for(path);
    if (!e) return raise_b200("prepare_embeddings");
    PyObject * seq = PySequence_Fast(tokens, "expected a list of token ids");
    if (!seq) return nullptr;
    std::vector<int32_t> ids((size_t) PySequence_Fast_GET_SIZE(seq));
    for (size_t i = 0; i < ids.size(); i++) {
        PyObject * it = PySequence_Fast_GET_ITEM(seq, (Py_ssize_t) i);
        if (!PyLong_Check(it)) { Py_DECREF(seq); PyErr_SetString(PyExc_TypeError, "token ids must be ints"); return nullptr; }
        ids[i] = (int32_t) PyLong_AsLong(it);
    }
    Py_DECREF(seq);
    int n_vocab = 0, n_embd = 0;
    b200_extra_dims(e, &n_vocab, &n_embd);
    std::vector<float> emb(ids.size() * (size_t) n_embd);
    if (!ids.empty()) {
        int rc;
        Py_BEGIN_ALLOW_THREADS
        rc = b200_extra_embed(e, ids.data(), (int) ids.size(), emb.data());
        Py_END_ALLOW_THREADS
        if (rc) return raise_b200("prepare_embeddings");
    }
    return floats_to_list(emb.data(), emb.size());
}

static PyObject * py_get_logits(PyObject *, PyObject * args) {
    const char * path; PyObject * values; int all_logits;
    if (!PyArg_ParseTuple(args, "sOp", &path, &values, &all_logits)) return nullptr;
    b200_extra_t * e = extra_for(path);
    if (!e) return raise_b200("get_logits");
    std::vector<float> x;
    if (!list_to_floats(values, x)) return nullptr;
    int n_vocab = 0, n_embd = 0;
    b200_extra_dims(e, &n_vocab, &n_embd);
    const int n_tokens = (int)(x.size() / (size_t) n_embd);
    if (n_tokens <= 0) { PyErr_SetString(PyExc_ValueError, "get_logits: empty embeddings"); return nullptr; }
    std::vector<float> logits((size_t)(all_logits ? n_tokens : 1) * n_vocab);
    int rc;
    Py_BEGIN_ALLOW_THREADS
    rc = b200_extra_logits(e, x.data(), n_tokens, all_logits, logits.data());
    Py_END_ALLOW_THREADS
    if (rc) return raise_b200("get_logits");
    return floats_to_list(logits.data(), logits.size());
}

static PyObject * py_get_next_token(PyObject *, PyObject * args) {
    const char * path; PyObject * values;
    if (!PyArg_ParseTuple(args, "sO", &path, &values)) return nullptr;
    b200_extra_t * e = extra_for(path);
    if (!e) return raise_b200("get_next_token");
    std::vector<float> x;
    if (!list_to_floats(values, x)) return nullptr;
    int n_vocab = 0, n_embd = 0;
    b200_extra_dims(e, &n_vocab, &n_embd);
    int32_t tok = 0; int rc;
    Py_BEGIN_ALLOW_THREADS
    rc = b200_extra_next_token(e, x.data(), (int)(x.size() / (size_t) n_embd), &tok);
    Py_END_ALLOW_THREADS
    if (rc) return raise_b200("get_next_token");
    return PyLong_FromLong(tok);
}

static PyObject * py_decode_token(PyObject *, PyObject * args) {
    const char * path; int id;
    if (!PyArg_ParseTuple(args, "si", &path, &id)) return nullptr;
    b200_extra_t * e = extra_for(path);
    if (!e) return raise_b200("decode_token");
    int len = 0;
    const char * text = b200_extra_token_text(e, id, &len);
    if (!text) { PyErr_SetString(PyExc_IndexError, "decode_token: token id out of range"); return nullptr; }
    return PyUnicode_DecodeUTF8(text, len, "replace");
}

static PyMethodDef Methods[] = {
    {"load_slice", (PyCFunction)(void (*)(void)) py_load_slice, METH_VARARGS | METH_KEYWORDS, "load_slice(path, n_ctx=0, device=-1, n_sessions=0): load the slice's layers onto the GPU"},
    {"slice_info", py_slice_info, METH_NOARGS, "dict describing the loaded slice (None if none)"},
    {"unload_slice", py_unload_slice, METH_VARARGS, "Unload the slice currently loaded"},
    {"clear_context", py_clear_context, METH_VARARGS, "Clear cached keys and values"},
    {"tokenize_prompt", py_tokenize_prompt, METH_VARARGS, "Convert a text prompt into a list of tokens"},
    {"prepare_embeddings", py_prepare_embeddings, METH_VARARGS, "Embed tokens for the first slice"},
    {"propagate_forward", py_propagate_forward, METH_VARARGS, "Propagate an embeddings vector through the layers of the slice"},
    {"propagate_forward_buffer", py_propagate_forward_buffer, METH_VARARGS, "Same, float32 bytes-like in, bytes out"},
    {"propagate_forward_session", py_propagate_forward_session, METH_VARARGS, "(session, float32 buffer) -> bytes: tokens of one of B200_SESSIONS contexts"},
    {"propagate_forward_batch", py_propagate_forward_batch, METH_VARARGS, "([sessions], float32 buffer) -> bytes: one token for each listed session in one pass"},
    {"propagate_forward_mixed", py_propagate_forward_mixed, METH_VARARGS,
     "([sessions], [n_tokens], float32 buffer) -> bytes: n_tokens[i] tokens of sessions[i], segments back to back, in one pass"},
    {"clear_session", py_clear_session, METH_VARARGS, "Clear one session's context (-1: all)"},
    {"get_logits", py_get_logits, METH_VARARGS, "Apply the output layers to embeddings to get logits"},
    {"get_next_token", py_get_next_token, METH_VARARGS, "Greedy next token"},
    {"decode_token", py_decode_token, METH_VARARGS, "Convert a token id to text"},
    {nullptr, nullptr, 0, nullptr}};

static struct PyModuleDef llmmodule = {PyModuleDef_HEAD_INIT, "llm", "B200 slice runtime behind DistributedLLM's llm module API", -1, Methods};

PyMODINIT_FUNC PyInit_llm(void) { return PyModule_Create(&llmmodule); }
