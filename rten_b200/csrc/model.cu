// Minimal graph executor behind the C ABI (include/rten_b200.h: rten_b200_model_*): what RTen's `Model::load` +
// `Graph::run_plan` do around the operators of this library (src/model.rs, src/graph.rs:880-1286), restated for the
// hot-path operator set:
//   load : ONNX bytes -> nodes + initialisers (onnx_reader.cu; int64 tensors become i32 like rten's loader does) ->
//          constants uploaded to HBM once -> load-time fusions (Conv + Relu, MatMul + Add(bias): the subset of
//          src/optimize.rs the models need) -> weights prepacked once (`Operator::prepack`, src/graph.rs:488-565).
//   run  : the nodes in topological (file) order, one C-ABI operator call each; temporaries are reference counted and
//          returned to the context pool after their last consumer (src/graph.rs:1100-1180); an operator that can run in
//          place does so when the executor holds the last reference to its input (src/graph.rs:973-1049); shape-only
//          operators (Reshape, Flatten, Squeeze, Unsqueeze, Transpose, Identity) are views -- no kernel, no copy.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <map>
#include <memory>
#include <set>
#include <string>
#include <vector>

#include "api_util.h"
#include "onnx_reader.h"
#include "rowops.h"

using namespace rtb;

namespace {

enum ValueKind { V_UNSET = 0, V_CONST, V_INPUT, V_TEMP };

struct ValueSlot {
    std::string name;
    ValueKind kind = V_UNSET;
    rten_tensor t{};
    bool has_host_ints = false;       // shape-like constant (int64 in the file): usable by Reshape / axes inputs
    std::vector<int64_t> host_ints;
    // run state
    int root = -1;        // value that owns the allocation (self for owners)
    int pending = 0;      // consumers still to run
    int views = 0;        // live views of this owner
    bool live = false;
    bool owned = false;   // allocation belongs to the executor (pool)
};

struct OpNode {
    onnx::Node n;
    std::vector<int> in, out;  // value ids (-1 = absent optional input)
    rten_packed* packed = nullptr;
    int activation = 0;        // fused Relu
    int bias_value = -1;       // fused Add(bias) of a MatMul
};

}  // namespace

struct rten_model {
    rten_ctx* ctx = nullptr;
    std::vector<ValueSlot> values;
    std::map<std::string, int> by_name;
    std::vector<OpNode> nodes;
    std::vector<int> inputs, outputs;
    std::vector<void*> const_allocs;
    float* one = nullptr;  // device scalar 1.0f (Cast int32 -> float through cast_scale)
    std::string summary;

    int value_id(const std::string& name) {
        if (name.empty()) return -1;
        auto it = by_name.find(name);
        if (it != by_name.end()) return it->second;
        ValueSlot v;
        v.name = name;
        values.push_back(v);
        by_name[name] = (int)values.size() - 1;
        return (int)values.size() - 1;
    }
};

namespace {

rten_status mfail(rten_ctx* ctx, rten_status st, const std::string& msg) {
    if (ctx) ctx->err = msg;
    return st;
}

int dtype_of(int32_t onnx_dt) {
    switch (onnx_dt) {
        case onnx::DT_FLOAT: return RTEN_F32;
        case onnx::DT_INT32: case onnx::DT_INT64: case onnx::DT_BOOL: return RTEN_I32;
        case onnx::DT_INT8: return RTEN_I8;
        case onnx::DT_UINT8: return RTEN_U8;
        default: return -1;
    }
}

// initialiser / Constant tensor -> device constant (int64 narrowed to i32, the only integer width of the path)
rten_status upload_constant(rten_model* m, const onnx::Tensor& t, ValueSlot* v) {
    rten_ctx* ctx = m->ctx;
    const int dt = dtype_of(t.data_type);
    if (dt < 0) return mfail(ctx, RTEN_ERR_UNSUPPORTED_TYPE, "unsupported tensor type in initializer '" + t.name + "'");
    if (t.external) return mfail(ctx, RTEN_ERR_UNSUPPORTED_VALUE, "external tensor data is not supported ('" + t.name + "')");
    if ((int)t.dims.size() > RTEN_MAX_DIMS) return mfail(ctx, RTEN_ERR_INVALID_VALUE, "tensor rank out of range");
    const int64_t n = t.numel();
    std::vector<uint8_t> conv;
    const uint8_t* src = t.data.data();
    if (t.data_type == onnx::DT_INT64) {
        conv.resize((size_t)n * 4);
        v->has_host_ints = true;
        v->host_ints.resize((size_t)n);
        for (int64_t i = 0; i < n; i++) {
            int64_t x;
            memcpy(&x, t.data.data() + 8 * i, 8);
            v->host_ints[(size_t)i] = x;
            const int32_t y = (int32_t)std::max<int64_t>(INT32_MIN, std::min<int64_t>(INT32_MAX, x));
            memcpy(conv.data() + 4 * i, &y, 4);
        }
        src = conv.data();
    } else if (t.data_type == onnx::DT_BOOL) {
        conv.resize((size_t)n * 4);
        for (int64_t i = 0; i < n; i++) {
            const int32_t y = t.data[(size_t)i] ? 1 : 0;
            memcpy(conv.data() + 4 * i, &y, 4);
        }
        src = conv.data();
    } else if (t.data_type == onnx::DT_INT32) {
        v->has_host_ints = true;
        v->host_ints.resize((size_t)n);
        for (int64_t i = 0; i < n; i++) {
            int32_t x;
            memcpy(&x, t.data.data() + 4 * i, 4);
            v->host_ints[(size_t)i] = x;
        }
    }
    const size_t bytes = (size_t)n * dtype_size(dt);
    void* d = nullptr;
    RTB_TRY(pool_alloc(ctx, bytes ? bytes : 16, &d));
    m->const_allocs.push_back(d);
    if (bytes) RTB_CUDA(ctx, cudaMemcpyAsync(d, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    RTB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // `conv` / the file buffer may go away
    v->kind = V_CONST;
    v->t.data = d;
    v->t.dtype = dt;
    v->t.ndim = (int)t.dims.size();
    for (int i = 0; i < v->t.ndim; i++) v->t.shape[i] = t.dims[(size_t)i];
    set_contiguous(&v->t);
    v->t.device = ctx->device;
    return RTEN_OK;
}

const std::set<std::string>& supported_ops() {
    static const std::set<std::string> s = {
        "Conv", "Relu", "MaxPool", "GlobalAveragePool", "ReduceMean", "Reshape", "Flatten", "Squeeze", "Unsqueeze", "Transpose",
        "Identity", "Gemm", "MatMul", "Add", "Mul", "Softmax", "LayerNormalization", "Gelu", "Erf", "Gather",
        "DynamicQuantizeLinear", "MatMulInteger", "ConvInteger", "Cast", "Attention", "Constant"};
    return s;
}

bool is_view_op(const std::string& op) {
    return op == "Reshape" || op == "Flatten" || op == "Squeeze" || op == "Unsqueeze" || op == "Transpose" || op == "Identity";
}
bool is_in_place_op(const std::string& op) { return op == "Relu" || op == "Gelu" || op == "Erf" || op == "Softmax"; }

rten_status fill_conv_params(rten_ctx* ctx, const onnx::Node& n, rten_conv_params* p) {
    memset(p, 0, sizeof(*p));
    const onnx::Attribute* ap = n.attr("auto_pad");
    if (ap && (ap->s == "SAME_UPPER" || ap->s == "SAME_LOWER")) p->auto_pad_same = 1;
    if (ap && ap->s == "SAME_LOWER") return mfail(ctx, RTEN_ERR_UNSUPPORTED_VALUE, "auto_pad SAME_LOWER is not supported");
    const std::vector<int64_t> pads = n.attr_ints("pads"), st = n.attr_ints("strides"), dl = n.attr_ints("dilations");
    if (pads.size() == 4) {  // ONNX [top, left, bottom, right]
        for (int i = 0; i < 4; i++) p->pads[i] = (int32_t)pads[(size_t)i];
    } else if (pads.size() == 2) {
        p->pads[0] = (int32_t)pads[0];
        p->pads[1] = (int32_t)pads[1];
    } else if (!pads.empty()) {
        return mfail(ctx, RTEN_ERR_INVALID_VALUE, "Wrong number of pad values");
    }
    p->groups = (int32_t)n.attr_i("group", 1);
    p->n_strides = st.empty() ? 2 : (int32_t)st.size();
    p->n_dilations = dl.empty() ? 2 : (int32_t)dl.size();
    for (int i = 0; i < 2; i++) {
        p->strides[i] = i < (int)st.size() ? (int32_t)st[(size_t)i] : 1;
        p->dilations[i] = i < (int)dl.size() ? (int32_t)dl[(size_t)i] : 1;
    }
    return RTEN_OK;
}

}  // namespace

extern "C" {

rten_status rten_b200_onnx_summary(const void* bytes, size_t len, char* json_out, size_t cap, size_t* needed) {
    onnx::Model m;
    std::string err;
    if (!onnx::decode_model(reinterpret_cast<const uint8_t*>(bytes), len, &m, &err)) return RTEN_ERR_INVALID_VALUE;
    const std::string s = onnx::summary_json(m);
    if (needed) *needed = s.size() + 1;
    if (json_out && cap) {
        const size_t n = std::min(cap - 1, s.size());
        memcpy(json_out, s.data(), n);
        json_out[n] = 0;
    }
    return RTEN_OK;
}

void rten_b200_model_free(rten_model* m) {
    if (!m) return;
    for (OpNode& n : m->nodes)
        if (n.packed) rten_b200_packed_free(m->ctx, n.packed);
    for (void* p : m->const_allocs) pool_free(m->ctx, p);
    delete m;
}

rten_status rten_b200_model_load(rten_ctx* ctx, const void* bytes, size_t len, rten_model** out) {
    if (!ctx || !out || (!bytes && len)) return RTEN_ERR_INVALID_VALUE;
    *out = nullptr;
    cudaSetDevice(ctx->device);
    onnx::Model om;
    std::string err;
    if (!onnx::decode_model(reinterpret_cast<const uint8_t*>(bytes), len, &om, &err)) return mfail(ctx, RTEN_ERR_INVALID_VALUE, "ONNX decode failed: " + err);
    if (!om.has_graph) return mfail(ctx, RTEN_ERR_INVALID_VALUE, "ONNX model has no graph");
    std::unique_ptr<rten_model, void (*)(rten_model*)> m(new rten_model(), rten_b200_model_free);
    m->ctx = ctx;
    m->summary = onnx::summary_json(om);
    // constants
    for (const onnx::Tensor& t : om.graph.initializers) {
        const int id = m->value_id(t.name);
        RTB_TRY(upload_constant(m.get(), t, &m->values[(size_t)id]));
    }
    {
        void* d = nullptr;
        RTB_TRY(pool_alloc(ctx, 16, &d));
        m->const_allocs.push_back(d);
        const float one = 1.0f;
        RTB_CUDA(ctx, cudaMemcpy(d, &one, 4, cudaMemcpyHostToDevice));
        m->one = (float*)d;
    }
    for (const onnx::ValueInfo& vi : om.graph.inputs) {
        const int id = m->value_id(vi.name);
        if (m->values[(size_t)id].kind == V_CONST) continue;  // (old exporters list initialisers among the inputs)
        m->values[(size_t)id].kind = V_INPUT;
        m->inputs.push_back(id);
    }
    // nodes (the file order is topological: onnx.proto3 requires it, like src/model.rs relies on)
    for (const onnx::Node& n : om.graph.nodes) {
        if (!n.domain.empty() && n.domain != "ai.onnx" && n.domain != "com.microsoft")
            return mfail(ctx, RTEN_ERR_UNSUPPORTED_VALUE, "unsupported operator domain '" + n.domain + "'");
        if (!supported_ops().count(n.op_type)) return mfail(ctx, RTEN_ERR_UNSUPPORTED_VALUE, "unsupported operator " + n.op_type);
        if (n.op_type == "Constant") {
            const onnx::Attribute* a = n.attr("value");
            if (!a || !a->has_t || n.outputs.size() != 1) return mfail(ctx, RTEN_ERR_UNSUPPORTED_VALUE, "Constant without a tensor value");
            onnx::Tensor t = a->t;
            t.name = n.outputs[0];
            const int id = m->value_id(t.name);
            RTB_TRY(upload_constant(m.get(), t, &m->values[(size_t)id]));
            continue;
        }
        OpNode on;
        on.n = n;
        for (const std::string& s : n.inputs) {
            const int id = m->value_id(s);
            if (id >= 0 && m->values[(size_t)id].kind == V_UNSET)
                return mfail(ctx, RTEN_ERR_INVALID_VALUE, "node '" + n.name + "' (" + n.op_type + ") reads '" + s + "' before it is produced");
            on.in.push_back(id);
        }
        for (const std::string& s : n.outputs) {
            const int id = m->value_id(s);
            if (id >= 0) m->values[(size_t)id].kind = V_TEMP;
            on.out.push_back(id);
        }
        m->nodes.push_back(on);
    }
    for (const onnx::ValueInfo& vi : om.graph.outputs) {
        auto it = m->by_name.find(vi.name);
        if (it == m->by_name.end() || m->values[(size_t)it->second].kind == V_UNSET)
            return mfail(ctx, RTEN_ERR_INVALID_VALUE, "graph output '" + vi.name + "' is never produced");
        m->outputs.push_back(it->second);
    }
    // ---- load-time fusions (src/optimize.rs: the two patterns the hot-path models contain)
    auto consumers = [&](int vid) {
        int c = 0;
        for (const OpNode& o : m->nodes)
            for (int i : o.in)
                if (i == vid) c++;
        for (int o : m->outputs)
            if (o == vid) c++;
        return c;
    };
    for (size_t i = 0; i + 1 < m->nodes.size(); i++) {
        OpNode& a = m->nodes[i];
        if (a.out.size() != 1 || consumers(a.out[0]) != 1) continue;
        // the single consumer
        size_t j = i + 1;
        for (; j < m->nodes.size(); j++)
            if (std::find(m->nodes[j].in.begin(), m->nodes[j].in.end(), a.out[0]) != m->nodes[j].in.end()) break;
        if (j == m->nodes.size()) continue;
        OpNode& b = m->nodes[j];
        if (a.n.op_type == "Conv" && b.n.op_type == "Relu" && a.activation == 0) {
            a.activation = 1;  // Relu in the convolution epilogue
            a.out = b.out;
            m->nodes.erase(m->nodes.begin() + (long)j);
        } else if (a.n.op_type == "MatMul" && b.n.op_type == "Add" && a.bias_value < 0 && b.in.size() == 2) {
            // MatMul + Add(constant vector over the last axis) -> FusedMatMul with a row bias (MatMulAddFusion)
            const int other = b.in[0] == a.out[0] ? b.in[1] : b.in[0];
            const ValueSlot& bv = m->values[(size_t)other];
            const ValueSlot& wv = m->values[(size_t)a.in[1]];
            if (bv.kind == V_CONST && bv.t.dtype == RTEN_F32 && bv.t.ndim == 1 && wv.t.ndim >= 2 && wv.kind == V_CONST &&
                bv.t.shape[0] == wv.t.shape[wv.t.ndim - 1]) {
                a.bias_value = other;
                a.out = b.out;
                m->nodes.erase(m->nodes.begin() + (long)j);
            }
        }
    }
    // ---- prepack constant weights once (Operator::prepack at load, src/graph.rs:488-565)
    for (OpNode& o : m->nodes) {
        const std::string& op = o.n.op_type;
        if ((op == "Conv" || op == "ConvInteger") && o.in.size() >= 2 && m->values[(size_t)o.in[1]].kind == V_CONST &&
            m->values[(size_t)o.in[1]].t.ndim == 4) {
            RTB_TRY(rten_b200_prepack_conv_weight(ctx, &m->values[(size_t)o.in[1]].t, (int)o.n.attr_i("group", 1), &o.packed));
        } else if ((op == "MatMul" || op == "MatMulInteger") && o.in.size() >= 2 && m->values[(size_t)o.in[1]].kind == V_CONST &&
                   m->values[(size_t)o.in[1]].t.ndim == 2) {
            RTB_TRY(rten_b200_prepack_b(ctx, &m->values[(size_t)o.in[1]].t, &o.packed));
        }
    }
    RTB_TRY(rten_b200_sync(ctx));
    *out = m.release();
    return RTEN_OK;
}

int32_t rten_b200_model_num_inputs(const rten_model* m) { return m ? (int32_t)m->inputs.size() : 0; }
int32_t rten_b200_model_num_outputs(const rten_model* m) { return m ? (int32_t)m->outputs.size() : 0; }
const char* rten_b200_model_input_name(const rten_model* m, int32_t i) {
    return (m && i >= 0 && i < (int32_t)m->inputs.size()) ? m->values[(size_t)m->inputs[(size_t)i]].name.c_str() : nullptr;
}
const char* rten_b200_model_output_name(const rten_model* m, int32_t i) {
    return (m && i >= 0 && i < (int32_t)m->outputs.size()) ? m->values[(size_t)m->outputs[(size_t)i]].name.c_str() : nullptr;
}
int32_t rten_b200_model_num_nodes(const rten_model* m) { return m ? (int32_t)m->nodes.size() : 0; }
const char* rten_b200_model_node_op(const rten_model* m, int32_t i) {
    return (m && i >= 0 && i < (int32_t)m->nodes.size()) ? m->nodes[(size_t)i].n.op_type.c_str() : nullptr;
}
const char* rten_b200_model_summary(const rten_model* m) { return m ? m->summary.c_str() : nullptr; }

}  // extern "C"

// ------------------------------------------------------------------------------------------
// run
// ------------------------------------------------------------------------------------------
namespace {

struct Runner {
    rten_model* m;
    rten_ctx* ctx;
    std::set<int> keep;  // requested outputs: never released, never overwritten in place

    ValueSlot& V(int id) { return m->values[(size_t)id]; }
    int root_of(int id) { return V(id).root < 0 ? id : V(id).root; }

    void release_owner(int id) {
        ValueSlot& v = V(id);
        if (v.owned && v.live && v.pending <= 0 && v.views <= 0 && !keep.count(id)) {
            pool_free(ctx, v.t.data);
            v.live = false;
            v.owned = false;
            v.t.data = nullptr;
        }
    }
    void consumed(int id) {
        if (id < 0) return;
        ValueSlot& v = V(id);
        if (v.kind != V_TEMP) return;
        v.pending--;
        if (v.pending > 0) return;
        const int r = root_of(id);
        if (r != id) {
            if (!keep.count(id)) {
                V(r).views--;
                release_owner(r);
            }
        } else {
            release_owner(id);
        }
    }
    void set_owned(int id, const rten_tensor& t) {
        ValueSlot& v = V(id);
        v.t = t;
        v.root = -1;
        v.live = true;
        v.owned = true;
        v.views = 0;
    }
    void set_view(int id, const rten_tensor& t, int src) {
        ValueSlot& v = V(id);
        v.t = t;
        v.live = true;
        v.owned = false;
        const int r = root_of(src);
        if (V(r).kind == V_TEMP && V(r).owned) {
            v.root = r;
            V(r).views++;
        } else {
            v.root = -1;  // view of a constant / graph input: nothing to keep alive
        }
    }

    static bool contiguous(const rten_tensor& t) { return is_contiguous(&t); }

    rten_status make_contiguous(const rten_tensor& src, rten_tensor* dst, bool* allocated) {
        *allocated = false;
        if (contiguous(src)) {
            *dst = src;
            return RTEN_OK;
        }
        rten_tensor c = src;
        set_contiguous(&c);
        void* d = nullptr;
        RTB_TRY(pool_alloc(ctx, (size_t)std::max<int64_t>(numel(&src), 1) * dtype_size(src.dtype), &d));
        c.data = d;
        rten_status st = rten_b200_copy(ctx, &src, &c);
        if (st != RTEN_OK) {
            pool_free(ctx, d);
            return st;
        }
        *dst = c;
        *allocated = true;
        return RTEN_OK;
    }

    rten_status ints_of(int id, std::vector<int64_t>* out) {
        if (id < 0 || !V(id).has_host_ints) return mfail(ctx, RTEN_ERR_UNSUPPORTED_VALUE, "shape-like operator input must be a constant");
        *out = V(id).host_ints;
        return RTEN_OK;
    }

    rten_status run_view(OpNode& o) {
        const std::string& op = o.n.op_type;
        const rten_tensor& x = V(o.in[0]).t;
        rten_tensor y = x;
        int src = o.in[0];
        if (op == "Transpose") {
            std::vector<int64_t> perm = o.n.attr_ints("perm");
            if (perm.empty())
                for (int i = x.ndim - 1; i >= 0; i--) perm.push_back(i);
            if ((int)perm.size() != x.ndim) return mfail(ctx, RTEN_ERR_INVALID_VALUE, "Transpose: perm has the wrong length");
            for (int i = 0; i < x.ndim; i++) {
                const int64_t a = perm[(size_t)i];
                if (a < 0 || a >= x.ndim) return mfail(ctx, RTEN_ERR_INVALID_VALUE, "Transpose: perm entry out of range");
                y.shape[i] = x.shape[a];
                y.strides[i] = x.strides[a];
            }
            set_view(o.out[0], y, src);
            return RTEN_OK;
        }
        if (op == "Identity") {
            set_view(o.out[0], y, src);
            return RTEN_OK;
        }
        // the remaining view operators re-shape: the data must be contiguous first
        rten_tensor c;
        bool alloc = false;
        RTB_TRY(make_contiguous(x, &c, &alloc));
        std::vector<int64_t> shape;
        const int64_t total = numel(&c);
        if (op == "Reshape") {
            std::vector<int64_t> want;
            RTB_TRY(ints_of(o.in.size() > 1 ? o.in[1] : -1, &want));
            int64_t known = 1;
            int infer = -1;
            for (size_t i = 0; i < want.size(); i++) {
                int64_t d = want[i];
                if (d == 0 && !o.n.attr_i("allowzero", 0)) d = (int)i < c.ndim ? c.shape[i] : 0;
                if (d == -1) {
                    if (infer >= 0) return mfail(ctx, RTEN_ERR_INVALID_VALUE, "Multiple dimensions in new shape set to -1");
                    infer = (int)i;
                    d = 1;
                }
                shape.push_back(d);
                known *= d;
            }
            if (infer >= 0) {
                if (known == 0 || total % known) return mfail(ctx, RTEN_ERR_INVALID_VALUE, "Input length must be a multiple of specified dimensions");
                shape[(size_t)infer] = total / known;
            }
        } else if (op == "Flatten") {
            int64_t axis = o.n.attr_i("axis", 1);
            if (axis < 0) axis += c.ndim;
            int64_t a = 1, b = 1;
            for (int i = 0; i < c.ndim; i++) (i < axis ? a : b) *= c.shape[i];
            shape = {a, b};
        } else {  // Squeeze / Unsqueeze: axes attribute (opset < 13) or second input
            std::vector<int64_t> axes = o.n.attr_ints("axes");
            if (axes.empty() && o.in.size() > 1 && o.in[1] >= 0) RTB_TRY(ints_of(o.in[1], &axes));
            if (op == "Squeeze") {
                for (int i = 0; i < c.ndim; i++) {
                    bool drop = axes.empty() ? c.shape[i] == 1 : false;
                    for (int64_t a : axes)
                        if ((a < 0 ? a + c.ndim : a) == i) drop = true;
                    if (!drop) shape.push_back(c.shape[i]);
                }
            } else {
                const int nd = c.ndim + (int)axes.size();
                std::vector<bool> ins((size_t)nd, false);
                for (int64_t a : axes) {
                    const int64_t p = a < 0 ? a + nd : a;
                    if (p < 0 || p >= nd) return mfail(ctx, RTEN_ERR_INVALID_VALUE, "Axes must be in range [-r, r-1]");
                    ins[(size_t)p] = true;
                }
                int k = 0;
                for (int i = 0; i < nd; i++) shape.push_back(ins[(size_t)i] ? 1 : c.shape[k++]);
            }
        }
        int64_t prod = 1;
        for (int64_t d : shape) prod *= d;
        if (prod != total) return mfail(ctx, RTEN_ERR_INVALID_VALUE, "New shape must have same total elements as current shape");
        if ((int)shape.size() > RTEN_MAX_DIMS) return mfail(ctx, RTEN_ERR_INVALID_VALUE, "tensor rank out of range");
        y = c;
        y.ndim = (int)shape.size();
        for (int i = 0; i < y.ndim; i++) y.shape[i] = shape[(size_t)i];
        set_contiguous(&y);
        if (alloc)
            set_owned(o.out[0], y);
        else
            set_view(o.out[0], y, src);
        return RTEN_OK;
    }

    rten_status run_node(OpNode& o) {
        const std::string& op = o.n.op_type;
        auto T = [&](size_t i) -> const rten_tensor* { return (i < o.in.size() && o.in[i] >= 0) ? &V(o.in[i]).t : nullptr; };
        if (!T(0)) return mfail(ctx, RTEN_ERR_MISSING_INPUTS, "missing inputs");
        if (is_view_op(op)) return run_view(o);
        rten_tensor y;
        memset(&y, 0, sizeof(y));
        rten_status st = RTEN_OK;
        // in place when the executor holds the last reference to input 0 (src/graph.rs:973-1049)
        bool in_place = false;
        if (is_in_place_op(op)) {
            ValueSlot& x = V(o.in[0]);
            in_place = x.kind == V_TEMP && x.owned && x.root < 0 && x.pending == 1 && x.views == 0 && !keep.count(o.in[0]) && contiguous(x.t);
            if (in_place) y = x.t;
        }
        if (op == "Conv" || op == "ConvInteger") {
            rten_conv_params p;
            RTB_TRY(fill_conv_params(ctx, o.n, &p));
            if (op == "Conv")
                st = rten_b200_conv2d_ex(ctx, T(0), T(1), o.packed, T(2), &p, nullptr, o.activation, &y);
            else
                st = rten_b200_conv_integer(ctx, T(0), T(1), o.packed, T(2), T(3), nullptr, &p, &y);
        } else if (op == "Relu") {
            st = rten_b200_relu(ctx, T(0), &y);
        } else if (op == "Gelu") {
            const onnx::Attribute* a = o.n.attr("approximate");
            st = rten_b200_gelu(ctx, T(0), (a && a->s == "tanh") ? 1 : 0, &y);
        } else if (op == "Erf") {
            st = rten_b200_erf(ctx, T(0), &y);
        } else if (op == "Softmax") {
            st = rten_b200_softmax(ctx, T(0), nullptr, (int)o.n.attr_i("axis", -1), 0, &y);
        } else if (op == "MaxPool") {
            const std::vector<int64_t> k = o.n.attr_ints("kernel_shape"), pd = o.n.attr_ints("pads"), sd = o.n.attr_ints("strides");
            if (k.size() != 2) return mfail(ctx, RTEN_ERR_UNSUPPORTED_VALUE, "MaxPool: only 2-D kernels are supported");
            int32_t kk[2] = {(int32_t)k[0], (int32_t)k[1]}, pp[4] = {0, 0, 0, 0}, ss[2] = {1, 1};
            for (size_t i = 0; i < pd.size() && i < 4; i++) pp[i] = (int32_t)pd[i];
            for (size_t i = 0; i < sd.size() && i < 2; i++) ss[i] = (int32_t)sd[i];
            st = rten_b200_max_pool(ctx, T(0), kk, pp, ss, &y);
        } else if (op == "GlobalAveragePool" || op == "ReduceMean") {
            const rten_tensor* x = T(0);
            bool keepdims = true;
            if (op == "ReduceMean") {
                std::vector<int64_t> axes = o.n.attr_ints("axes");
                if (axes.empty() && o.in.size() > 1 && o.in[1] >= 0) RTB_TRY(ints_of(o.in[1], &axes));
                keepdims = o.n.attr_i("keepdims", 1) != 0;
                bool spatial = x->ndim == 4 && axes.size() == 2;
                for (int64_t a : axes) {
                    const int64_t p = a < 0 ? a + x->ndim : a;
                    if (p != 2 && p != 3) spatial = false;
                }
                if (!spatial) return mfail(ctx, RTEN_ERR_UNSUPPORTED_VALUE, "ReduceMean: only the spatial axes of an NCHW tensor are supported");
            }
            st = rten_b200_global_average_pool(ctx, x, &y);
            if (st == RTEN_OK && !keepdims) {
                y.ndim = 2;
                set_contiguous(&y);
            }
        } else if (op == "Gemm") {
            st = rten_b200_gemm(ctx, T(0), T(1), T(2), o.n.attr_f("alpha", 1.0f), o.n.attr_f("beta", 1.0f), (int)o.n.attr_i("transA", 0),
                                (int)o.n.attr_i("transB", 0), &y);
        } else if (op == "MatMul") {
            const rten_tensor* bias = o.bias_value >= 0 ? &V(o.bias_value).t : nullptr;
            st = rten_b200_matmul(ctx, T(0), T(1), o.packed, bias, 1.0f, &y);
        } else if (op == "MatMulInteger") {
            st = rten_b200_matmul_integer(ctx, T(0), T(1), o.packed, T(2), T(3), nullptr, &y);
        } else if (op == "Add") {
            if (!T(1)) return mfail(ctx, RTEN_ERR_MISSING_INPUTS, "missing inputs");
            st = rten_b200_add(ctx, T(0), T(1), &y);
        } else if (op == "Mul") {
            if (!T(1)) return mfail(ctx, RTEN_ERR_MISSING_INPUTS, "missing inputs");
            st = rten_b200_mul(ctx, T(0), T(1), &y);
        } else if (op == "LayerNormalization") {
            st = rten_b200_layer_norm(ctx, T(0), T(1), T(2), (int)o.n.attr_i("axis", -1), o.n.attr_f("epsilon", 1e-5f), &y);
        } else if (op == "Gather") {
            if (o.n.attr_i("axis", 0) != 0 || T(0)->ndim != 2)
                return mfail(ctx, RTEN_ERR_UNSUPPORTED_VALUE, "Gather: only axis 0 of a 2-D table is supported");
            st = rten_b200_gather_rows(ctx, T(0), T(1), &y);
        } else if (op == "DynamicQuantizeLinear") {
            rten_tensor s, z;
            memset(&s, 0, sizeof(s));
            memset(&z, 0, sizeof(z));
            st = rten_b200_dynamic_quantize_linear(ctx, T(0), &y, &s, &z, nullptr);
            if (st == RTEN_OK) {
                if (o.out.size() > 1 && o.out[1] >= 0) set_owned(o.out[1], s); else pool_free(ctx, s.data);
                if (o.out.size() > 2 && o.out[2] >= 0) set_owned(o.out[2], z); else pool_free(ctx, z.data);
            }
        } else if (op == "Cast") {
            const int64_t to = o.n.attr_i("to", 0);
            const rten_tensor* x = T(0);
            if (to == onnx::DT_FLOAT && x->dtype == RTEN_I32) {
                rten_tensor c;
                bool alloc = false;
                RTB_TRY(make_contiguous(*x, &c, &alloc));
                y = c;
                y.dtype = RTEN_F32;
                void* d = nullptr;
                st = pool_alloc(ctx, (size_t)std::max<int64_t>(numel(&c), 1) * 4, &d);
                if (st == RTEN_OK) {
                    y.data = d;
                    const long long n = numel(&c);
                    st = launch_cast_scale(ctx, (const int*)c.data, (float*)d, n, 1, m->one, 1);  // f32(x) * 1.0f: exact
                }
                if (alloc) pool_free(ctx, c.data);
            } else if ((to == onnx::DT_FLOAT && x->dtype == RTEN_F32) || ((to == onnx::DT_INT32 || to == onnx::DT_INT64) && x->dtype == RTEN_I32)) {
                set_view(o.out[0], *x, o.in[0]);
                return RTEN_OK;
            } else {
                return mfail(ctx, RTEN_ERR_UNSUPPORTED_VALUE, "Cast: only int32 -> float is supported");
            }
        } else if (op == "Attention") {
            rten_attention_params p;
            memset(&p, 0, sizeof(p));
            p.is_causal = (int32_t)o.n.attr_i("is_causal", 0);
            p.q_num_heads = (int32_t)o.n.attr_i("q_num_heads", 0);
            p.kv_num_heads = (int32_t)o.n.attr_i("kv_num_heads", 0);
            p.scale = o.n.attr_f("scale", 0.0f);
            p.softcap = o.n.attr_f("softcap", 0.0f);
            if (T(4) || T(5)) return mfail(ctx, RTEN_ERR_UNSUPPORTED_VALUE, "Attention: past_key / past_value inputs are not supported by the executor");
            st = rten_b200_attention(ctx, T(0), T(1), T(2), T(3), T(6), &p, nullptr, nullptr, &y);
        } else {
            return mfail(ctx, RTEN_ERR_UNSUPPORTED_VALUE, "unsupported operator " + op);
        }
        RTB_TRY(st);
        if (in_place) {
            // the input's buffer now belongs to the output value
            ValueSlot& x = V(o.in[0]);
            x.owned = false;
            x.live = false;
        }
        set_owned(o.out[0], y);
        return RTEN_OK;
    }
};

}  // namespace

extern "C" rten_status rten_b200_model_run(rten_model* m, int32_t n_inputs, const char* const* input_names, const rten_tensor* inputs,
                                           int32_t n_outputs, const char* const* output_names, rten_tensor* outputs) {
    if (!m || (n_inputs && (!input_names || !inputs)) || n_outputs < 1 || !output_names || !outputs) return RTEN_ERR_INVALID_VALUE;
    rten_ctx* ctx = m->ctx;
    cudaSetDevice(ctx->device);
    Runner r{m, ctx, {}};
    // reset run state
    for (ValueSlot& v : m->values) {
        if (v.kind == V_TEMP || v.kind == V_INPUT) {
            v.live = false;
            v.owned = false;
            v.root = -1;
            v.views = 0;
            v.pending = 0;
            if (v.kind == V_TEMP) v.t.data = nullptr;
        }
    }
    std::vector<void*> staged;  // device copies of host inputs
    auto cleanup = [&](rten_status st) {
        for (ValueSlot& v : m->values)
            if (v.kind == V_TEMP && v.owned && v.live && (st != RTEN_OK || !r.keep.count((int)(&v - m->values.data())))) {
                pool_free(ctx, v.t.data);
                v.live = false;
                v.owned = false;
            }
        for (void* p : staged) pool_free(ctx, p);
        return st;
    };
    for (int32_t i = 0; i < n_inputs; i++) {
        auto it = m->by_name.find(input_names[i] ? input_names[i] : "");
        if (it == m->by_name.end() || m->values[(size_t)it->second].kind != V_INPUT)
            return mfail(ctx, RTEN_ERR_INVALID_VALUE, std::string("unknown model input '") + (input_names[i] ? input_names[i] : "") + "'");
        ValueSlot& v = m->values[(size_t)it->second];
        v.t = inputs[i];
        if (inputs[i].device < 0) {  // host tensor: staged through HBM for the duration of the run
            rten_tensor d = inputs[i];
            set_contiguous(&d);
            void* p = nullptr;
            rten_status st = pool_alloc(ctx, (size_t)std::max<int64_t>(numel(&d), 1) * dtype_size(d.dtype), &p);
            if (st != RTEN_OK) return cleanup(st);
            staged.push_back(p);
            d.data = p;
            d.device = ctx->device;
            st = rten_b200_copy(ctx, &inputs[i], &d);
            if (st != RTEN_OK) return cleanup(st);
            v.t = d;
        }
        v.live = true;
    }
    for (int id : m->inputs)
        if (!m->values[(size_t)id].live) return cleanup(mfail(ctx, RTEN_ERR_MISSING_INPUTS, "model input '" + m->values[(size_t)id].name + "' was not provided"));
    std::vector<int> want;
    for (int32_t i = 0; i < n_outputs; i++) {
        auto it = m->by_name.find(output_names[i] ? output_names[i] : "");
        if (it == m->by_name.end()) return cleanup(mfail(ctx, RTEN_ERR_INVALID_VALUE, std::string("unknown model output '") + (output_names[i] ? output_names[i] : "") + "'"));
        want.push_back(it->second);
        r.keep.insert(it->second);
    }
    // consumer counts (the plan is the whole node list: pruning to the requested outputs is not needed for these models)
    for (OpNode& o : m->nodes) {
        for (int i : o.in)
            if (i >= 0) m->values[(size_t)i].pending++;
        if (o.bias_value >= 0) m->values[(size_t)o.bias_value].pending++;
    }
    for (OpNode& o : m->nodes) {
        rten_status st = r.run_node(o);
        if (st != RTEN_OK) return cleanup(st);
        std::set<int> seen;
        for (int i : o.in) r.consumed(i);
        (void)seen;
    }
    // hand the requested outputs over: owned buffers move to the caller; views / constants / inputs are copied
    for (int32_t i = 0; i < n_outputs; i++) {
        ValueSlot& v = m->values[(size_t)want[(size_t)i]];
        if (!v.live && v.kind != V_CONST) return cleanup(mfail(ctx, RTEN_ERR_INVALID_VALUE, "requested output '" + v.name + "' was not computed"));
        const bool movable = v.kind == V_TEMP && v.owned && v.root < 0 && v.views == 0 && is_contiguous(&v.t);
        bool dup = false;
        for (int32_t k = 0; k < i; k++) dup = dup || want[(size_t)k] == want[(size_t)i];
        if (movable && !dup) {
            outputs[i] = v.t;
            v.owned = false;
            v.live = false;
        } else {
            rten_tensor c = v.t;
            set_contiguous(&c);
            void* p = nullptr;
            rten_status st = pool_alloc(ctx, (size_t)std::max<int64_t>(numel(&c), 1) * dtype_size(c.dtype), &p);
            if (st != RTEN_OK) return cleanup(st);
            c.data = p;
            st = rten_b200_copy(ctx, &v.t, &c);
            if (st != RTEN_OK) {
                pool_free(ctx, p);
                return cleanup(st);
            }
            outputs[i] = c;
        }
    }
    r.keep.clear();
    return cleanup(RTEN_OK);
}
