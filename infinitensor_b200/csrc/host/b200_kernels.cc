// b200_kernels.cc -- the plugin layer: one Kernel subclass per hot operator, registered through
// REGISTER_KERNEL(Device::CUDA, OpType::X, ...) exactly like the reference's src/kernels/cuda/*.cc,
// each bottoming out in one extern "C" it_b200_* launcher (include/it_b200.h).  Because the registry
// rejects duplicate keys (reference include/core/kernel.h:150-156) this set REPLACES the reference's
// src/kernels/cuda directory in a build; there is no second backend and no CPU fallback.
//
// SEAM-A BUILD (-DITB_SEAM_A, oracle/Makefile target `seam_a`): this very file is compiled against the REFERENCE's own headers
// (/root/reference/include: core/kernel.h:32-195, cuda/cuda_kernel_wihtout_config.h, cuda/cuda_runtime.h, operators/*.h) and
// linked, together with libit_b200.so, in place of the reference's src/kernels/cuda directory; the reference's gtests then
// run against these kernels (oracle/_ref/seam_a/seam_a_tests).  Only what does not exist in the reference is compiled out there:
// the fused executors of this repo's schedule, the per-row-position extension and the dlopen'ed NCCL collectives.
#ifdef ITB_SEAM_A
#include "core/kernel.h"
#include "cuda/cuda_kernel_wihtout_config.h"
#include "cuda/cuda_runtime.h"
#include "operators/attention_kvcache.h"
#include "operators/batch_norm.h"
#include "operators/concat.h"
#include "operators/conv.h"
#include "operators/element_wise.h"
#include "operators/expand.h"
#include "operators/gather.h"
#include "operators/layer_norm.h"
#include "operators/matmul.h"
#include "operators/pad.h"
#include "operators/pooling.h"
#include "operators/reduce.h"
#include "operators/reshape.h"
#include "operators/rms_norm.h"
#include "operators/rope.h"
#include "operators/slice.h"
#include "operators/softmax.h"
#include "operators/split.h"
#include "operators/transpose.h"
#include "operators/unary.h"
#include "operators/where.h"
#include "it_b200.h"
#else
#include "b200_runtime.h"
#include "nccl_dl.h"
#include "it_b200.h"
#include "operators.h"
#endif

namespace infini {

static inline void CK(int ret, const Operator &op) {
    if (ret != 0) throw Exception(string(it_b200_last_error()) + " in " + op->toString());
}
static inline void *S() { return (void *)CUDAStream::getCurrentStream(); }
static inline const CudaRuntimeObj *RT(const RuntimeObj *ctx) {
    auto rt = dynamic_cast<const CudaRuntimeObj *>(ctx);
    IT_ASSERT(rt != nullptr, "kernel invoked on a non-CUDA runtime");
    return rt;
}
static inline int DTI(const Tensor &t) { return t->getDTypeIndex(); }  // ONNX dtype code (reference data_type.h:6-23)
static inline void *P(const Tensor &t) { return t->getRawDataPtr<void *>(); }

// numpy-broadcast strides of `shape` against `out` (elements; 0 on broadcast dims)
static vector<int64_t> bstrides(const Shape &shape, const Shape &out) {
    size_t r = out.size(), off = r - shape.size();
    vector<int64_t> st(r, 0);
    int64_t acc = 1;
    for (int i = (int)shape.size() - 1; i >= 0; --i) {
        st[off + i] = (shape[i] == 1 && out[off + i] != 1) ? 0 : acc;
        acc *= shape[i];
    }
    return st;
}
static vector<int64_t> to64(const Shape &s) { return vector<int64_t>(s.begin(), s.end()); }

// ---------------------------------------------------------------- unary family
static int unaryCode(OpType t) {
    switch (t.underlying()) {
    case OpType::Relu: return ITB_RELU;
    case OpType::Sigmoid: return ITB_SIGMOID;
    case OpType::Tanh: return ITB_TANH;
    case OpType::Gelu: return ITB_GELU;
    case OpType::Silu: return ITB_SILU;
    case OpType::Erf: return ITB_ERF;
    case OpType::Neg: return ITB_NEG;
    case OpType::Abs: return ITB_ABS;
    case OpType::Sqrt: return ITB_SQRT;
    case OpType::HardSigmoid: return ITB_HARDSIGMOID;
    case OpType::HardSwish: return ITB_HARDSWISH;
    case OpType::Exp: return ITB_EXP;
    }
    return -1;
}
class UnaryB200 : public CudaKernelWithoutConfig {
    void compute(const Operator &op, const RuntimeObj *) const override {
        auto x = op->getInputs(0), y = op->getOutput();
        CK(it_b200_unary(unaryCode(op->getOpType()), DTI(x), P(x), P(y), (int64_t)x->size(), S()), op);
    }
};

class UnaryAlphaB200 : public CudaKernelWithoutConfig {
    void compute(const Operator &op, const RuntimeObj *) const override {
        auto x = op->getInputs(0), y = op->getOutput();
        const bool leaky = op->getOpType() == OpType::LeakyRelu;
        const float alpha = leaky ? as<LeakyReluObj>(op)->getAlpha() : as<EluObj>(op)->getAlpha();
        CK(it_b200_unary_alpha(leaky ? ITB_LEAKYRELU : ITB_ELU, DTI(x), P(x), P(y), (int64_t)x->size(), alpha, S()), op);
    }
};

static int binaryCode(OpType t) {
    switch (t.underlying()) {
    case OpType::Add: return ITB_ADD;
    case OpType::Sub: return ITB_SUB;
    case OpType::Mul: return ITB_MUL;
    case OpType::Div: return ITB_DIV;
    case OpType::Pow: return ITB_POW;
    case OpType::Min: return ITB_MIN;
    case OpType::Max: return ITB_MAX;
    case OpType::Less: return ITB_LESS;
    case OpType::Equal: return ITB_EQUAL;
    case OpType::Greater: return ITB_GREATER;
    }
    return -1;
}
class ElementWiseB200 : public CudaKernelWithoutConfig {
    void compute(const Operator &op, const RuntimeObj *) const override {
        auto a = op->getInputs(0), b = op->getInputs(1), c = op->getOutput();
        IT_ASSERT(a->getDType() == b->getDType(), "elementwise operands must share a dtype");
        auto dims = to64(c->getDims());
        auto sa = bstrides(a->getDims(), c->getDims()), sb = bstrides(b->getDims(), c->getDims());
        CK(it_b200_binary(binaryCode(op->getOpType()), DTI(a), P(a), P(b), P(c), (int)dims.size(), dims.data(),
                          sa.data(), sb.data(), S()), op);
    }
};

class CastB200 : public CudaKernelWithoutConfig {
    void compute(const Operator &op, const RuntimeObj *) const override {
        auto x = op->getInputs(0), y = op->getOutput();
        CK(it_b200_cast(DTI(x), DTI(y), P(x), P(y), (int64_t)x->size(), S()), op);
    }
};

class WhereB200 : public CudaKernelWithoutConfig {
    void compute(const Operator &op, const RuntimeObj *) const override {
        auto x = op->getInputs(0), y = op->getInputs(1), c = op->getInputs(2), o = op->getOutput();
        IT_ASSERT(c->getDType().getSize() == 1, "Where: condition must be bool/uint8");
        auto dims = to64(o->getDims());
        auto sc = bstrides(c->getDims(), o->getDims()), sx = bstrides(x->getDims(), o->getDims()),
             sy = bstrides(y->getDims(), o->getDims());
        CK(it_b200_where((int)x->getDType().getSize(), P(c), P(x), P(y), P(o), (int)dims.size(), dims.data(),
                         sc.data(), sx.data(), sy.data(), S()), op);
    }
};

class ExpandB200 : public CudaKernelWithoutConfig {
    void compute(const Operator &op, const RuntimeObj *) const override {
        auto x = op->getInputs(0), o = op->getOutput();
        auto dims = to64(o->getDims());
        auto sx = bstrides(x->getDims(), o->getDims());
        CK(it_b200_expand((int)x->getDType().getSize(), P(x), P(o), (int)dims.size(), dims.data(), sx.data(), S()),
           op);
    }
};

// ---------------------------------------------------------------- norms / softmax / rope
static void axisView(const Shape &d, int axis, int64_t &outer, int &dim, int64_t &inner) {
    outer = inner = 1;
    for (int i = 0; i < axis; ++i) outer *= d[i];
    dim = d[axis];
    for (int i = axis + 1; i < (int)d.size(); ++i) inner *= d[i];
}
class SoftmaxB200 : public CudaKernelWithoutConfig {
    void compute(const Operator &_op, const RuntimeObj *) const override {
        auto op = as<SoftmaxObj>(_op);
        auto x = op->getInputs(0);
        int64_t outer, inner;
        int dim;
        axisView(x->getDims(), op->getAxis(), outer, dim, inner);
        CK(it_b200_softmax(DTI(x), P(x), P(op->getOutput()), outer, dim, inner, S()), _op);
    }
};
class LayerNormB200 : public CudaKernelWithoutConfig {
    void compute(const Operator &_op, const RuntimeObj *) const override {
        auto op = as<LayerNormObj>(_op);
        auto x = op->getInputs(0), sc = op->getInputs(1);
        auto bias = op->getBias();
        int64_t outer, inner;
        int dim;
        axisView(x->getDims(), op->getAxis(), outer, dim, inner);
        CK(it_b200_layernorm(DTI(x), P(x), P(sc), bias ? P(bias) : nullptr, P(op->getOutput()), outer, dim, inner,
                             (int)sc->size(), bias ? (int)bias->size() : 0, op->getEps(), S()), _op);
    }
};
class RMSNormB200 : public CudaKernelWithoutConfig {
    void compute(const Operator &op, const RuntimeObj *) const override {
        auto x = op->getInputs(0), w = op->getInputs(1);
        int hidden = x->getDims().back();
        IT_ASSERT((int)w->size() == hidden, "RMSNorm: weight length must equal the hidden size");
        auto fn = w->isWeight() ? it_b200_rmsnorm_constw : it_b200_rmsnorm;
        CK(fn(DTI(x), P(x), P(w), P(op->getOutput()), (int64_t)(x->size() / hidden), hidden, S()), op);
    }
};
class RoPEB200 : public CudaKernelWithoutConfig {
    void compute(const Operator &op, const RuntimeObj *) const override {
        auto pos = op->getInputs(0), x = op->getInputs(1);
        const auto &d = x->getDims();
        IT_ASSERT(d.size() == 3 && pos->getRank() == 2, "RoPE: input [B,S,dim_model], pos [B,S]");
        IT_ASSERT(d[0] == pos->getDims()[0] && d[1] == pos->getDims()[1], "RoPE: pos / input mismatch");
        const int dim_head = 128;  // hard-coded in the reference (rope.cc:25)
        CK(it_b200_rope(DTI(x), P(pos), DTI(pos), P(x), P(op->getOutput()), d[0], d[1], d[2], dim_head, S()), op);
    }
};

// ---------------------------------------------------------------- data movement
class TransposeB200 : public CudaKernelWithoutConfig {
    void compute(const Operator &_op, const RuntimeObj *) const override {
        auto op = as<TransposeObj>(_op);
        auto x = op->getInputs(0);
        auto dims = to64(x->getDims());
        CK(it_b200_transpose((int)x->getDType().getSize(), P(x), P(op->getOutput()), (int)dims.size(), dims.data(),
                             op->getPermute().data(), S()), _op);
    }
};
// DepthToSpace = the rank-6 permutation of the operator's reshaped view (reference transpose.cc:48-90)
class DepthToSpaceB200 : public CudaKernelWithoutConfig {
    void compute(const Operator &_op, const RuntimeObj *) const override {
        auto op = as<DepthToSpaceObj>(_op);
        auto x = op->getInputs(0);
        auto rd = op->getReshapeDim();
        vector<int64_t> dims(rd.begin(), rd.end());
        vector<int> perm = op->getMode() == 0 ? vector<int>{0, 3, 4, 1, 5, 2} : vector<int>{0, 1, 4, 2, 5, 3};
        CK(it_b200_transpose((int)x->getDType().getSize(), P(x), P(op->getOutput()), (int)dims.size(), dims.data(), perm.data(),
                             S()), _op);
    }
};
class ConcatB200 : public CudaKernelWithoutConfig {
    void compute(const Operator &_op, const RuntimeObj *) const override {
        auto op = as<ConcatObj>(_op);
        auto out = op->getOutput();
        int dim = op->getDim();
        int64_t outer = 1, inner = 1;
        for (int i = 0; i < dim; ++i) outer *= out->getDims()[i];
        for (int i = dim + 1; i < (int)out->getRank(); ++i) inner *= out->getDims()[i];
        vector<const void *> parts;
        vector<int64_t> lens;
        for (auto &t : op->getInputs()) {
            if (t->size() == 0) continue;  // empty operands contribute nothing (reference split_concat.cc:64-78)
            parts.push_back(P(t));
            lens.push_back(t->getDims()[dim]);
        }
        if (parts.empty()) return;
        CK(it_b200_concat((int)out->getDType().getSize(), (int)parts.size(), parts.data(), lens.data(), P(out), outer,
                          inner, S()), _op);
    }
};
class SplitB200 : public CudaKernelWithoutConfig {
    void compute(const Operator &_op, const RuntimeObj *) const override {
        auto op = as<SplitObj>(_op);
        auto in = op->getInputs(0);
        int dim = op->getDim();
        int64_t outer = 1, inner = 1;
        for (int i = 0; i < dim; ++i) outer *= in->getDims()[i];
        for (int i = dim + 1; i < (int)in->getRank(); ++i) inner *= in->getDims()[i];
        vector<void *> parts;
        vector<int64_t> lens;
        for (auto &t : op->getOutputs()) {
            parts.push_back(t->size() ? P(t) : nullptr);
            lens.push_back(t->getDims()[dim]);
        }
        CK(it_b200_split((int)in->getDType().getSize(), (int)parts.size(), parts.data(), lens.data(), P(in), outer,
                         inner, S()), _op);
    }
};
class GatherB200 : public CudaKernelWithoutConfig {
    void compute(const Operator &_op, const RuntimeObj *) const override {
        auto op = as<GatherObj>(_op);
        auto x = op->getInputs(0), idx = op->getInputs(1);
        int axis = op->getAxis();
        int64_t outer = 1, inner = 1;
        for (int i = 0; i < axis; ++i) outer *= x->getDims()[i];
        for (int i = axis + 1; i < (int)x->getRank(); ++i) inner *= x->getDims()[i];
        CK(it_b200_gather((int)x->getDType().getSize(), DTI(idx), P(x), P(idx), P(op->getOutput()), outer,
                          x->getDims()[axis], inner, (int64_t)idx->size(), S()), _op);
    }
};
// Reshape / Flatten / Identity / Squeeze / Unsqueeze: a copy into the planner-assigned output
class CopyB200 : public CudaKernelWithoutConfig {
    void compute(const Operator &op, const RuntimeObj *) const override {
        auto x = op->getInputs(0), y = op->getOutput();
        IT_ASSERT(x->getBytes() == y->getBytes(), "reshape-like op changes the byte count");
        CK(it_b200_copy(P(x), P(y), (int64_t)x->getBytes(), S()), op);
    }
};
class SliceB200 : public CudaKernelWithoutConfig {
    void compute(const Operator &_op, const RuntimeObj *) const override {
        auto op = as<SliceObj>(_op);
        auto x = op->getInputs(0), y = op->getOutput();
        auto din = to64(x->getDims()), dout = to64(y->getDims());
        auto st = op->getStarts(), sp = op->getSteps();
        vector<int64_t> start(st.begin(), st.end()), step(sp.begin(), sp.end());
        CK(it_b200_pad_slice((int)x->getDType().getSize(), P(x), P(y), (int)din.size(), din.data(), dout.data(),
                             start.data(), step.data(), S()), _op);
    }
};
class PadB200 : public CudaKernelWithoutConfig {
    void compute(const Operator &_op, const RuntimeObj *) const override {
        auto op = as<PadObj>(_op);
        auto x = op->getInputs(0), y = op->getOutput();
        auto din = to64(x->getDims()), dout = to64(y->getDims());
        int rank = (int)din.size();
        vector<int64_t> start(rank), step(rank, 1);
        for (int i = 0; i < rank; ++i) start[i] = -op->getPads()[i];
        CK(it_b200_pad_slice((int)x->getDType().getSize(), P(x), P(y), rank, din.data(), dout.data(), start.data(),
                             step.data(), S()), _op);
    }
};
class ReduceB200 : public CudaKernelWithoutConfig {
    void compute(const Operator &_op, const RuntimeObj *) const override {
        auto op = as<ReduceBaseObj>(_op);
        auto x = op->getInputs(0);
        auto dims = to64(x->getDims());
        vector<int> mask(dims.size());
        for (int i = 0; i < (int)dims.size(); ++i) mask[i] = op->isReduced(i);
        CK(it_b200_reduce(DTI(x), _op->getOpType() == OpType::ReduceMean, P(x), P(op->getOutput()), (int)dims.size(),
                          dims.data(), mask.data(), S()), _op);
    }
};
class PoolingB200 : public CudaKernelWithoutConfig {
    void compute(const Operator &_op, const RuntimeObj *) const override {
        auto op = as<PoolingObj>(_op);
        auto x = op->getInputs(0), y = op->getOutput();
        const int kh = op->getKh(), kw = op->getKw(), dh = op->getDh(), dw = op->getDw(), ph = op->getPh(), pw = op->getPw(),
                  sh = op->getSh(), sw = op->getSw();
        const auto &d = x->getDims();
        const auto &o = y->getDims();
        CK(it_b200_pool2d(DTI(x), _op->getOpType() == OpType::MaxPool, P(x), P(y), d[0], d[1], d[2], d[3], kh, kw, dh,
                          dw, ph, pw, sh, sw, o[2], o[3], S()), _op);
    }
};
class BatchNormB200 : public CudaKernelWithoutConfig {
    void compute(const Operator &_op, const RuntimeObj *) const override {
        auto op = as<BatchNormObj>(_op);
        auto x = op->getInputs(0);
        for (int i = 1; i <= 4; ++i)
            IT_ASSERT(op->getInputs(i)->getDType() == DataType::Float32, "BatchNorm statistics must be fp32");
        const auto &d = x->getDims();
        int64_t hw = 1;
        for (size_t i = 2; i < d.size(); ++i) hw *= d[i];
        CK(it_b200_batchnorm(DTI(x), P(x), op->getInputs(1)->getRawDataPtr<float *>(),
                             op->getInputs(2)->getRawDataPtr<float *>(), op->getInputs(3)->getRawDataPtr<float *>(),
                             op->getInputs(4)->getRawDataPtr<float *>(), P(op->getOutput()), d[0], d[1], hw,
                             op->getEps(), S()), _op);
    }
};

// ---------------------------------------------------------------- MatMul / Conv / Attention
namespace b200 {
// MatMul with optional fused residual: C = A.B (+ bias) ; when `residual` is given (MatMul -> Add fusion) the
// product is rounded to the storage dtype first, the residual added in the epilogue and the result written to
// `outOverride` (the Add's output) -- bit-identical to the two separate kernels.
void runMatmul(const Operator &_op, const RuntimeObj *ctx, const Tensor &residual, const Tensor &outOverride) {
    auto op = as<MatmulObj>(_op);
    auto A = op->getInputs(0), B = op->getInputs(1);
    auto C = outOverride ? outOverride : op->getOutput();
#ifdef ITB_SEAM_A
    IT_ASSERT(A->getDType() == B->getDType(), "MatMul operands must share a dtype");
#else
    IT_ASSERT(A->getDType() == B->getDType() || op->getWScale(), "MatMul operands must share a dtype (or B = FP8 codes + scale)");
#endif
    auto [b_, m_, n, k] = op->getBMNK();
    int b = b_, m = m_;
    // batch rule of the reference (matmul.cc:124-137): full batch or stride-0 broadcast
    auto batchOf = [](const Tensor &t) {
        int64_t v = 1;
        for (int i = 0; i + 2 < (int)t->getRank(); ++i) v *= t->getDims()[i];
        return v;
    };
    int64_t ba = batchOf(A), bb = batchOf(B);
    IT_ASSERT((ba == b || ba == 1) && (bb == b || bb == 1), "MatMul: unsupported partial batch broadcast");
    int64_t sa = (ba == 1 && b > 1) ? 0 : (int64_t)m * k, sb = (bb == 1 && b > 1) ? 0 : (int64_t)n * k;
    const void *bias = nullptr;
    int64_t bsb = 0, bsm = 0, bsn = 0;
    int act = 0;  // MatmulObj::act is ignored like the reference does (quirk q5)
    auto bt = residual ? residual : op->getBias();
    if (bt) {
        IT_ASSERT(!(residual && op->getBias()), "MatMul: residual fusion needs a bias-free MatMul");
        bias = P(bt);
        Shape bd = bt->getDims();
        Shape cd = op->getOutput()->getDims();
        auto st = bstrides(bd, cd);
        bsn = st[cd.size() - 1];
        bsm = st[cd.size() - 2];
        bool anyBatch = false;
        for (size_t i = 0; i + 2 < cd.size(); ++i) anyBatch = anyBatch || st[i] != 0;
        if (anyBatch) {
            int64_t bbias = 1;
            for (int i = 0; i + 2 < (int)bd.size(); ++i) bbias *= bd[i];
            IT_ASSERT(bbias == b, "MatMul: bias batch dims must be full or broadcast");
            bsb = (int64_t)(bd[bd.size() - 2]) * bd[bd.size() - 1];
        }
        if (residual) act |= ITB_ACT_ROUND_BEFORE_BIAS;
    }
    if (B->isWeight()) act |= ITB_MATMUL_B_CONST;
#ifndef ITB_SEAM_A
    if (auto ws = op->getWScale()) {
        // FP8 E4M3 weight, dequantised inside the GEMM (decode shapes: the skinny kernel); bias only as the fused residual
        IT_ASSERT(!op->getBias() && !op->getTransA() && !op->getTransB() && bb == 1, "MatMul(fp8 weight): plain [.., K] x [K, N] only");
        const int rows = (int)((int64_t)b * m);
        const void *W[1] = {P(B)};
        const float *Sc[1] = {ws->getRawDataPtr<float *>()};
        void *Cp[1] = {P(C)};
        int N[1] = {n};
        CK(it_b200_matmul_fp8w(DTI(A), P(A), 1, W, Sc, Cp, N, rows, k, residual ? P(residual) : nullptr, S()), _op);
        return;
    }
#endif
    // [b, m, k] x [k, n] with the weight broadcast over the batch (how the frontend emits every Linear layer of a
    // decode step: b = batch, m = 1) is ONE GEMM with M = b*m -- the reference instead runs b strided-batched GEMMs
    // with stride 0 (matmul.cc:124-168)
    if (b > 1 && sb == 0 && !op->getTransA() && sa == (int64_t)m * k && (m == 1 || bsb == bsm * m)) {
        if (m == 1) bsm = bsb;
        bsb = 0;
        m = b * m;
        b = 1;
        sa = (int64_t)m * k;
    }
    int64_t wsb = it_b200_matmul_workspace(DTI(A), b, m, n, k);
    void *ws = wsb ? RT(ctx)->getWorkspace((size_t)wsb) : nullptr;
    CK(it_b200_matmul(DTI(A), P(A), P(B), bias, P(C), b, m, n, k, sa, sb, op->getTransA(), op->getTransB(), bsb, bsm, bsn,
                      act, ws, wsb, S()), _op);
}

#ifndef ITB_SEAM_A  // ---- this repo's schedule-level executors (no counterpart in the reference)
// MatMul (+ bias) -> [Gelu] -> [Add(residual)]: ops = {MatMul, [Gelu], [Add]} in one tcgen05 epilogue.  false = the shape is not
// taken (nothing launched): the caller runs the operators one by one.
bool matmulAddIsPlain(const OpVec &ops) {
    return ops.size() == 2 && ops[1]->getOpType() == OpType::Add && !as<MatmulObj>(ops[0])->getBias();
}
bool runMatmulFused(const OpVec &ops, const RuntimeObj *) {
    auto mm = as<MatmulObj>(ops[0]);
    Operator actOp, add;
    for (size_t i = 1; i < ops.size(); ++i) {
        if (ops[i]->getOpType() == OpType::Add) add = ops[i];
        else actOp = ops[i];
    }
    auto A = mm->getInputs(0), B = mm->getInputs(1), bias = mm->getBias();
    if (B->getRank() != 2 || mm->getTransA() || mm->getWScale()) return false;
    if (bias && !(bias->getRank() == 1 && bias->getDims()[0] == mm->getN())) return false;
    int act = 0;
    if (actOp) {
        if (actOp->getOpType() != OpType::Gelu) return false;
        act = 4;
    }
    int64_t rows = 1;
    for (size_t i = 0; i + 1 < A->getRank(); ++i) rows *= A->getDims()[i];
    if (rows > (1ll << 30)) return false;
    Tensor res;
    if (add) {
        Tensor prev = ops[ops.size() - 2]->getOutput();
        res = add->getInputs(0) == prev ? add->getInputs(1) : add->getInputs(0);
    }
    if (B->isWeight()) act |= ITB_MATMUL_B_CONST;
    const int n = mm->getN(), k = mm->getK();
    int rc = it_b200_matmul_fused(DTI(A), P(A), P(B), bias ? P(bias) : nullptr, res ? P(res) : nullptr, P(ops.back()->getOutput()), 1,
                                  (int)rows, n, k, rows * k, 0, 0, mm->getTransB() ? 1 : 0, 0, 0, 1, act, S());
    if (rc == 2) return false;
    CK(rc, ops.back());
    return true;
}

// q/k/v or gate/up: MatMuls sharing the activation operand, weights [K, N_i]: one grouped launch
void runMatmulGroup(const OpVec &ops, const RuntimeObj *) {
    auto A = ops[0]->getInputs(0);
    int k = as<MatmulObj>(ops[0])->getK();
    int64_t rows = 1;
    for (size_t i = 0; i + 1 < A->getRank(); ++i) rows *= A->getDims()[i];
    const void *W[4];
    void *C[4];
    int N[4];
    IT_ASSERT(ops.size() <= 4);
    const float *Sc[4] = {nullptr, nullptr, nullptr, nullptr};
    for (size_t i = 0; i < ops.size(); ++i) {
        W[i] = P(ops[i]->getInputs(1));
        C[i] = P(ops[i]->getOutput());
        N[i] = as<MatmulObj>(ops[i])->getN();
        if (auto ws = as<MatmulObj>(ops[i])->getWScale()) Sc[i] = ws->getRawDataPtr<float *>();
    }
    if (Sc[0]) {  // FP8 weights (the schedule groups like with like)
        CK(it_b200_matmul_fp8w(DTI(A), P(A), (int)ops.size(), W, Sc, C, N, (int)rows, k, nullptr, S()), ops[0]);
        return;
    }
    CK(it_b200_matmul_grouped(DTI(A), P(A), (int)ops.size(), W, C, N, (int)rows, k, S()), ops[0]);
}

void runSiluMul(const Operator &silu, const Operator &mul, const RuntimeObj *) {
    auto g = silu->getInputs(0);
    auto sout = silu->getOutput();
    auto u = mul->getInputs(0) == sout ? mul->getInputs(1) : mul->getInputs(0);
    CK(it_b200_silu_mul(DTI(g), P(g), P(u), P(mul->getOutput()), (int64_t)g->size(), S()), mul);
}
// position dtype + ITB_POS_* flags of an AttentionKVCache launch.  The kernel reads the position, the RoPE positions and the
// cache rows below the position AHEAD of griddepcontrol.wait, which is only sound when a whole step separates them from their
// writer: any of them produced by an operator of this graph (in-graph position arithmetic, Concat of the past) -> IN_STEP.
static int attnPosFlags(const Operator &att, const Tensor &ropePos) {
    auto pos = att->getInputs(5);
    int flags = DTI(pos);
    if (as<AttentionKVCacheObj>(att)->getPerRowPositions()) {
        IT_ASSERT((int64_t)pos->size() >= att->getInputs(0)->getDims()[0], "AttentionKVCache: per-row positions need one entry per batch row");
        flags |= ITB_POS_PER_ROW;
    }
    bool inStep = pos->getSource() != nullptr || att->getInputs(0)->getSource() != nullptr || att->getInputs(1)->getSource() != nullptr;
    if (ropePos && ropePos->getSource() != nullptr) inStep = true;
    if (inStep) flags |= ITB_POS_IN_STEP;
    return flags;
}
// RoPE(q), RoPE(k) folded into the decode attention kernel (the aliases between them are storage no-ops)
void runAttentionRope(const Operator &ropeQ, const Operator &ropeK, const Operator &att, const RuntimeObj *ctx) {
    auto kc = att->getInputs(0), vc = att->getInputs(1), v = att->getInputs(4), pos = att->getInputs(5);
    auto qpre = ropeQ->getInputs(1), kpre = ropeK->getInputs(1), rpos = ropeQ->getInputs(0);
    IT_ASSERT(ropeK->getInputs(0) == rpos, "RoPE(q) and RoPE(k) must share the position tensor");
    const auto &d = kc->getDims();
    int64_t wsb = it_b200_attention_kvcache_workspace(d[0], d[1], d[2], d[3]);
    void *ws = wsb ? RT(ctx)->getWorkspace((size_t)wsb) : nullptr;
    CK(it_b200_attention_kvcache_rope(DTI(qpre), P(kc), P(vc), P(qpre), P(kpre), P(v), P(pos), attnPosFlags(att, rpos), P(rpos), DTI(rpos),
                                      P(att->getOutput()), d[0], d[1], d[2], d[3], ws, wsb, S()), att);
}

bool runPrefillAttention(const OpVec &ops, const RuntimeObj *) {
    static const bool off = [] {
        const char *e = std::getenv("ITB_NO_PREFILL_ATTENTION");
        return e && e[0] == '1';
    }();
    if (off) return false;
    // extended form (schedule.cc extendPrefillChain): {Split, Rq, Tq, Rk, Tk, Rv, Tv, <chain>, mm2, Tout, Rout}
    const bool ext = ops[0]->getOpType() == OpType::Split;
    const size_t c0 = ext ? 7 : 0, cend = ext ? ops.size() - 2 : ops.size();  // [c0, cend) = Transpose(k), mm1, .., Softmax, mm2
    auto tr = ops[c0], mm1 = ops[c0 + 1], sm = ops[cend - 2], mm2 = ops[cend - 1];
    Tensor q = mm1->getInputs(0), k = tr->getInputs(0), v = mm2->getInputs(1), out = mm2->getOutput();
    const void *scale = nullptr, *maskp = nullptr;
    int isDiv = 0;
    int64_t ms[4] = {0, 0, 0, 0};
    Tensor cur = mm1->getOutput();
    const auto &qd = q->getDims();
    const Shape full = {qd[0], qd[1], qd[2], k->getDims()[2]};
    for (size_t i = c0 + 2; i + 2 < cend; ++i) {
        auto &o = ops[i];
        Tensor other = o->getInputs(0) == cur ? o->getInputs(1) : o->getInputs(0);
        if (o->getOpType() == OpType::Add) {
            auto st = bstrides(other->getDims(), full);
            for (int d = 0; d < 4; ++d) ms[d] = st[d];
            maskp = P(other);
        } else {
            scale = P(other);
            isDiv = o->getOpType() == OpType::Div;
        }
        cur = o->getOutput();
    }
    (void)sm;
    if (ext) {
        // q / k / v = thirds of every row of the projection output [B, S, 3 H D]; the result goes straight to [B, S, H D]
        Tensor qkv = ops[0]->getInputs(0), fin = ops.back()->getOutput();
        const int64_t B = qd[0], H = qd[1], Sq = qd[2], D = qd[3], d = H * D, row = qkv->getDims()[2];
        const int64_t view[3] = {Sq * row, D, row}, ost[3] = {Sq * d, D, d};
        const char *base = (const char *)P(qkv);
        const int64_t es = (int64_t)qkv->getDType().getSize();
        CK(it_b200_attention_prefill_strided(DTI(q), base, base + d * es, base + 2 * d * es, P(fin), (int)B, (int)H, (int)Sq, (int)k->getDims()[2],
                                             (int)D, view, view, view, ost, scale, isDiv, maskp, ms[0], ms[1], ms[2], ms[3], S()), mm2);
        return true;
    }
    CK(it_b200_attention_prefill(DTI(q), P(q), P(k), P(v), P(out), qd[0], qd[1], qd[2], k->getDims()[2], qd[3], scale, isDiv, maskp,
                                 ms[0], ms[1], ms[2], ms[3], S()), mm2);
    return true;
}

// DecoderStack: st.sub = per layer { RMSNorm | MatMulGroup{3} | AttentionRope | MatMulAdd | RMSNorm | MatMulGroup{2} | SiluMul |
// MatMulAdd } with Alias steps in between (schedule.cc: matchDecoderLayer)
bool runDecoderStack(const ExecStep &st, const RuntimeObj *ctx) {
    static const bool off = [] {
        const char *e = std::getenv("ITB_NO_DECODE_STACK");
        return e && e[0] == '1';
    }();
    if (off) return false;
    vector<const ExecStep *> cs;
    for (auto &sb : st.sub) {
        if (sb.kind == ExecStep::Alias) {
            // the kernel writes each tensor once: an alias must really share its input's storage (not the naive allocator)
            if (sb.ops[0]->getInputs(0)->rawPtrOrNull() != sb.ops[0]->getOutput()->rawPtrOrNull()) return false;
            continue;
        }
        cs.push_back(&sb);
    }
    if (cs.empty() || cs.size() % 8) return false;
    const int L = (int)cs.size() / 8;
    vector<itb_llama_layer> layers((size_t)L);
    Tensor x0, pos, rpos;
    Operator att0;
    int B = 0, d = 0, H = 0, Smax = 0, f = 0;
    for (int li = 0; li < L; ++li) {
        const ExecStep *const *c = &cs[(size_t)li * 8];
        auto n1 = c[0]->ops[0];
        auto ropeQ = c[2]->ops[0], ropeK = c[2]->ops[1], att = c[2]->ops[2];
        auto mo = c[3]->ops[0], add1 = c[3]->ops[1];
        auto n2 = c[4]->ops[0];
        auto silu = c[6]->ops[0], mul = c[6]->ops[1];
        auto md = c[7]->ops[0], add2 = c[7]->ops[1];
        Tensor qpre = ropeQ->getInputs(1), kpre = ropeK->getInputs(1);
        Tensor vin = att->getInputs(4);
        while (vin->getSource() && vin->getSource()->getOutput()->rawPtrOrNull() == vin->getSource()->getInputs(0)->rawPtrOrNull() &&
               vin->getSource()->getOpType() != OpType::MatMul)
            vin = vin->getSource()->getInputs(0);
        Operator mq, mk, mv;
        for (auto &mm : c[1]->ops) {
            if (mm->getOutput() == qpre) mq = mm;
            if (mm->getOutput() == kpre) mk = mm;
            if (mm->getOutput() == vin) mv = mm;
        }
        if (!mq || !mk || !mv) return false;
        Tensor gate = silu->getInputs(0);
        Operator mg, mu;
        for (auto &mm : c[5]->ops) (mm->getOutput() == gate ? mg : mu) = mm;
        if (!mg || !mu) return false;
        itb_llama_layer &Ly = layers[(size_t)li];
        Ly.ln1_w = P(n1->getInputs(1));
        Ly.wq = P(mq->getInputs(1));
        Ly.wk = P(mk->getInputs(1));
        Ly.wv = P(mv->getInputs(1));
        Ly.wo = P(mo->getInputs(1));
        Ly.ln2_w = P(n2->getInputs(1));
        Ly.wg = P(mg->getInputs(1));
        Ly.wu = P(mu->getInputs(1));
        Ly.wd = P(md->getInputs(1));
        Ly.k_cache = P(att->getInputs(0));
        Ly.v_cache = P(att->getInputs(1));
        Ly.q = P(qpre);
        Ly.k = P(kpre);
        Ly.v = P(vin);
        Ly.attn_out = P(att->getOutput());
        Ly.x_mid = P(add1->getOutput());
        Ly.gate = P(mg->getOutput());
        Ly.up = P(mu->getOutput());
        Ly.x_out = P(add2->getOutput());
        (void)mul;
        if (li == 0) {
            x0 = n1->getInputs(0);
            pos = att->getInputs(5);
            rpos = ropeQ->getInputs(0);
            att0 = att;
            const auto &cd = att->getInputs(0)->getDims();
            B = cd[0];
            H = cd[1];
            Smax = cd[2];
            d = x0->getDims().back();
            f = as<MatmulObj>(mg)->getN();
        }
    }
    auto rt = RT(ctx);
    int64_t wsb = it_b200_decode_stack_workspace(L, B, d, H, Smax, f);
    void *ws = rt->getWorkspace((size_t)wsb);
    int rc = it_b200_llama_decode_stack(DTI(x0), L, layers.data(), P(x0), P(pos), attnPosFlags(att0, rpos), P(rpos), DTI(rpos), B, d, H, Smax, f,
                                        ws, (int64_t)rt->getWorkspaceSize(), S());
    CK(rc, att0);
    return true;
}

// Conv -> BatchNorm -> [Add(residual)] -> [Relu]: ops = {conv, bn, [add], [relu]}; a lone Conv when ops.size() == 1.
// layout (ExecStep::layout): bit 0 = x is NHWC -> implicit-GEMM kernel; bit 1 = y (and the residual) are NHWC
bool runConvBnAct(const OpVec &ops, const RuntimeObj *ctx, int layout) {
    auto conv = as<ConvObj>(ops[0]);
    auto bn = ops.size() > 1 ? as<BatchNormObj>(ops[1]) : nullptr;
    Operator add, relu;
    for (size_t i = 2; i < ops.size(); ++i) {
        if (ops[i]->getOpType() == OpType::Add) add = ops[i];
        if (ops[i]->getOpType() == OpType::Relu) relu = ops[i];
    }
    auto x = conv->getInputs(0), w = conv->getInputs(1);
    auto [n, c, h, wd, f, r, s] = conv->getNCHWFRS();
    auto [ph, pw, sh, sw, dh, dw] = conv->getPadStrideDilation();
    int g = conv->getNumGroups();
    for (int i = 1; bn && i <= 4; ++i)
        if (bn->getInputs(i)->getDType() != DataType::Float32) {
            IT_ASSERT(!layout, "NHWC conv step with non-fp32 BatchNorm statistics");
            return false;
        }
    Tensor res;
    if (add) {
        Tensor prev = bn->getOutput();
        res = add->getInputs(0) == prev ? add->getInputs(1) : add->getInputs(0);
    }
    const float *bm = bn ? bn->getInputs(1)->getRawDataPtr<float *>() : nullptr, *bv = bn ? bn->getInputs(2)->getRawDataPtr<float *>() : nullptr,
                *bs = bn ? bn->getInputs(3)->getRawDataPtr<float *>() : nullptr, *bb = bn ? bn->getInputs(4)->getRawDataPtr<float *>() : nullptr;
    const float eps = bn ? bn->getEps() : 0.f;
    if (layout & 1) {
        int64_t wsb = it_b200_conv2d_nhwc_workspace(DTI(x), c, f, r, s);
        void *ws = nullptr;
        if (wsb) {
            auto packed = RT(ctx)->findPackedFilter(P(w));  // repacked at the start of this step (prepConvFilters)
            if (packed.first && (int64_t)packed.second >= wsb) {
                ws = packed.first;
                wsb = -(int64_t)packed.second;
            } else {
                ws = RT(ctx)->getWorkspace((size_t)wsb);  // a step executed on its own (tune): repack in place
            }
        }
        CK(it_b200_conv2d_nhwc(DTI(x), P(x), P(w), P(ops.back()->getOutput()), (layout & 2) ? 1 : 0, n, c, h, wd, f, r, s, ph, pw, sh, sw, dh,
                               dw, bm, bv, bs, bb, eps, res ? P(res) : nullptr, relu ? 1 : 0, ws, wsb, S()), ops.back());
        return true;
    }
    int64_t wsb = it_b200_conv2d_workspace(DTI(x), n, c, h, wd, f, r, s, ph, pw, sh, sw, dh, dw, g);
    void *ws = wsb ? RT(ctx)->getWorkspace((size_t)wsb) : nullptr;
    if ((layout & 2) && !res && it_b200_conv2d_stem_supported(DTI(x), c, f, r, s, ph, pw, sh, sw, dh, dw, g)) {
        CK(it_b200_conv2d_stem(DTI(x), P(x), P(w), P(ops.back()->getOutput()), n, c, h, wd, f, r, s, ph, pw, sh, sw, bm, bv, bs, bb, eps,
                               relu ? 1 : 0, S()), ops.back());
        return true;
    }
    if (layout & 2) {
        int rc = it_b200_conv2d_fused_nhwc_out(DTI(x), P(x), P(w), P(ops.back()->getOutput()), n, c, h, wd, f, r, s, ph, pw, sh, sw, dh, dw, g,
                                               bm, bv, bs, bb, eps, res ? P(res) : nullptr, relu ? 1 : 0, ws, wsb, S());
        IT_ASSERT(rc != 2, "NHWC-output conv step on a shape the im2col GEMM does not scatter (schedule / kernel disagree)");
        CK(rc, ops.back());
        return true;
    }
    IT_ASSERT(bn, "runConvBnAct: a lone Conv runs through its registered kernel");
    int rc = it_b200_conv2d_fused(DTI(x), P(x), P(w), P(ops.back()->getOutput()), n, c, h, wd, f, r, s, ph, pw, sh, sw, dh,
                                  dw, g, bn->getInputs(1)->getRawDataPtr<float *>(),
                                  bn->getInputs(2)->getRawDataPtr<float *>(), bn->getInputs(3)->getRawDataPtr<float *>(),
                                  bn->getInputs(4)->getRawDataPtr<float *>(), bn->getEps(), res ? P(res) : nullptr,
                                  relu ? 1 : 0, ws, wsb, S());
    if (rc == 2) return false;
    CK(rc, ops.back());
    return true;
}

// Step i is a decode attention launch: tell it which weights the next GEMM will stream (it_b200_l2_prefetch_hint) -- the attention
// kernel leaves ~30 % of HBM idle and the next GEMM cannot become resident beside it, so its weights are prefetched into L2 meanwhile
void setPrefetchHint(const vector<ExecStep> &sched, size_t i) {
    const auto &st = sched[i];
    if (st.ops.back()->getOpType() != OpType::AttentionKVCache) return;
    for (size_t j = i + 1; j < sched.size() && j <= i + 6; ++j) {
        const auto &nx = sched[j];
        if (nx.kind == ExecStep::Alias) continue;
        if (nx.ops[0]->getOpType() != OpType::MatMul) return;
        auto w = nx.ops[0]->getInputs(1);
        if (!w->isWeight() || w->getBytes() > (size_t)96 << 20) return;  // (leave room in the 126 MB L2 for the stream itself)
        it_b200_l2_prefetch_hint(P(w), (long long)w->getBytes());
        return;
    }
}

// every NHWC conv of the schedule with filters larger than 1x1: re-order all the filter banks in one launch, into buffers the
// runtime keeps per weight tensor (so no conv waits for a repack kernel of its own)
void prepConvFilters(const vector<ExecStep> &sched, const RuntimeObj *ctx) {
    vector<const void *> src[2];
    vector<void *> dst[2];
    vector<int> nF[2], nC[2], nR[2], nS[2];
    for (auto &st : sched) {
        if (!(st.layout & 1) || st.ops[0]->getOpType() != OpType::Conv) continue;
        auto conv = as<ConvObj>(st.ops[0]);
        auto x = conv->getInputs(0), w = conv->getInputs(1);
        auto [n, c, h, wd, f, r, s] = conv->getNCHWFRS();
        (void)n; (void)h; (void)wd;
        const int64_t bytes = it_b200_conv2d_nhwc_workspace(DTI(x), c, f, r, s);
        if (bytes == 0) continue;
        const int k = DTI(x) == ITB_F16 ? 0 : 1;
        src[k].push_back(P(w));
        dst[k].push_back(RT(ctx)->packedFilterBuffer(P(w), (size_t)bytes));
        nF[k].push_back(f);
        nC[k].push_back(c);
        nR[k].push_back(r);
        nS[k].push_back(s);
    }
    for (int k = 0; k < 2; ++k)
        if (!src[k].empty())
            CK(it_b200_conv_repack_filters(k == 0 ? ITB_F16 : ITB_BF16, (int)src[k].size(), src[k].data(), dst[k].data(), nF[k].data(),
                                           nC[k].data(), nR[k].data(), nS[k].data(), S()), sched.front().ops.back());
}

// MaxPool / AveragePool inside the NHWC domain
void runPoolNhwc(const Operator &_op, const RuntimeObj *) {
    auto op = as<PoolingObj>(_op);
    auto x = op->getInputs(0), y = op->getOutput();
    const auto &d = x->getDims();
    const auto &o = y->getDims();
    CK(it_b200_pool2d_nhwc(DTI(x), _op->getOpType() == OpType::MaxPool, P(x), P(y), d[0], d[1], d[2], d[3], op->getKh(), op->getKw(),
                           op->getDh(), op->getDw(), op->getPh(), op->getPw(), op->getSh(), op->getSw(), o[2], o[3], S()), _op);
}

// AllReduceSum -> Add(residual) [-> RMSNorm] through the one-shot NVLink kernel
bool runAllReduceAddNorm(const OpVec &ops, const RuntimeObj *ctx) {
    auto rt = RT(ctx);
    if (!rt->hasPeerComm()) return false;
    const auto &ar = ops[0], &add = ops[1];
    auto in = ar->getInputs(0);
    auto dt = in->getDType();
    if (!dt.isFloat()) return false;
    int hidden = in->getDims().back();
    int64_t tokens = (int64_t)in->size() / hidden;
    if (tokens > 64 || (int64_t)hidden * (int64_t)dt.getSize() > 16384 || (hidden * dt.getSize()) % 16 != 0) return false;
    auto arOut = ar->getOutput();
    auto res = add->getInputs(0) == arOut ? add->getInputs(1) : add->getInputs(0);
    const void *nw = nullptr;
    void *on = nullptr;
    if (ops.size() > 2) {
        nw = P(ops[2]->getInputs(1));
        on = P(ops[2]->getOutput());
    }
    CK(it_b200_allreduce_fused(dt.getIndex(), P(in), P(res), nw, P(add->getOutput()), on, (int)tokens, hidden,
                               rt->peerWorkspaces(), rt->p2pWorldSize(), rt->p2pRank(), rt->p2pTimeoutFlagDevice(), S()), ar);
    return true;
}
#endif  // !ITB_SEAM_A
}  // namespace b200

// MatMul: tune() times the production dispatch and each GEMM kernel pinned on the operator's own shape and records the winner
// (MatmulPerfRecordObj); compute(op, record) re-applies it.  Reference: matmul.cc:187-208 (tune over cuBLAS algorithms).
class MatmulB200 : public CudaKernelWithoutConfig {
    void compute(const Operator &_op, const RuntimeObj *ctx) const override {
        b200::runMatmul(_op, ctx, nullptr, nullptr);
    }
#ifndef ITB_SEAM_A  // (the reference's PerfRecord types differ: under Seam A the base class's timing-only tune() stays)
    void compute(const Operator &_op, const PerfRecord &record, const RuntimeObj *ctx) const override {
        auto mr = std::dynamic_pointer_cast<MatmulPerfRecordObj>(record);
        if (!mr || (mr->impl == 0 && mr->nb == 0)) return compute(_op, ctx);
        it_b200_matmul_select(mr->impl, mr->nb);
        try {
            b200::runMatmul(_op, ctx, nullptr, nullptr);
        } catch (...) {
            it_b200_matmul_select(0, 0);
            throw;
        }
        it_b200_matmul_select(0, 0);
    }
    PerfRecord tune(const Operator &_op, const RuntimeObj *ctx) const override {
        auto best = make_ref<MatmulPerfRecordObj>();
        best->time = 1e30;
        if (as<MatmulObj>(_op)->getWScale()) {  // FP8 weights: one kernel
            best->time = CudaKernelWithoutConfig::tune(_op, ctx)->time;
            return best;
        }
        static const int cand[][2] = {{0, 0}, {1, 1}, {1, 2}, {2, 0}};
        for (auto &c : cand) {
            it_b200_matmul_select(c[0], c[1]);
            double t = 1e30;
            try {
                t = CudaKernelWithoutConfig::tune(_op, ctx)->time;
            } catch (...) {
                it_b200_matmul_select(0, 0);
                throw;
            }
            if (t < best->time) {
                best->time = t;
                best->impl = c[0];
                best->nb = c[1];
            }
        }
        it_b200_matmul_select(0, 0);
        return best;
    }
#endif
};
class ConvB200 : public CudaKernelWithoutConfig {
    void compute(const Operator &_op, const RuntimeObj *ctx) const override {
        auto op = as<ConvObj>(_op);
        auto x = op->getInputs(0), w = op->getInputs(1);
        auto [n, c, h, wd, f, r, s] = op->getNCHWFRS();
        auto [ph, pw, sh, sw, dh, dw] = op->getPadStrideDilation();
        int g = op->getNumGroups();
        int64_t wsb = it_b200_conv2d_workspace(DTI(x), n, c, h, wd, f, r, s, ph, pw, sh, sw, dh, dw, g);
        void *ws = wsb ? RT(ctx)->getWorkspace((size_t)wsb) : nullptr;
        CK(it_b200_conv2d(DTI(x), P(x), P(w), P(op->getOutput()), n, c, h, wd, f, r, s, ph, pw, sh, sw, dh, dw, g, ws,
                          wsb, S()), _op);
    }
};
class AttentionKVCacheB200 : public CudaKernelWithoutConfig {
    void compute(const Operator &op, const RuntimeObj *ctx) const override {
        auto kc = op->getInputs(0), vc = op->getInputs(1), q = op->getInputs(2), k = op->getInputs(3),
             v = op->getInputs(4), pos = op->getInputs(5);
        const auto &d = kc->getDims();
        int64_t wsb = it_b200_attention_kvcache_workspace(d[0], d[1], d[2], d[3]);
        void *ws = wsb ? RT(ctx)->getWorkspace((size_t)wsb) : nullptr;
        CK(it_b200_attention_kvcache(DTI(q), P(kc), P(vc), P(q), P(k), P(v), P(pos),
#ifdef ITB_SEAM_A
                                     DTI(pos) | (pos->getSource() || kc->getSource() || vc->getSource() ? ITB_POS_IN_STEP : 0),
#else
                                     b200::attnPosFlags(op, nullptr),
#endif
                                     P(op->getOutput()), d[0],
                                     d[1], d[2], d[3], ws, wsb, S()), op);
    }
};

// ---------------------------------------------------------------- collectives (NCCL on the runtime stream,
// capturable; reference all_reduce.cc:8-63, all_gather.cc:8-43 -- the latter's stream-0 + memcpy fan-out is
// a defect (quirk q7) and is not reproduced)
#ifndef ITB_SEAM_A
static ncclDataType_t ncclType(DataType dt) {
    if (dt == DataType::Float32) return ncclFloat;
    if (dt == DataType::Float16) return ncclHalf;
    if (dt == DataType::BFloat16) return ncclBfloat16;
    if (dt == DataType::Int8) return ncclInt8;
    if (dt == DataType::Int32) return ncclInt32;
    if (dt == DataType::Int64) return ncclInt64;
    throw Exception("collective: unsupported dtype " + dt.toString());
}
class AllReduceB200 : public CudaKernelWithoutConfig {
    void compute(const Operator &op, const RuntimeObj *ctx) const override {
        auto x = op->getInputs(0), y = op->getOutput();
        auto comm = (ncclComm_t)RT(ctx)->getCommunicator().getNcclComm();
        ncclRedOp_t red;
        switch (op->getOpType().underlying()) {
        case OpType::AllReduceSum: red = ncclSum; break;
        case OpType::AllReduceProd: red = ncclProd; break;
        case OpType::AllReduceMin: red = ncclMin; break;
        case OpType::AllReduceMax: red = ncclMax; break;
        default: red = ncclAvg;
        }
        ncclResult_t r = nccl().AllReduce(P(x), P(y), x->size(), ncclType(x->getDType()), red, comm,
                                       CUDAStream::getCurrentStream());
        IT_ASSERT(r == ncclSuccess, string("ncclAllReduce: ") + nccl().GetErrorString(r));
    }
};
class AllGatherB200 : public CudaKernelWithoutConfig {
    void compute(const Operator &op, const RuntimeObj *ctx) const override {
        auto x = op->getInputs(0);
        auto rt = RT(ctx);
        auto &c = rt->getCommunicator();
        int world = c.getWorldSize();
        IT_ASSERT((int)op->getOutputs().size() == world, "AllGather: one output per rank");
        // outputs planned back-to-back -> gather straight into them; otherwise through the workspace
        bool contiguous = true;
        char *base = op->getOutput(0)->getRawDataPtr<char *>();
        for (int i = 0; i < world; ++i)
            contiguous = contiguous && op->getOutput(i)->getRawDataPtr<char *>() == base + (size_t)i * x->getBytes();
        auto st = CUDAStream::getCurrentStream();
        void *dst = contiguous ? (void *)base : rt->getWorkspace(x->getBytes() * world);
        ncclResult_t r = nccl().AllGather(P(x), dst, x->size(), ncclType(x->getDType()), (ncclComm_t)c.getNcclComm(), st);
        IT_ASSERT(r == ncclSuccess, string("ncclAllGather: ") + nccl().GetErrorString(r));
        if (!contiguous)
            for (int i = 0; i < world; ++i)
                CK(it_b200_copy((char *)dst + (size_t)i * x->getBytes(), P(op->getOutput(i)), (int64_t)x->getBytes(),
                                st), op);
    }
};

#endif  // !ITB_SEAM_A (collectives: the reference builds them only with BUILD_DIST)

}  // namespace infini

#define REG(OP, K, NAME) REGISTER_KERNEL(Device::CUDA, OpType::OP, K, NAME)
REG(Relu, UnaryB200, "Relu_B200")
REG(Sigmoid, UnaryB200, "Sigmoid_B200")
REG(Tanh, UnaryB200, "Tanh_B200")
REG(Gelu, UnaryB200, "Gelu_B200")
REG(Silu, UnaryB200, "Silu_B200")
REG(Erf, UnaryB200, "Erf_B200")
REG(Neg, UnaryB200, "Neg_B200")
REG(Abs, UnaryB200, "Abs_B200")
REG(Sqrt, UnaryB200, "Sqrt_B200")
REG(HardSigmoid, UnaryB200, "HardSigmoid_B200")
REG(HardSwish, UnaryB200, "HardSwish_B200")
REG(Exp, UnaryB200, "Exp_B200")
REG(LeakyRelu, UnaryAlphaB200, "LeakyRelu_B200")
REG(Elu, UnaryAlphaB200, "Elu_B200")
REG(Add, ElementWiseB200, "Add_B200")
REG(Sub, ElementWiseB200, "Sub_B200")
REG(Mul, ElementWiseB200, "Mul_B200")
REG(Div, ElementWiseB200, "Div_B200")
REG(Pow, ElementWiseB200, "Pow_B200")
REG(Min, ElementWiseB200, "Min_B200")
REG(Max, ElementWiseB200, "Max_B200")
REG(Less, ElementWiseB200, "Less_B200")
REG(Equal, ElementWiseB200, "Equal_B200")
REG(Greater, ElementWiseB200, "Greater_B200")
REG(Cast, CastB200, "Cast_B200")
REG(Where, WhereB200, "Where_B200")
REG(Expand, ExpandB200, "Expand_B200")
REG(Softmax, SoftmaxB200, "Softmax_B200")
REG(LayerNormalization, LayerNormB200, "LayerNorm_B200")
REG(RMSNorm, RMSNormB200, "RMSNorm_B200")
REG(RoPE, RoPEB200, "RoPE_B200")
REG(Transpose, TransposeB200, "Transpose_B200")
REG(DepthToSpace, DepthToSpaceB200, "DepthToSpace_B200")
REG(Concat, ConcatB200, "Concat_B200")
REG(Split, SplitB200, "Split_B200")
REG(Gather, GatherB200, "Gather_B200")
REG(Reshape, CopyB200, "Reshape_B200")
REG(Flatten, CopyB200, "Flatten_B200")
REG(Identity, CopyB200, "Identity_B200")
REG(Squeeze, CopyB200, "Squeeze_B200")
REG(Unsqueeze, CopyB200, "Unsqueeze_B200")
REG(Slice, SliceB200, "Slice_B200")
REG(Pad, PadB200, "Pad_B200")
REG(ReduceMean, ReduceB200, "ReduceMean_B200")
REG(ReduceSum, ReduceB200, "ReduceSum_B200")
REG(MaxPool, PoolingB200, "MaxPool_B200")
REG(AveragePool, PoolingB200, "AvgPool_B200")
REG(BatchNormalization, BatchNormB200, "BatchNorm_B200")
REG(MatMul, MatmulB200, "Matmul_B200_tma")  // decode shapes: TMA + mma.sync (gemm_skinny.cu); the rest: tcgen05/TMEM (gemm_tc.cu)
REG(Conv, ConvB200, "Conv_B200_im2col_gemm")
REG(AttentionKVCache, AttentionKVCacheB200, "AttentionKVCache_B200")
#ifndef ITB_SEAM_A
REG(AllReduceSum, AllReduceB200, "AllReduceSum_B200")
REG(AllReduceProd, AllReduceB200, "AllReduceProd_B200")
REG(AllReduceMin, AllReduceB200, "AllReduceMin_B200")
REG(AllReduceMax, AllReduceB200, "AllReduceMax_B200")
REG(AllReduceAvg, AllReduceB200, "AllReduceAvg_B200")
REG(AllGather, AllGatherB200, "AllGather_B200")
#endif
