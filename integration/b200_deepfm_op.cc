// TensorFlow custom-op translation unit for libdeepfm_b200.so (BASELINE.json north_star: "calls hand-written sm_100a
// CUDA through a thin C-ABI shim loaded as a TF custom op").  NOT compiled in this repository: the image has no
// TensorFlow headers / libtensorflow_framework (SURVEY.md §8c); a maintainer of the reference builds it with
//
//   TF_CFLAGS=$(python -c 'import tensorflow as tf; print(" ".join(tf.sysconfig.get_compile_flags()))')
//   TF_LFLAGS=$(python -c 'import tensorflow as tf; print(" ".join(tf.sysconfig.get_link_flags()))')
//   g++ -std=c++14 -shared -fPIC integration/b200_deepfm_op.cc -o b200_deepfm_op.so -I include $TF_CFLAGS $TF_LFLAGS \
//       -L recommender_tensorflow_b200 -ldeepfm_b200 -DGOOGLE_CUDA=1
//
// and uses it inside trainers/deep_fm.py:model_fn in place of the graph built at trainers/deep_fm.py:36-125:
//
//   mod = tf.load_op_library("b200_deepfm_op.so")
//   loss, logits = mod.b200_deep_fm_train_step(handle=h, int_columns=[...], string_columns=[...], numeric=[...], labels=y)
//   train_op = tf.group(loss.op, tf.assign_add(tf.train.get_global_step(), 1))
//   return tf.estimator.EstimatorSpec(mode, loss=loss, train_op=train_op, predictions={"logits": logits, ...})
//
// The handle is created once per model instance (Python side, ctypes or a resource op) from the feature-column
// descriptors of trainers/ml_100k.py:18-39 and the params of trainers/deep_fm.py:13-26; it is passed to the ops as an
// int64 scalar.  Every op enqueues on TF's own CUDA stream: there is no hidden synchronisation.
#include <cstdint>
#include <vector>

#include "tensorflow/core/framework/op.h"
#include "tensorflow/core/framework/op_kernel.h"
#include "tensorflow/core/framework/shape_inference.h"
#include "tensorflow/core/util/gpu_kernel_helper.h"

#include "deepfm_b200.h"

namespace tf = tensorflow;

REGISTER_OP("B200DeepFmTransform")
    .Input("handle: int64")
    .Input("int_columns: n_int * int32")
    .Input("string_bytes: n_str * uint8")
    .Input("string_offsets: n_str * int32")
    .Attr("n_int: int >= 0")
    .Attr("n_str: int >= 0")
    .Attr("cat_order: list(int)")          // for every model-order categorical column: index into int (>= 0) or ~index into str (< 0)
    .Output("ids: int32")                 // [B, n_slots]
    .SetShapeFn([](tf::shape_inference::InferenceContext* c) { c->set_output(0, c->UnknownShapeOfRank(2)); return tf::Status::OK(); });

REGISTER_OP("B200DeepFmTrainStep")
    .Input("handle: int64")
    .Input("int_columns: n_int * int32")
    .Input("string_bytes: n_str * uint8")
    .Input("string_offsets: n_str * int32")
    .Input("numeric: n_num * float")
    .Input("labels: float")
    .Attr("n_int: int >= 0")
    .Attr("n_str: int >= 0")
    .Attr("n_num: int >= 0")
    .Attr("cat_order: list(int)")
    .Output("loss: float")                // scalar
    .Output("logits: float")              // [B]
    .SetIsStateful()
    .SetShapeFn([](tf::shape_inference::InferenceContext* c) {
        c->set_output(0, c->Scalar());
        c->set_output(1, c->UnknownShapeOfRank(1));
        return tf::Status::OK();
    });

REGISTER_OP("B200DeepFmForward")
    .Input("handle: int64")
    .Input("int_columns: n_int * int32")
    .Input("string_bytes: n_str * uint8")
    .Input("string_offsets: n_str * int32")
    .Input("numeric: n_num * float")
    .Attr("n_int: int >= 0")
    .Attr("n_str: int >= 0")
    .Attr("n_num: int >= 0")
    .Attr("cat_order: list(int)")
    .Output("logits: float")
    .SetIsStateful()
    .SetShapeFn([](tf::shape_inference::InferenceContext* c) { c->set_output(0, c->UnknownShapeOfRank(1)); return tf::Status::OK(); });

namespace {

// gathers the device pointers of the op's inputs into the dfm_raw_batch the C ABI takes (caller-owned buffers)
struct Batch {
    std::vector<const void*> cat;
    std::vector<const int32_t*> off;
    std::vector<const float*> num;
    dfm_raw_batch raw;
};

tf::Status Collect(tf::OpKernelContext* ctx, const std::vector<int>& cat_order, bool with_num, bool with_labels, Batch* b) {
    tf::OpInputList ints, sbytes, soffs, nums;
    TF_RETURN_IF_ERROR(ctx->input_list("int_columns", &ints));
    TF_RETURN_IF_ERROR(ctx->input_list("string_bytes", &sbytes));
    TF_RETURN_IF_ERROR(ctx->input_list("string_offsets", &soffs));
    int64_t B = -1;
    for (int c : cat_order) {
        if (c >= 0) {
            b->cat.push_back(ints[c].flat<int32_t>().data());
            b->off.push_back(nullptr);
            B = ints[c].NumElements();
        } else {
            b->cat.push_back(sbytes[~c].flat<uint8_t>().data());
            b->off.push_back(soffs[~c].flat<int32_t>().data());
            B = soffs[~c].NumElements() - 1;
        }
    }
    if (with_num) {
        TF_RETURN_IF_ERROR(ctx->input_list("numeric", &nums));
        for (int j = 0; j < nums.size(); ++j) { b->num.push_back(nums[j].flat<float>().data()); B = nums[j].NumElements(); }
    }
    if (B <= 0) return tf::errors::InvalidArgument("empty batch");
    b->raw.batch_size = static_cast<int32_t>(B);
    b->raw.cat_data = b->cat.data();
    b->raw.cat_offsets = b->off.data();
    b->raw.num_data = b->num.data();
    b->raw.labels = nullptr;
    // per-example weights (dfm_raw_batch.weights) are read only by handles created with dfm_config.weighted != 0; this
    // op creates unweighted handles and has no weights input yet
    b->raw.weights = nullptr;
    if (with_labels) {
        // float32 labels as they are: 0/1 for a handle with the logistic head, any value (the rating) for one created
        // with dfm_config.head = DFM_HEAD_SQUARED; the head belongs to the handle, the op needs no attr for it
        const tf::Tensor* y;
        TF_RETURN_IF_ERROR(ctx->input("labels", &y));
        b->raw.labels = y->flat<float>().data();
    }
    return tf::Status::OK();
}

dfm_handle* HandleOf(tf::OpKernelContext* ctx) { return reinterpret_cast<dfm_handle*>(ctx->input(0).scalar<tf::int64>()()); }
void* StreamOf(tf::OpKernelContext* ctx) { return ctx->eigen_device<Eigen::GpuDevice>().stream(); }

class TrainStepOp : public tf::OpKernel {
 public:
    explicit TrainStepOp(tf::OpKernelConstruction* c) : tf::OpKernel(c) { OP_REQUIRES_OK(c, c->GetAttr("cat_order", &cat_order_)); }
    void Compute(tf::OpKernelContext* ctx) override {
        Batch b;
        OP_REQUIRES_OK(ctx, Collect(ctx, cat_order_, true, true, &b));
        tf::Tensor *loss, *logits;
        OP_REQUIRES_OK(ctx, ctx->allocate_output(0, tf::TensorShape({}), &loss));
        OP_REQUIRES_OK(ctx, ctx->allocate_output(1, tf::TensorShape({b.raw.batch_size}), &logits));
        dfm_handle* h = HandleOf(ctx);
        const int rc = dfm_train_step(h, &b.raw, loss->flat<float>().data(), logits->flat<float>().data(), StreamOf(ctx));
        OP_REQUIRES(ctx, rc == DFM_OK, tf::errors::Internal("dfm_train_step: ", dfm_last_error(h)));
    }
 private:
    std::vector<int> cat_order_;
};

class ForwardOp : public tf::OpKernel {
 public:
    explicit ForwardOp(tf::OpKernelConstruction* c) : tf::OpKernel(c) { OP_REQUIRES_OK(c, c->GetAttr("cat_order", &cat_order_)); }
    void Compute(tf::OpKernelContext* ctx) override {
        Batch b;
        OP_REQUIRES_OK(ctx, Collect(ctx, cat_order_, true, false, &b));
        tf::Tensor* logits;
        OP_REQUIRES_OK(ctx, ctx->allocate_output(0, tf::TensorShape({b.raw.batch_size}), &logits));
        dfm_handle* h = HandleOf(ctx);
        const int rc = dfm_forward(h, &b.raw, logits->flat<float>().data(), StreamOf(ctx));
        OP_REQUIRES(ctx, rc == DFM_OK, tf::errors::Internal("dfm_forward: ", dfm_last_error(h)));
    }
 private:
    std::vector<int> cat_order_;
};

class TransformOp : public tf::OpKernel {
 public:
    explicit TransformOp(tf::OpKernelConstruction* c) : tf::OpKernel(c) { OP_REQUIRES_OK(c, c->GetAttr("cat_order", &cat_order_)); }
    void Compute(tf::OpKernelContext* ctx) override {
        Batch b;
        OP_REQUIRES_OK(ctx, Collect(ctx, cat_order_, false, false, &b));
        dfm_handle* h = HandleOf(ctx);
        tf::Tensor* ids;
        OP_REQUIRES_OK(ctx, ctx->allocate_output(0, tf::TensorShape({b.raw.batch_size, dfm_num_slots(h)}), &ids));
        const int rc = dfm_transform(h, &b.raw, ids->flat<int32_t>().data(), StreamOf(ctx));
        OP_REQUIRES(ctx, rc == DFM_OK, tf::errors::Internal("dfm_transform: ", dfm_last_error(h)));
    }
 private:
    std::vector<int> cat_order_;
};

}  // namespace

REGISTER_KERNEL_BUILDER(Name("B200DeepFmTrainStep").Device(tf::DEVICE_GPU).HostMemory("handle"), TrainStepOp);
REGISTER_KERNEL_BUILDER(Name("B200DeepFmForward").Device(tf::DEVICE_GPU).HostMemory("handle"), ForwardOp);
REGISTER_KERNEL_BUILDER(Name("B200DeepFmTransform").Device(tf::DEVICE_GPU).HostMemory("handle"), TransformOp);
