#!/usr/bin/env python
"""Generates jni/se_jni.cpp and scala/org/apache/spark/ml/se/SeNative.scala from ONE table, so the JNI symbol list, the
Scala @native list and the bound subset of include/se_abi.h cannot drift apart (tests/test_host_cpu.py re-runs the
generator and compares; it also checks that every ABI function is either bound or listed in NOT_BOUND with a reason).

    python jni/gen_jni.py            # rewrites both files

Conventions of the generated shim (ADVICE r1: no JNI critical regions across blocking calls):
  * small arrays (alpha, step, gradients, tree nodes, weights) are COPIED with Get/Set<Type>ArrayRegion into native
    buffers before the ABI call and copied back afterwards — nothing is pinned while a kernel, a collective or a
    cudaMalloc runs, so the GC is never locked out;
  * bulk transfers have two forms: `upload/download(float[] ...)` stream through a native staging chunk with
    Get/SetFloatArrayRegion, and `uploadDirect/downloadDirect(java.nio.ByteBuffer ...)` take a DIRECT buffer —
    ideally one returned by hostAlloc (page-locked), which the DMA engine reads without any copy;
  * scalar outputs come back as the return value (one) or a double[] (several, ints widened);
  * non-zero status -> IllegalArgumentException (SE_ERR_ARG) / RuntimeException (others) with se_last_error's text.
"""
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# kind -> (jni C type, scala type)
SCALARS = {"i32": ("jint", "Int"), "i64": ("jlong", "Long"), "u64": ("jlong", "Long"), "f32": ("jfloat", "Float"),
           "f64": ("jdouble", "Double"), "bool": ("jboolean", "Boolean"), "str": ("jstring", "String")}
ARRAYS = {"in_f64": ("jdoubleArray", "Array[Double]", "double", "Double"), "in_f32": ("jfloatArray", "Array[Float]", "float", "Float"),
          "in_i32": ("jintArray", "Array[Int]", "int32_t", "Int"), "out_f64": ("jdoubleArray", "Array[Double]", "double", "Double"),
          "io_f64": ("jdoubleArray", "Array[Double]", "double", "Double")}
OUTS = {"o_f64": "double", "o_i32": "int", "o_i64": "int64_t"}

# (scala name, abi function, [(param name, kind)...], doc)
TABLE = [
    ("abiVersion", "se_abi_version", [], "ABI version of the loaded library"),
    ("deviceCount", "se_device_count", [("out", "o_i32")], ""),
    ("ctxDestroy", "se_ctx_destroy", [("ctx", "ctx")], ""),
    ("ctxSync", "se_ctx_sync", [("ctx", "ctx")], ""),
    ("ctxDevice", "se_ctx_device", [("ctx", "ctx"), ("device", "o_i32")], ""),
    ("ctxLaunchCount", "se_ctx_launch_count", [("ctx", "ctx"), ("out", "o_i64")], ""),
    ("ctxLastMs", "se_ctx_last_ms", [("ctx", "ctx"), ("out", "o_f64")], ""),
    ("ctxSetTiming", "se_ctx_set_timing", [("ctx", "ctx"), ("on", "bool")], ""),
    ("ctxTimerStart", "se_ctx_timer_start", [("ctx", "ctx")], ""),
    ("ctxTimerStop", "se_ctx_timer_stop", [("ctx", "ctx"), ("ms", "o_f64")], ""),
    ("ctxKernelTiming", "se_ctx_kernel_timing", [("ctx", "ctx"), ("on", "bool")], ""),
    ("ctxKernelTime", "se_ctx_kernel_time", [("ctx", "ctx"), ("family", "i32"), ("totalMs", "o_f64"), ("launches", "o_i64")],
     "(totalMs, launches)"),
    ("ctxKernelTimeReset", "se_ctx_kernel_time_reset", [("ctx", "ctx")], ""),
    ("ctxSetOption", "se_ctx_set_option", [("ctx", "ctx"), ("key", "str"), ("value", "f64")], ""),
    ("ctxGetOption", "se_ctx_get_option", [("ctx", "ctx"), ("key", "str"), ("value", "o_f64")], ""),
    ("commP2pActive", "se_comm_p2p_active", [("ctx", "ctx"), ("active", "o_i32")], ""),
    ("commClearError", "se_comm_clear_error", [("ctx", "ctx")], ""),
    ("commDestroy", "se_comm_destroy", [("ctx", "ctx")], ""),
    ("commInfo", "se_comm_info", [("ctx", "ctx"), ("nranks", "o_i32"), ("rank", "o_i32")], "(nranks, rank)"),
    ("commAllreduceHost", "se_comm_allreduce_host", [("ctx", "ctx"), ("values", "io_f64"), ("count", "i32")], "in place"),
    ("slotAlloc", "se_slot_alloc", [("ctx", "ctx"), ("slot", "i32"), ("count", "i64")], ""),
    ("slotAlloc2d", "se_slot_alloc2d", [("ctx", "ctx"), ("slot", "i32"), ("rows", "i64"), ("cols", "i64")], ""),
    ("slotLayout", "se_slot_layout", [("ctx", "ctx"), ("slot", "i32"), ("rows", "o_i64"), ("cols", "o_i64"), ("ld", "o_i64")],
     "(rows, cols, ld)"),
    ("slotFree", "se_slot_free", [("ctx", "ctx"), ("slot", "i32")], ""),
    ("fill", "se_fill", [("ctx", "ctx"), ("slot", "i32"), ("value", "f32"), ("count", "i64"), ("offset", "i64")], ""),
    ("copySlot", "se_copy_slot", [("ctx", "ctx"), ("dstSlot", "i32"), ("srcSlot", "i32")], ""),
    ("fillSynthetic", "se_fill_synthetic", [("ctx", "ctx"), ("slot", "i32"), ("kind", "i32"), ("seed", "u64"), ("a", "f64"),
                                            ("b", "f64"), ("count", "i64"), ("offset", "i64")], ""),
    ("quantile", "se_quantile", [("ctx", "ctx"), ("which", "i32"), ("slot", "i32"), ("count", "i64"), ("q", "f64"), ("out", "o_f64")],
     "exact quantile: which = 0 slot values, 1 |y - F| (huber delta)"),
    ("slotSum", "se_slot_sum", [("ctx", "ctx"), ("slot", "i32"), ("count", "i64"), ("out", "o_f64")], ""),
    ("gbmConfigure", "se_gbm_configure", [("ctx", "ctx"), ("nTrain", "i64"), ("nValid", "i64"), ("dim", "i32"), ("loss", "i32"),
                                          ("param", "f64"), ("hasWeights", "bool")], ""),
    ("gbmSetLossParam", "se_gbm_set_loss_param", [("ctx", "ctx"), ("param", "f64")], ""),
    ("gbmSetBag", "se_gbm_set_bag", [("ctx", "ctx"), ("on", "bool")], ""),
    ("gbmPseudoResiduals", "se_gbm_pseudo_residuals", [("ctx", "ctx"), ("newton", "bool"), ("sumHess", "out_f64")], ""),
    ("gbmLinesearchEval", "se_gbm_linesearch_eval", [("ctx", "ctx"), ("alpha", "in_f64"), ("loss", "o_f64"), ("grad", "out_f64")],
     "DiffFunction.calculate(alpha): returns lossSum/weightSum, fills grad (nullable: objective only)"),
    ("gbmLinesearchStats", "se_gbm_linesearch_stats", [("ctx", "ctx"), ("stats4", "out_f64")], ""),
    ("gbmUpdate", "se_gbm_update", [("ctx", "ctx"), ("step", "in_f64"), ("flags", "i32"), ("lossSum", "o_f64"), ("sumHess", "out_f64")], ""),
    ("gbmMeanLoss", "se_gbm_mean_loss", [("ctx", "ctx"), ("which", "i32"), ("out", "o_f64")], ""),
    ("gbmUpdateValidation", "se_gbm_update_validation", [("ctx", "ctx"), ("step", "in_f64"), ("meanLoss", "o_f64")], ""),
    ("gbmLinesearchBrent", "se_gbm_linesearch_brent", [("ctx", "ctx"), ("lo", "f64"), ("hi", "f64"), ("start", "f64"), ("rel", "f64"),
                                                       ("absTol", "f64"), ("maxEval", "i32"), ("alpha", "o_f64"), ("loss", "o_f64"),
                                                       ("nEval", "o_i32")], "(alpha, objective, evaluations)"),
    ("gbmRound", "se_gbm_round", [("ctx", "ctx"), ("learningRate", "f64"), ("optimized", "bool"), ("tol", "f64"), ("maxIter", "i32"),
                                  ("flags", "i32"), ("alpha", "o_f64"), ("lossSum", "o_f64"), ("nEval", "o_i32")],
     "line search + update in one call (squared loss: ONE cooperative kernel launch): (alpha, lossSum, evaluations)"),
    ("gbmLinesearchEval2", "se_gbm_linesearch_eval2", [("ctx", "ctx"), ("alpha", "f64"), ("loss", "o_f64"), ("d1", "o_f64"), ("d2", "o_f64")],
     "(loss, first, second derivative along the direction)"),
    ("gbmLinesearchNewton", "se_gbm_linesearch_newton", [("ctx", "ctx"), ("lo", "f64"), ("hi", "f64"), ("start", "f64"), ("rel", "f64"),
                                                         ("absTol", "f64"), ("maxEval", "i32"), ("alpha", "o_f64"), ("loss", "o_f64"),
                                                         ("nEval", "o_i32")], "opt-in: (alpha, objective, evaluations)"),
    ("gbmRoundSquaredAsync", "se_gbm_round_squared_async", [("ctx", "ctx"), ("learningRate", "f64")], ""),
    ("gbmRoundResult", "se_gbm_round_result", [("ctx", "ctx"), ("alpha", "o_f64"), ("lossSum", "o_f64")], "(alpha, lossSum)"),
    ("boostConfigure", "se_boost_configure", [("ctx", "ctx"), ("n", "i64"), ("numClasses", "i32"), ("real", "bool")], ""),
    ("boostRealUpdate", "se_boost_real_update", [("ctx", "ctx"), ("sumWeights", "f64"), ("estErr", "o_f64"), ("newSum", "o_f64")],
     "(estimatorError, sumWeights')"),
    ("boostDiscreteError", "se_boost_discrete_error", [("ctx", "ctx"), ("sumWeights", "f64"), ("estErr", "o_f64")], ""),
    ("boostDiscreteUpdate", "se_boost_discrete_update", [("ctx", "ctx"), ("sumWeights", "f64"), ("beta", "f64"), ("newSum", "o_f64")], ""),
    ("boostregConfigure", "se_boostreg_configure", [("ctx", "ctx"), ("n", "i64")], ""),
    ("boostregMaxError", "se_boostreg_max_error", [("ctx", "ctx"), ("maxError", "o_f64")], ""),
    ("boostregError", "se_boostreg_error", [("ctx", "ctx"), ("sumWeights", "f64"), ("lossType", "i32"), ("maxError", "f64"),
                                            ("estErr", "o_f64")], ""),
    ("boostregUpdate", "se_boostreg_update", [("ctx", "ctx"), ("sumWeights", "f64"), ("lossType", "i32"), ("maxError", "f64"),
                                              ("beta", "f64"), ("newSum", "o_f64")], ""),
    ("aggConfigure", "se_agg_configure", [("ctx", "ctx"), ("kind", "i32"), ("numModels", "i32"), ("numClasses", "i32"), ("dim", "i32"),
                                          ("loss", "i32"), ("n", "i64")], ""),
    ("aggRun", "se_agg_run", [("ctx", "ctx"), ("weights", "in_f64"), ("init", "in_f64")], ""),
    ("treePredict", "se_tree_predict", [("ctx", "ctx"), ("which", "i32"), ("nNodes", "i32"), ("feature", "in_i32"), ("threshold", "in_f32"),
                                        ("left", "in_i32"), ("right", "in_i32"), ("value", "in_f32"), ("subspace", "in_i32"),
                                        ("nSubspace", "i32"), ("outSlot", "i32"), ("outRow", "i32")],
     "DecisionTreeRegressionModel.predict over the resident column-major feature matrix"),
    ("treePredictMulti", "se_tree_predict_multi", [("ctx", "ctx"), ("which", "i32"), ("nNodes", "i32"), ("feature", "in_i32"),
                                                   ("threshold", "in_f32"), ("left", "in_i32"), ("right", "in_i32"), ("values", "in_f32"),
                                                   ("nOut", "i32"), ("subspace", "in_i32"), ("nSubspace", "i32"), ("outSlot", "i32")], ""),
    ("forestPredict", "se_forest_predict", [("ctx", "ctx"), ("which", "i32"), ("nTrees", "i32"), ("offsets", "in_i32"), ("feature", "in_i32"),
                                            ("threshold", "in_f32"), ("left", "in_i32"), ("right", "in_i32"), ("value", "in_f32"),
                                            ("weights", "in_f64"), ("init", "f64"), ("outSlot", "i32"), ("outRow", "i32")],
     "GBMRegressionModel.predict / BaggingRegressionModel.predict for tree members: init + sum of weight * tree(x) in one pass"),
    ("forestClassify", "se_forest_classify", [("ctx", "ctx"), ("which", "i32"), ("kind", "i32"), ("numClasses", "i32"), ("dim", "i32"),
                                              ("loss", "i32"), ("nTrees", "i32"), ("offsets", "in_i32"), ("feature", "in_i32"),
                                              ("threshold", "in_f32"), ("left", "in_i32"), ("right", "in_i32"), ("leaf", "in_f32"),
                                              ("leafWidth", "i32"), ("weights", "in_f64"), ("init", "in_f64")],
     "predictRaw / probability / prediction of a classifier ensemble of tree members in one pass: RAW, PROB, LABEL slots"),
    ("forestWeightedMedian", "se_forest_weighted_median", [("ctx", "ctx"), ("which", "i32"), ("nTrees", "i32"), ("offsets", "in_i32"),
                                                           ("feature", "in_i32"), ("threshold", "in_f32"), ("left", "in_i32"),
                                                           ("right", "in_i32"), ("value", "in_f32"), ("weights", "in_f64"),
                                                           ("outSlot", "i32"), ("outRow", "i32")],
     "BoostingRegressionModel.predict (median) for tree members: weighted median of tree(x) in one pass"),
    ("linearPredict", "se_linear_predict", [("ctx", "ctx"), ("which", "i32"), ("nCoef", "i32"), ("coef", "in_f32"), ("intercept", "f32"),
                                            ("subspace", "in_i32"), ("outSlot", "i32"), ("outRow", "i32")], ""),
]

# hand-written natives (bulk transfers, handles, byte arrays): scala signature + which ABI functions they cover
HAND = [
    ("ctxCreate", "def ctxCreate(device: Int): Long", ["se_ctx_create"]),
    ("commUniqueId", "def commUniqueId(): Array[Byte]", ["se_comm_unique_id"]),
    ("commInit", "def commInit(ctx: Long, nranks: Int, rank: Int, id: Array[Byte]): Unit", ["se_comm_init"]),
    ("hostAlloc", "def hostAlloc(bytes: Long): java.nio.ByteBuffer // page-locked, direct: feed to uploadDirect/downloadDirect", ["se_host_alloc"]),
    ("hostFree", "def hostFree(buffer: java.nio.ByteBuffer): Unit", ["se_host_free"]),
    ("upload", "def upload(ctx: Long, slot: Int, host: Array[Float], count: Long, offset: Long): Unit", ["se_upload"]),
    ("uploadF64", "def uploadF64(ctx: Long, slot: Int, host: Array[Double], count: Long, offset: Long): Unit", ["se_upload_f64"]),
    ("uploadRowmajor", "def uploadRowmajor(ctx: Long, slot: Int, host: Array[Float], nRows: Long, d: Int, rowOffset: Long): Unit",
     ["se_upload_rowmajor"]),
    ("download", "def download(ctx: Long, slot: Int, host: Array[Float], count: Long, offset: Long): Unit", ["se_download"]),
    ("downloadScaled", "def downloadScaled(ctx: Long, slot: Int, scale: Double, host: Array[Float], count: Long, offset: Long): Unit",
     ["se_download_scaled"]),
    ("uploadDirect", "def uploadDirect(ctx: Long, slot: Int, host: java.nio.ByteBuffer, count: Long, offset: Long): Unit", ["se_upload"]),
    ("uploadRowmajorDirect", "def uploadRowmajorDirect(ctx: Long, slot: Int, host: java.nio.ByteBuffer, nRows: Long, d: Int, rowOffset: Long): Unit",
     ["se_upload_rowmajor"]),
    ("downloadDirect", "def downloadDirect(ctx: Long, slot: Int, host: java.nio.ByteBuffer, count: Long, offset: Long): Unit", ["se_download"]),
]

NOT_BOUND = {
    "se_last_error": "consumed inside the shim: its text becomes the exception message",
    "se_brent_minimize": "takes a C callback; the JVM side keeps commons-math3's BrentOptimizer (or calls gbmLinesearchBrent / gbmRound)",
    "se_slot_info": "returns a raw device pointer: not exposed to the JVM",
    "se_spark_bernoulli_sample": "restates Spark's BernoulliSampler for hosts WITHOUT Spark; the JVM side draws with Spark itself",
}

HAND_CPP = r'''
SE_JNI(jlong, ctxCreate)(JNIEnv* env, jclass, jint device) {
  se_ctx* ctx = nullptr;
  if (raise(env, nullptr, se_ctx_create(device, &ctx))) return 0;
  return reinterpret_cast<jlong>(ctx);
}
SE_JNI(jbyteArray, commUniqueId)(JNIEnv* env, jclass) {
  jbyte id[SE_COMM_ID_BYTES];
  if (raise(env, nullptr, se_comm_unique_id(id, SE_COMM_ID_BYTES))) return nullptr;
  jbyteArray out = env->NewByteArray(SE_COMM_ID_BYTES);
  env->SetByteArrayRegion(out, 0, SE_COMM_ID_BYTES, id);
  return out;
}
SE_JNI(void, commInit)(JNIEnv* env, jclass, jlong h, jint nranks, jint rank, jbyteArray id) {
  jbyte buf[SE_COMM_ID_BYTES] = {0};
  if (id) env->GetByteArrayRegion(id, 0, SE_COMM_ID_BYTES, buf);
  raise(env, H(h), se_comm_init(H(h), nranks, rank, id ? buf : nullptr, id ? SE_COMM_ID_BYTES : 0));
}
SE_JNI(jobject, hostAlloc)(JNIEnv* env, jclass, jlong bytes) {
  void* p = nullptr;
  if (raise(env, nullptr, se_host_alloc(bytes, &p))) return nullptr;
  return env->NewDirectByteBuffer(p, bytes);
}
SE_JNI(void, hostFree)(JNIEnv* env, jclass, jobject buffer) {
  if (buffer) raise(env, nullptr, se_host_free(env->GetDirectBufferAddress(buffer)));
}

// Bulk transfers from/to JVM arrays: streamed through a native chunk with Get/Set<Type>ArrayRegion (a bounded copy;
// no critical region is held while the DMA, a kernel or a collective runs).
namespace {
constexpr jlong kChunk = 1 << 22;  // elements per staging chunk (16 MB of floats)
}
SE_JNI(void, upload)(JNIEnv* env, jclass, jlong h, jint slot, jfloatArray host, jlong count, jlong offset) {
  std::vector<float> buf((size_t)(count < kChunk ? count : kChunk));
  for (jlong done = 0; done < count; done += kChunk) {
    const jlong m = (count - done < kChunk) ? count - done : kChunk;
    env->GetFloatArrayRegion(host, (jsize)done, (jsize)m, buf.data());
    if (env->ExceptionCheck()) return;
    if (raise(env, H(h), se_upload(H(h), slot, buf.data(), m, offset + done))) return;
  }
}
SE_JNI(void, uploadF64)(JNIEnv* env, jclass, jlong h, jint slot, jdoubleArray host, jlong count, jlong offset) {
  std::vector<double> buf((size_t)(count < kChunk ? count : kChunk));
  for (jlong done = 0; done < count; done += kChunk) {
    const jlong m = (count - done < kChunk) ? count - done : kChunk;
    env->GetDoubleArrayRegion(host, (jsize)done, (jsize)m, buf.data());
    if (env->ExceptionCheck()) return;
    if (raise(env, H(h), se_upload_f64(H(h), slot, buf.data(), m, offset + done))) return;
  }
}
SE_JNI(void, uploadRowmajor)(JNIEnv* env, jclass, jlong h, jint slot, jfloatArray host, jlong nRows, jint d, jlong rowOffset) {
  const jlong rows_per = (kChunk / (d > 0 ? d : 1)) > 0 ? (kChunk / (d > 0 ? d : 1)) : 1;
  std::vector<float> buf((size_t)((nRows < rows_per ? nRows : rows_per) * d));
  for (jlong done = 0; done < nRows; done += rows_per) {
    const jlong m = (nRows - done < rows_per) ? nRows - done : rows_per;
    env->GetFloatArrayRegion(host, (jsize)(done * d), (jsize)(m * d), buf.data());
    if (env->ExceptionCheck()) return;
    if (raise(env, H(h), se_upload_rowmajor(H(h), slot, buf.data(), m, d, rowOffset + done))) return;
  }
}
SE_JNI(void, download)(JNIEnv* env, jclass, jlong h, jint slot, jfloatArray host, jlong count, jlong offset) {
  std::vector<float> buf((size_t)(count < kChunk ? count : kChunk));
  for (jlong done = 0; done < count; done += kChunk) {
    const jlong m = (count - done < kChunk) ? count - done : kChunk;
    if (raise(env, H(h), se_download(H(h), slot, buf.data(), m, offset + done))) return;
    env->SetFloatArrayRegion(host, (jsize)done, (jsize)m, buf.data());
  }
}
SE_JNI(void, downloadScaled)(JNIEnv* env, jclass, jlong h, jint slot, jdouble scale, jfloatArray host, jlong count, jlong offset) {
  std::vector<float> buf((size_t)(count < kChunk ? count : kChunk));
  for (jlong done = 0; done < count; done += kChunk) {
    const jlong m = (count - done < kChunk) ? count - done : kChunk;
    if (raise(env, H(h), se_download_scaled(H(h), slot, scale, buf.data(), m, offset + done))) return;
    env->SetFloatArrayRegion(host, (jsize)done, (jsize)m, buf.data());
  }
}
// Direct ByteBuffers (ideally from hostAlloc: page-locked): zero-copy, nothing for the GC to move.
SE_JNI(void, uploadDirect)(JNIEnv* env, jclass, jlong h, jint slot, jobject host, jlong count, jlong offset) {
  const float* p = static_cast<const float*>(env->GetDirectBufferAddress(host));
  if (!p || env->GetDirectBufferCapacity(host) < count * 4) { raise_arg(env, "a direct ByteBuffer of >= 4*count bytes is required"); return; }
  raise(env, H(h), se_upload(H(h), slot, p, count, offset));
}
SE_JNI(void, uploadRowmajorDirect)(JNIEnv* env, jclass, jlong h, jint slot, jobject host, jlong nRows, jint d, jlong rowOffset) {
  const float* p = static_cast<const float*>(env->GetDirectBufferAddress(host));
  if (!p || env->GetDirectBufferCapacity(host) < nRows * d * 4) { raise_arg(env, "a direct ByteBuffer of >= 4*nRows*d bytes is required"); return; }
  raise(env, H(h), se_upload_rowmajor(H(h), slot, p, nRows, d, rowOffset));
}
SE_JNI(void, downloadDirect)(JNIEnv* env, jclass, jlong h, jint slot, jobject host, jlong count, jlong offset) {
  float* p = static_cast<float*>(env->GetDirectBufferAddress(host));
  if (!p || env->GetDirectBufferCapacity(host) < count * 4) { raise_arg(env, "a direct ByteBuffer of >= 4*count bytes is required"); return; }
  raise(env, H(h), se_download(H(h), slot, p, count, offset));
}
'''

CPP_HEAD = r'''// se_jni.cpp — GENERATED by jni/gen_jni.py (edit the table there, not this file).
// Thin JNI shim over the C ABI of include/se_abi.h for scala/org/apache/spark/ml/se/SeNative.scala: one JNI function
// per bound ABI entry point; non-zero status becomes IllegalArgumentException (SE_ERR_ARG) or RuntimeException.
// No GetPrimitiveArrayCritical anywhere: small arrays are copied with Get/Set<Type>ArrayRegion before / after the ABI
// call, bulk transfers go through a native staging chunk or a direct (page-locked) ByteBuffer — the GC is never locked
// out while a DMA, a kernel, a collective or a cudaMalloc runs.
//
// Not compiled in this image (no JDK, hence no <jni.h>); syntax-checked against a stub jni.h by tests/test_host_cpu.py.
//   g++ -O2 -fPIC -shared -I$JAVA_HOME/include -I$JAVA_HOME/include/linux -Iinclude jni/se_jni.cpp \
//       -Lspark_ensemble_b200/lib -lse_b200 -o libse_jni.so
#if defined(SE_JNI_STUB)
#include "jni_stub.h"
#define SE_HAVE_JNI 1
#elif defined(__has_include)
#if __has_include(<jni.h>)
#include <jni.h>
#define SE_HAVE_JNI 1
#endif
#endif

#ifdef SE_HAVE_JNI
#include <stdint.h>

#include <string>
#include <vector>

#include "../include/se_abi.h"

namespace {

inline se_ctx* H(jlong h) { return reinterpret_cast<se_ctx*>(h); }

bool raise(JNIEnv* env, se_ctx* ctx, int rc) {
  if (rc == SE_OK) return false;
  const char* cls = (rc == SE_ERR_ARG) ? "java/lang/IllegalArgumentException" : "java/lang/RuntimeException";
  env->ThrowNew(env->FindClass(cls), se_last_error(ctx));
  return true;
}
void raise_arg(JNIEnv* env, const char* msg) { env->ThrowNew(env->FindClass("java/lang/IllegalArgumentException"), msg); }

// small JVM arrays copied into native buffers (nullable)
struct DoubleIn {
  std::vector<double> v; bool has;
  DoubleIn(JNIEnv* e, jdoubleArray a) : has(a != nullptr) { if (has) { v.resize((size_t)e->GetArrayLength(a)); if (!v.empty()) e->GetDoubleArrayRegion(a, 0, (jsize)v.size(), v.data()); } }
  const double* p() const { return has ? v.data() : nullptr; }
  double* pm() { return has ? v.data() : nullptr; }
};
struct FloatIn {
  std::vector<float> v; bool has;
  FloatIn(JNIEnv* e, jfloatArray a) : has(a != nullptr) { if (has) { v.resize((size_t)e->GetArrayLength(a)); if (!v.empty()) e->GetFloatArrayRegion(a, 0, (jsize)v.size(), v.data()); } }
  const float* p() const { return has ? v.data() : nullptr; }
};
struct IntIn {
  std::vector<int32_t> v; bool has;
  IntIn(JNIEnv* e, jintArray a) : has(a != nullptr) { if (has) { v.resize((size_t)e->GetArrayLength(a)); if (!v.empty()) e->GetIntArrayRegion(a, 0, (jsize)v.size(), reinterpret_cast<jint*>(v.data())); } }
  const int32_t* p() const { return has ? v.data() : nullptr; }
};
// caller-provided output array: native buffer of the same length, copied back after the call
struct DoubleOut {
  JNIEnv* e; jdoubleArray a; std::vector<double> v;
  DoubleOut(JNIEnv* env, jdoubleArray arr, bool read_first) : e(env), a(arr) {
    if (a) { v.resize((size_t)e->GetArrayLength(a)); if (read_first && !v.empty()) e->GetDoubleArrayRegion(a, 0, (jsize)v.size(), v.data()); }
  }
  double* p() { return a ? v.data() : nullptr; }
  void commit() { if (a && !v.empty()) e->SetDoubleArrayRegion(a, 0, (jsize)v.size(), v.data()); }
};
struct Utf {
  JNIEnv* e; jstring s; const char* c;
  Utf(JNIEnv* env, jstring str) : e(env), s(str), c(str ? env->GetStringUTFChars(str, nullptr) : nullptr) {}
  ~Utf() { if (c) e->ReleaseStringUTFChars(s, c); }
};

}  // namespace

#define SE_JNI(ret, name) extern "C" JNIEXPORT ret JNICALL Java_org_apache_spark_ml_se_SeNative_##name
'''


def gen_cpp_fn(name, abi, params, doc):
    jargs, pre, call, outs, commits = ["JNIEnv* env", "jclass"], [], [], [], []
    ctx_expr = "nullptr"
    for pname, kind in params:
        if kind == "ctx":
            jargs.append("jlong h"); call.append("H(h)"); ctx_expr = "H(h)"
        elif kind in SCALARS:
            jt = SCALARS[kind][0]
            jargs.append(f"{jt} {pname}")
            if kind == "bool":
                call.append(f"{pname} ? 1 : 0")
            elif kind == "str":
                pre.append(f"Utf {pname}_u(env, {pname});"); call.append(f"{pname}_u.c")
            elif kind == "u64":
                call.append(f"(uint64_t){pname}")
            else:
                call.append(pname)
        elif kind in ("in_f64", "in_f32", "in_i32"):
            jt = ARRAYS[kind][0]
            cls = {"in_f64": "DoubleIn", "in_f32": "FloatIn", "in_i32": "IntIn"}[kind]
            jargs.append(f"{jt} {pname}"); pre.append(f"{cls} {pname}_in(env, {pname});"); call.append(f"{pname}_in.p()")
        elif kind in ("out_f64", "io_f64"):
            jargs.append(f"jdoubleArray {pname}")
            pre.append(f"DoubleOut {pname}_out(env, {pname}, {'true' if kind == 'io_f64' else 'false'});")
            call.append(f"{pname}_out.p()"); commits.append(f"{pname}_out.commit();")
        elif kind in OUTS:
            ct = OUTS[kind]
            pre.append(f"{ct} {pname}_o = 0;"); call.append(f"&{pname}_o"); outs.append((pname, kind))
        else:
            raise ValueError(kind)
    if abi == "se_abi_version":
        return "SE_JNI(jint, abiVersion)(JNIEnv*, jclass) { return se_abi_version(); }\n"
    if len(outs) == 0:
        ret = "void"
    elif len(outs) == 1:
        ret = {"o_f64": "jdouble", "o_i32": "jint", "o_i64": "jlong"}[outs[0][1]]
    else:
        ret = "jdoubleArray"
    body = [f"SE_JNI({ret}, {name})({', '.join(jargs)}) {{"]
    body += [f"  {l}" for l in pre]
    body.append(f"  const int rc = {abi}({', '.join(call)});")
    body += [f"  {l}" for l in commits]
    zero = {"void": "", "jdouble": " 0.0", "jint": " 0", "jlong": " 0", "jdoubleArray": " nullptr"}[ret]
    body.append(f"  if (raise(env, {ctx_expr}, rc)) return{zero};")
    if len(outs) == 1:
        body.append(f"  return {outs[0][0]}_o;")
    elif len(outs) > 1:
        vals = ", ".join(f"(double){o}_o" for o, _ in outs)
        body.append(f"  const double vals[{len(outs)}] = {{{vals}}};")
        body.append(f"  jdoubleArray r = env->NewDoubleArray({len(outs)});")
        body.append(f"  env->SetDoubleArrayRegion(r, 0, {len(outs)}, vals);")
        body.append("  return r;")
    body.append("}")
    return "\n".join(body) + "\n"


def scala_sig(name, abi, params, doc):
    args, outs = [], []
    for pname, kind in params:
        if kind == "ctx":
            args.append("ctx: Long")
        elif kind in SCALARS:
            args.append(f"{pname}: {SCALARS[kind][1]}")
        elif kind in ARRAYS:
            args.append(f"{pname}: {ARRAYS[kind][1]}")
        else:
            outs.append(kind)
    if abi == "se_abi_version":
        ret = "Int"
    elif not outs:
        ret = "Unit"
    elif len(outs) == 1:
        ret = {"o_f64": "Double", "o_i32": "Int", "o_i64": "Long"}[outs[0]]
    else:
        ret = "Array[Double]"
    line = f"  @native def {name}({', '.join(args)}): {ret}"
    if doc:
        line += f" // {doc}"
    return line


def generate():
    cpp = [CPP_HEAD, HAND_CPP]
    for row in TABLE:
        cpp.append(gen_cpp_fn(*row))
    cpp.append("#endif  // SE_HAVE_JNI\n")
    scala = ['''/*
 * SeNative.scala — GENERATED by jni/gen_jni.py (edit the table there, not this file).
 * JVM side of the drop-in boundary: @native bindings of jni/se_jni.cpp, which forwards 1:1 to the C ABI of
 * include/se_abi.h (libse_b200.so, sm_100a kernels).  Not compiled in this repository's image (no JDK/scalac/sbt);
 * INTEGRATION.md shows how the reference's train()/predict() bodies call these in place of their per-row RDD closures
 * and scala/org/apache/spark/ml/regression/GBMRegressorNative.scala is the rewired GBMRegressor.train().
 */
package org.apache.spark.ml.se

object SeNative {
  System.loadLibrary("se_jni") // links libse_b200.so

  // enum se_slot / se_loss / se_agg_kind / update flags (include/se_abi.h)
  object Slot { val Y = 0; val W = 1; val F = 2; val H = 3; val R = 4; val WOUT = 5; val VY = 6; val VF = 7
    val VH = 8; val BW = 9; val PROBA = 10; val PRED = 11; val P = 12; val RAW = 13; val PROB = 14
    val LABEL = 15; val X = 16; val VX = 17; val BAG = 18 }
  object Loss { val Squared = 0; val Absolute = 1; val Huber = 2; val Quantile = 3; val LogCosh = 4
    val ScaledLogCosh = 5; val Bernoulli = 6; val Exponential = 7; val LogLoss = 8 }
  object Upd { val Residual = 1; val Newton = 2; val Loss = 4 }
  object Agg { val GbmRegressor = 0; val BaggingRegressor = 1; val GbmClassifier = 2; val BaggingSoft = 3; val BaggingHard = 4
    val BoostingReal = 5; val BoostingDiscrete = 6; val BoostingRegMedian = 7; val BoostingRegMean = 8 }

  // ---- handles, communicator bootstrap, bulk transfers (hand-written in the shim)''']
    for _, sig, _ in HAND:
        scala.append(f"  @native {sig}")
    scala.append("\n  // ---- one native per ABI entry point (generated)")
    for row in TABLE:
        scala.append(scala_sig(*row))
    scala.append("}\n")
    return "\n".join(cpp), "\n".join(scala)


def bound_abi():
    s = {abi for _, abi, _, _ in TABLE}
    for _, _, abis in HAND:
        s.update(abis)
    return s


def native_names():
    return [n for n, _, _ in HAND] + [n for n, _, _, _ in TABLE]


if __name__ == "__main__":
    cpp, scala = generate()
    open(os.path.join(ROOT, "jni", "se_jni.cpp"), "w").write(cpp)
    p = os.path.join(ROOT, "scala", "org", "apache", "spark", "ml", "se", "SeNative.scala")
    open(p, "w").write(scala)
    print(f"wrote jni/se_jni.cpp ({len(native_names())} natives) and {os.path.relpath(p, ROOT)}")
