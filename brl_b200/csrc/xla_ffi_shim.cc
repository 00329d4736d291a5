// xla_ffi_shim.cc -- adapters that expose the C-ABI ops (include/brl_b200.h) to a jitted
// JAX program, so that brl's `ppo.py` / `eval.py` loops can call the CUDA env as a drop-in
// for `pgx.bridge_bidding` (src/roll_out.py:51, src/duplicate.py:134,149, src/gae.py:32-38).
//
// ONE table (BRL_XLA_OPS) drives both XLA conventions.  Per op it holds a layout string with one character per
// buffer of the op, in the op's documented order:
//     i  input            -> an XLA operand
//     o  output           -> an XLA result
//     s  scratch          -> an XLA result nobody reads
//     x  updated in place -> an XLA operand AND the result aliased to it (input_output_aliases /
//                            operand_output_aliases); the adapter checks the two pointers are equal
// XLA hands a custom call its operands first, then its results, each in declaration order; the adapter re-orders them
// into the op's buffer list.  An op's optional (NULL-able) buffers are all present in its XLA form.
//   (1) legacy GPU custom call, API_VERSION_STATUS_RETURNING (what jax 0.4.23 -- the version brl pins,
//       requirements.txt:25-26 -- offers):
//         void <op>_xla(cudaStream_t, void** buffers, const char* opaque, size_t len, XlaCustomCallStatus*)
//       opaque = the bytes of one BrlParams (BrlPpoParams / BrlAdamParams for the update ops).  Always built; exercised by
//       tests/test_cuda_xla.py through ctypes with exactly this signature.
//   (2) typed FFI (jax >= 0.4.31): <op>_ffi = one generic handler over RemainingArgs / RemainingRets + a byte-span
//       attribute "opaque", instantiated per op by the same table.  Compiled only when `xla/ffi/api/ffi.h` is on the
//       include path (build.py probes jaxlib); this image has no jaxlib, so (2) has never been compiled here --
//       INTEGRATION.md says so.
// A failing op reports through XlaCustomCallStatusSetFailure, which XLA's runtime exports: the symbol is looked up with
// dlsym(RTLD_DEFAULT) at call time (this library is not linked against XLA).  If the process has no such symbol the
// failure cannot reach XLA; it is then counted (brl_xla_unreported_failures) and stays readable in brl_last_error().
#if defined(__has_include)
#if __has_include("xla/ffi/api/ffi.h")
#define BRL_HAVE_XLA_FFI 1
#endif
#endif

#include <dlfcn.h>

#include <atomic>
#include <cstdio>
#include <cstring>

#include "../../include/brl_b200.h"

#define BRL_XLA_OPS(X) \
    X(brl_make_keys, "o") \
    X(brl_init, "iioooooo") \
    X(brl_reset_fields, "iiiiiiioooooo") \
    X(brl_step, "iiiooooooo") \
    X(brl_duplicate_step, "iiixxxxxxxxxxxxoooooo") \
    X(brl_duplicate_init, "iioooooo") \
    X(brl_observe, "iiio") \
    X(brl_legal_mask, "io") \
    X(brl_rollout_random, "xiooooooxio") \
    X(brl_imp_reward, "iio") \
    X(brl_gae, "iiiioo") \
    X(brl_categorical, "iioo") \
    X(brl_match_stats, "ix") \
    X(brl_state_fields, "iooooooooooo") \
    X(brl_gather_reward, "iioix") \
    X(brl_team_rows, "iiooo") \
    X(brl_mlp_pack, "iiiiiiiiiiiio") \
    X(brl_obs_to_bf16, "io") \
    X(brl_mlp_forward, "iisoo") \
    X(brl_policy_act, "iisiooooi") \
    X(brl_policy_act_rows, "iisixixx") \
    X(brl_ppo_loss, "iiiiiiiiiooos") \
    X(brl_adam_clip, "xixxs") \
    X(brl_adam_apply, "xixxi") \
    X(brl_gather_rows, "iio") \
    X(brl_eval_act_log, "iiiiiox") \
    X(brl_eval_summary, "iiiiiiiiiiiiiiix") \
    X(brl_mlp_pack_train, "io") \
    X(brl_mlp_adam_step, "xixxix") \
    X(brl_ppo_grad, "iisiiiiiiioos") \
    X(brl_sl_examples, "iiiiiooooo") \
    X(brl_sl_grad, "iisiioos") \
    X(brl_sl_eval, "iisiios") \
    X(brl_model_rows, "iiioooo") \
    X(brl_policy_act_grouped, "iisixiixi") \
    X(brl_match_stats_ranges, "iix") \
    X(brl_duplicate_match, "iiiiisoxooooooooooooo") \
    X(brl_evaluate_match, "iiisooxooooooooooooooooooo") \
    X(brl_ppo_grad_grouped, "iiisoos") \
    X(brl_mlp_adam_step_grouped, "xixxix") \
    X(brl_ppo_grad_anchored, "iisiiiiiiioosii") \
    X(brl_ppo_grad_grouped_anchored, "iiisoosii") \
    X(brl_par, "iioo") \
    X(brl_gather_reward_par, "iiiiox") \
    X(brl_par_stats, "iiiiiiiix") \
    X(brl_system_stats, "iiiiix") \
    X(brl_system_stats_auctions, "iiiiix") \
    X(brl_call_values, "iiiiiisoooooooooooo") \
    X(brl_cv_grad, "iisioos") \
    X(brl_cv_eval, "iisios") \
    X(brl_hand_posterior, "iiiiiiiiisoooo") \
    X(brl_hand_posterior_smc, "iiiiiiiiisooooooo") \
    /* end */

namespace {
constexpr int kMaxBuffers = 32;

typedef void (*status_fn_t)(XlaCustomCallStatus_*, const char*, size_t);
std::atomic<status_fn_t> g_status_fn{nullptr};
std::atomic<long long> g_unreported{0};

void report_failure(XlaCustomCallStatus_* status, const char* msg) {
    status_fn_t fn = g_status_fn.load(std::memory_order_acquire);
    if (fn == nullptr) {
        fn = reinterpret_cast<status_fn_t>(dlsym(RTLD_DEFAULT, "XlaCustomCallStatusSetFailure"));
        if (fn != nullptr) g_status_fn.store(fn, std::memory_order_release);
    }
    if (fn != nullptr && status != nullptr) fn(status, msg, std::strlen(msg));
    else g_unreported.fetch_add(1, std::memory_order_relaxed);
}

// XLA order (operands, then results) -> the op's buffer order.  Returns NULL on success, else a message.
const char* reorder(const char* layout, void* const* xla, void** out, char* msg, size_t msg_len) {
    int n_in = 0;
    for (const char* c = layout; *c; ++c) n_in += (*c == 'i' || *c == 'x');
    int in = 0, res = n_in, k = 0;
    for (const char* c = layout; *c; ++c, ++k) {
        if (k >= kMaxBuffers) return "layout too long";
        if (*c == 'i') out[k] = xla[in++];
        else if (*c == 'o' || *c == 's') out[k] = xla[res++];
        else {  // 'x'
            out[k] = xla[in++];
            if (xla[res++] != out[k]) {
                std::snprintf(msg, msg_len, "buffer %d is updated in place: alias the result to the operand (input_output_aliases)", k);
                return msg;
            }
        }
    }
    for (; k < kMaxBuffers; ++k) out[k] = nullptr;
    return nullptr;
}

void legacy_call(brl_op_fn op, const char* name, const char* layout, brl_stream_t stream, void** buffers, const char* opaque,
                 size_t opaque_len, XlaCustomCallStatus_* status) {
    void* b[kMaxBuffers];
    char msg[160];
    if (const char* err = reorder(layout, buffers, b, msg, sizeof(msg))) {
        char full[224];
        std::snprintf(full, sizeof(full), "%s_xla: %s", name, err);
        report_failure(status, full);
        return;
    }
    if (op(stream, b, opaque, opaque_len) != BRL_OK) report_failure(status, brl_last_error());
}
}  // namespace

extern "C" {

#define BRL_LEGACY_CUSTOM_CALL(op, layout)                                                                        \
    void op##_xla(brl_stream_t stream, void** buffers, const char* opaque, size_t opaque_len,                     \
                  struct XlaCustomCallStatus_* status) {                                                          \
        legacy_call(op, #op, layout, stream, buffers, opaque, opaque_len, status); \
    }
BRL_XLA_OPS(BRL_LEGACY_CUSTOM_CALL)

// layout string of an op ("brl_step" -> "iiiooooooo"), NULL for an unknown name: the registration code on the JAX side
// derives operand / result order and the aliases from it (INTEGRATION.md)
const char* brl_xla_layout(const char* op_name) {
#define BRL_LAYOUT_CASE(op, layout) \
    if (std::strcmp(op_name, #op) == 0) return layout;
    BRL_XLA_OPS(BRL_LAYOUT_CASE)
    return nullptr;
}

long long brl_xla_unreported_failures(void) { return g_unreported.load(std::memory_order_relaxed); }

}  // extern "C"

// ---- (2) typed FFI handlers --------------------------------------------------------------
#ifdef BRL_HAVE_XLA_FFI
#include <string>

#include "xla/ffi/api/ffi.h"
namespace ffi = xla::ffi;
// brl_stream_t is `struct CUstream_st*`, i.e. cudaStream_t: PlatformStream<brl_stream_t> needs no CUDA header here

namespace {
ffi::Error typed_call(brl_op_fn op, const char* name, const char* layout, brl_stream_t stream, ffi::RemainingArgs args,
                      ffi::RemainingRets rets, ffi::Span<const uint8_t> opaque) {
    void* xla[kMaxBuffers];
    size_t n = 0;
    for (size_t i = 0; i < args.size() && n < kMaxBuffers; ++i) xla[n++] = args.get<ffi::AnyBuffer>(i).value().untyped_data();
    for (size_t i = 0; i < rets.size() && n < kMaxBuffers; ++i) xla[n++] = rets.get<ffi::AnyBuffer>(i).value()->untyped_data();
    if (n != std::strlen(layout) + (size_t)[&] { int x = 0; for (const char* c = layout; *c; ++c) x += *c == 'x'; return x; }())
        return ffi::Error(ffi::ErrorCode::kInvalidArgument, std::string(name) + "_ffi: wrong number of operands + results");
    void* b[kMaxBuffers];
    char msg[160];
    if (const char* err = reorder(layout, xla, b, msg, sizeof(msg)))
        return ffi::Error(ffi::ErrorCode::kInvalidArgument, std::string(name) + "_ffi: " + err);
    if (op(stream, b, opaque.begin(), opaque.size()) != BRL_OK)
        return ffi::Error(ffi::ErrorCode::kInvalidArgument, brl_last_error());
    return ffi::Error::Success();
}
}  // namespace

#define BRL_TYPED_FFI(op, layout)                                                                                         \
    static ffi::Error op##_ffi_impl(brl_stream_t stream, ffi::RemainingArgs args, ffi::RemainingRets rets,                \
                                    ffi::Span<const uint8_t> opaque) {                                                    \
        return typed_call(op, #op, layout, stream, args, rets, opaque);                                                   \
    }                                                                                                                     \
    XLA_FFI_DEFINE_HANDLER_SYMBOL(op##_ffi, op##_ffi_impl,                                                                \
                                  ffi::Ffi::Bind().Ctx<ffi::PlatformStream<brl_stream_t>>().RemainingArgs().RemainingRets() \
                                      .Attr<ffi::Span<const uint8_t>>("opaque"));
BRL_XLA_OPS(BRL_TYPED_FFI)
#endif  // BRL_HAVE_XLA_FFI
