// The C ABI of trace validation (include/csg.h, csg_validate_*): argument checks and the context's traces; the work is validate.cu's.
#include "../prover_ctx.cuh"
#include "validate.cuh"

namespace {

// Every check before anything is enqueued; `airs` receives the AirDesc of each trace.  K traces of length n and `repr`.
void check_validate(csg_ctx *ctx, int air_id, size_t K, int repr, size_t n, const uint64_t *pubs, size_t npub, csg_trace_report *out,
                    std::vector<AirDesc> &airs) {
    if (ctx->comm && ctx->comm->world > 1) throw std::runtime_error("trace validation does not run on a context attached to a group");
    if (!pubs || !out) throw ArgError("null argument");
    csg_ctx::check_repr(repr);
    airs.resize(K);
    // on the host threads from 32 traces on (the Schnorr AIR builds trace-length periodic columns per trace); the first error wins
    std::string err;
    bool failed = false, arg = false;
#pragma omp parallel for schedule(dynamic, 4) if (K >= 32)
    for (long k = 0; k < (long)K; k++) {
        try { airs[k] = make_air(air_id, n, pubs + k * npub, npub); }
        catch (const std::exception &e) {
            const bool is_arg = dynamic_cast<const std::invalid_argument *>(&e) != nullptr;
#pragma omp critical
            { if (!failed) { failed = true; arg = is_arg; err = e.what(); } }
        }
    }
    if (failed) { if (arg) throw ArgError(err); throw std::runtime_error(err); }
}

void run_validate(csg_ctx *ctx, int air_id, const std::vector<AirDesc> &airs, const uint64_t *host, const uint64_t *dev, int repr, size_t n,
                  csg_trace_report *out) {
    const AirDesc &air = airs[0];
    size_t ncells = 0;
    for (const Assertion &s : air.assertions) ncells += s.stride ? n / s.stride : 1;
    const size_t need = validate_footprint(air_id, airs.size(), air.width, n, periodic_runs(air).total, ncells);
    size_t free_b = 0, total_b = 0;
    CSG_CUDA(cudaMemGetInfo(&free_b, &total_b));
    const size_t held = validator_held(ctx->validator);
    if (need > free_b + held) {
        char msg[200];
        snprintf(msg, sizeof msg, "the validation needs %.2f GB of device memory, %.2f GB are available", need / 1e9, (free_b + held) / 1e9);
        throw ArgError(msg);
    }
    if (!ctx->validator) ctx->validator = validator_new();
    validate_traces(ctx->validator, ctx->st, air_id, airs, host, dev, repr, n, out);
}

}  // namespace

extern "C" {

int csg_validate_trace(csg_ctx *ctx, int air_id, const uint64_t *trace, int repr, size_t trace_len, const uint64_t *pub, size_t npub,
                       csg_trace_report *out) {
    return guarded(ctx, [&] {
        if (!trace) throw ArgError("null trace");
        if (trace_len > ((size_t)1 << 22)) throw ArgError("trace length above 2^22 is not supported");
        std::vector<AirDesc> airs;
        check_validate(ctx, air_id, 1, repr, trace_len, pub, npub, out, airs);
        run_validate(ctx, air_id, airs, trace, nullptr, repr, trace_len, out);
    });
}

int csg_validate_resident_trace(csg_ctx *ctx, csg_trace_report *out) {
    return guarded(ctx, [&] {
        if (ctx->comm && ctx->comm->world > 1) throw std::runtime_error("trace validation does not run on a context attached to a group");
        if (!out) throw ArgError("null argument");
        ctx->need(S_TRACE, "no resident trace: csg_load_trace or a device witness builder must run first");
        run_validate(ctx, ctx->air.id, std::vector<AirDesc>{ctx->air}, nullptr, ctx->d_io.p, ctx->trace_repr, ctx->n, out);
    });
}

int csg_validate_many_device(csg_ctx *ctx, int air_id, size_t count, const uint64_t *traces_dev, int repr, size_t trace_len,
                             const uint64_t *pubs, size_t npub, csg_trace_report *out) {
    return guarded(ctx, [&] {
        if (ctx->comm && ctx->comm->world > 1) throw std::runtime_error("trace validation does not run on a context attached to a group");
        if (!traces_dev) throw ArgError("null argument");
        if (count == 0 || count > MANY_MAX_COUNT) throw ArgError("count must be in 1..1024");
        if (trace_len > ((size_t)1 << MANY_MAX_LOG_TRACE)) throw std::runtime_error("csg_validate_many_device takes traces of at most 2^16 rows: validate longer ones with csg_validate_trace");
        try { check_device_buffer(traces_dev, "the traces"); } catch (const ManyArgError &e) { throw ArgError(e.what()); }
        std::vector<AirDesc> airs;
        check_validate(ctx, air_id, count, repr, trace_len, pubs, npub, out, airs);
        if (count * airs[0].width > MANY_MAX_COLUMNS) throw ArgError("count * trace width must not exceed 65535");
        run_validate(ctx, air_id, airs, nullptr, traces_dev, repr, trace_len, out);
    });
}

}  // extern "C"
