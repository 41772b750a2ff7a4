// TEST AID ONLY: compiles the device-side machines (json_machine.cuh / stream_machine.cuh, rollup.cuh) for
// the host so the CPU test-suite can fuzz them against CPython and the oracle without a GPU.
// Never linked into the product library; the product has no CPU path.
#include <stddef.h>
#include <string.h>
#include <vector>
#include "../../include/llmgw_b200.h"
#include "../../llmapigateway_b200/csrc/stream_machine.cuh"

using namespace lgw;

static_assert(sizeof(Val) == sizeof(lgw_val), "Val");
static_assert(sizeof(UsageRec) == sizeof(lgw_usage_rec), "UsageRec");
static_assert(sizeof(StreamState) == sizeof(lgw_stream_state), "StreamState");
static_assert(sizeof(RowEvent) == sizeof(lgw_row_event), "RowEvent");
static_assert(sizeof(SegResult) == sizeof(lgw_seg_result), "SegResult");

extern "C" {

// parse one event text exactly as the stream machine would (cls: 1 = "data: {" part, 2 = "{" part;
// `text` is the whole part).  Returns TopKey|PartFlag bits, fills the normalised record.
uint32_t lgwt_parse_part(const uint8_t* text, uint32_t n, lgw_usage_rec* rec_out, int* cls_out) {
    Rope r{nullptr, 0, text, n};
    const uint8_t cls = classify_part(r, 0, n);
    *cls_out = cls;
    if (cls == PC_NONE) return 0;
    UsageRaw raw;
    const uint32_t f = parse_part<true>(r, 0, n, cls, &raw);
    const uint32_t f2 = parse_part<false>(r, 0, n, cls, nullptr);
    if (f != f2) return 0xFFFFFFFFu;       // the flags-only machine must agree with the extracting one
    UsageRec rec;
    normalise_usage(raw, f, rec);
    memcpy(rec_out, &rec, sizeof(rec));
    return f;
}

// the bulk kernel's lean recogniser on the same text (flags subset)
uint32_t lgwt_lean_parse(const uint8_t* text, uint32_t n) {
    Rope r{nullptr, 0, text, n};
    const uint8_t cls = classify_part(r, 0, n);
    if (cls == PC_NONE) return 0;
    PlainEnv env{nullptr, 0, text, n, g_lean_tables_host.cls, g_lean_tables_host.trans};
    return lean_parse(env, cls == PC_DATA ? 6u : 0u, n, cls == PC_DATA);
}

int lgwt_utf8_valid(const uint8_t* p, uint32_t n) { return utf8_valid(p, n) ? 1 : 0; }

int lgwt_dec_to_double(uint64_t man, int exp10, uint64_t* bits) { return dec_to_double(man, exp10, *bits) ? 1 : 0; }

// run one stream through `n_steps` steps; step k covers chunks [step_chunk[k], step_chunk[k+1])
int lgwt_run_stream(const uint8_t* data, const uint32_t* chunk_off, const uint32_t* step_chunk, uint32_t n_steps,
                    int http_status, uint32_t carry_cap, uint32_t detail_cap,
                    lgw_seg_result* seg_out, lgw_stream_state* final_state,
                    uint8_t* detail_out, lgw_row_event* rows_out, uint32_t rows_cap, uint32_t* n_rows) {
    StreamState st;
    init_stream(st, http_status);
    std::vector<uint8_t> ca(carry_cap + 1), cb(carry_cap + 1), det(detail_cap + 1), pend(LGW_PENDING_STRIDE);
    std::vector<RowEvent> rq(rows_cap + 1);
    uint32_t rcount = 0;
    StepIO io{&st.h, &st.rec, pend.data(), ca.data(), cb.data(), det.data(), carry_cap, detail_cap, rq.data(), &rcount, rows_cap, 0};
    for (uint32_t k = 0; k < n_steps; ++k) {
        SegResult res;
        run_segment(io, data, chunk_off, step_chunk[k], step_chunk[k + 1], res);
        memcpy(&seg_out[k], &res, sizeof(res));
    }
    memcpy(final_state, &st, sizeof(st));
    memcpy(detail_out, det.data(), st.h.detail_len);
    *n_rows = rcount < rows_cap ? rcount : rows_cap;
    memcpy(rows_out, rq.data(), sizeof(RowEvent) * (*n_rows));
    return 0;
}

}  // extern "C"

// ---- request-body rewrite (body_machine.cuh) ----------------------------------------------------
#include "../../llmapigateway_b200/csrc/body_machine.cuh"
static_assert(sizeof(BodyOp) == sizeof(lgw_body_op), "BodyOp");
static_assert(sizeof(BodyScan) == sizeof(lgw_body_scan), "BodyScan");

extern "C" {

static uint32_t g_last_root_kind = 0;
uint32_t lgwt_last_root_kind(void) { return g_last_root_kind; }

uint32_t lgwt_rewrite_body(const uint8_t* in, uint32_t n, int mode, const lgw_body_op* ops, uint32_t n_ops,
                           const uint8_t* blob, uint8_t* out, uint32_t cap, uint32_t* out_len, uint32_t* matched_out) {
    BodyRewriter m;
    const uint32_t st = rewrite_body(m, in, n, mode, (const BodyOp*)ops, n_ops, blob, out, cap, out_len);
    if (matched_out) *matched_out = m.matched;
    g_last_root_kind = m.root_kind;
    return st;
}

void lgwt_scan_body(const uint8_t* in, uint32_t n, lgw_body_scan* sc, uint8_t* model_buf, uint32_t model_cap) {
    BodyRewriter m;
    scan_body(m, in, n, (BodyScan*)sc, model_buf, model_cap);
}

}  // extern "C"

// ---- data-parallel body rewrite (body_fast.cuh), phases emulated thread by thread ---------------------
#include "../../llmapigateway_b200/csrc/body_fast.cuh"
extern "C" uint32_t lgwt_rewrite_body_fast(const uint8_t* in, uint32_t n, int mode, const lgw_body_op* ops, uint32_t n_ops,
                                           const uint8_t* blob, uint8_t* out, uint32_t cap, uint32_t* out_len, uint32_t* matched_out) {
    static FastShared sh;
    uint32_t matched = 0;
    const uint32_t st = fast_rewrite(&sh, in, n, mode, (const BodyOp*)ops, n_ops, blob, out, cap, out_len, &matched);
    if (matched_out) *matched_out = matched;
    g_last_root_kind = KD_OBJ;
    return st;
}

// ---- error detail of failing non-streaming responses (error_detail.cuh) -----------------------------------
#include "../../llmapigateway_b200/csrc/error_detail.cuh"
static_assert(sizeof(lgw::DocError) == sizeof(lgw_doc_error), "DocError");
extern "C" void lgwt_error_detail(const uint8_t* doc, uint32_t n, lgw_doc_error* out, uint8_t* text, uint32_t cap) {
    lgw::error_detail_of(doc, n, *(lgw::DocError*)out, text, cap);
}

// ---- response tap of a non-streaming response: what lane 0 of k_docs_usage does for one document (doc_kernels.cuh:32-50; the
//      kernel itself holds __global__ code and is not included here -- the same machine calls in the same order) ---------------
extern "C" void lgwt_doc_usage(const uint8_t* doc, uint32_t len, lgw_doc_usage* out) {
    out->flags = 0; out->rec_valid = 0; out->error_row = 0; out->exotic = 0; out->_pad = 0;
    UsageRec& rec = *(UsageRec*)&out->rec;
    default_usage(rec);
    Rope r{nullptr, 0, doc, len};
    const uint8_t cls = classify_part(r, 0, len);                       // chat_logging.py:116-121
    if (cls == PC_NONE) return;
    UsageRaw raw;
    const uint32_t f = parse_part<true>(r, 0, len, cls, &raw);          // :123
    out->flags = f;
    if ((f & PF_VALID_B) && (f & (TK_USAGE | TK_ERROR))) {
        if (f & PF_EXOTIC) out->exotic = 1;
        else if (!((f & TK_CHOICES) && (f & PF_TYPE_ERROR))) {
            if (f & TK_USAGE) { normalise_usage(raw, f, rec); out->rec_valid = 1; if (rec.exotic) out->exotic = 1; }   // :134-135
            if (f & TK_ERROR) out->error_row = 1;                        // :137-139
        }
    }
}

// ---- exact cost accumulation of the usage rollup (rollup.cuh): the same integer code the kernels run ---------------------
#include "../../llmapigateway_b200/csrc/rollup.cuh"
extern "C" int lgwt_cost_to_limbs(double c, uint32_t limb[4]) { return lgw::cost_to_limbs(c, limb) ? 1 : 0; }
extern "C" double lgwt_limbs_to_cost(const uint64_t cell[4]) { return lgw::limbs_to_cost(cell); }
// the limbs of n records added into four 64-bit cells (wrap-around) as the rollup kernels add them; 0 when any record was not exact
extern "C" int lgwt_sum_costs(const double* c, uint64_t n, uint64_t cell[4]) {
    int exact = 1;
    cell[0] = cell[1] = cell[2] = cell[3] = 0;
    for (uint64_t i = 0; i < n; ++i) {
        uint32_t limb[4];
        exact &= lgw::cost_to_limbs(c[i], limb) ? 1 : 0;
        for (int k = 0; k < 4; ++k) cell[k] += limb[k];
    }
    return exact;
}
