// engine.cu -- plan loader, per-batch launch programs, CUDA-graph replay and the C ABI (include/adas_b200.h).
//
// Replaces the engine layer of the reference (coreEngine.py): TensorRTBase.__init__/_allocate_buffers (:41-88),
// TensorRTBase.inference (:93-118), TensorRTEngine/OnnxEngine shape queries (:144-148,178-182) and
// engine_inference (:150-157,184-186).  One handle = one device + one private stream; every activation
// tensor of the network owns its own HBM buffer (180 GB: no reuse planning, zero halos stay zero forever).
#include "common.h"
#include "plan.h"
#include "../../include/adas_b200.h"
#include <stdarg.h>
#include <time.h>
#include <stdlib.h>
#include <string.h>
#include <map>
#include <memory>
#include <functional>

namespace adas {

static thread_local char g_err[1024] = "";
std::atomic<long long> g_launches{0};

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int launch_iou_cost(int problems, const double* a, const int32_t* a_off, const double* b, const int32_t* b_off,
                    const double* det_scores, int fuse, double* cost, const int64_t* cost_off, cudaStream_t st);
int launch_lap(int problems, const double* cost, const int64_t* cost_off, const int32_t* T, const int32_t* D,
               const double* thresh, int32_t* x, const int32_t* x_off, int32_t* y, const int32_t* y_off, double* work_v,
               double* work_minv, int32_t* work_i, cudaStream_t st);
int lap_max_cols();

struct DevBuf {
    void* ptr = nullptr;
    size_t bytes = 0;
};

struct Program {   // launch list for one batch size
    std::vector<std::function<int(cudaStream_t)>> steps;
    std::vector<uint32_t> step_type;
    std::vector<std::string> step_desc;   // human-readable shape / tile choice per step (adas_engine_step_desc)
    std::vector<std::vector<std::pair<int, int>>> step_tiles;   // (BN, MT) tiles a tcgen05 GEMM step could run with (adas_engine_step_tiles)
    std::vector<int> step_chosen;                               // index into step_tiles of the tile the step runs
    cudaGraphExec_t graph = nullptr;
    int runs = 0;
    int n_launch() const { int n = 0; for (uint32_t t : step_type) n += (t != 31); return n; }   // steps folded into a chain launch do not launch
};

}  // namespace adas

using namespace adas;

struct adas_engine {
    int device = 0;
    int max_batch = 1;
    int conv_impl = 0;
    bool use_graph = true;
    int use_chain = 0;            // ADAS_B200_CHAIN: 0 (default) = one launch per layer; 2 = chain a run where the chain launch (gemm_chain.cu) timed
                                  // faster than its per-layer launches when the program was built; 1 = chain every eligible run.  Off by default:
                                  // one bench process in ~6 hung on the device with chains enabled (never with ADAS_B200_CHAIN=0, 16 runs) --
                                  // root cause not found, see DESIGN.md section 4.2
    bool autotune = true;         // ADAS_B200_AUTOTUNE=0: modelled tile choice only
    cudaStream_t stream = nullptr;
    PlanHeader hdr;
    std::vector<PlanBuffer> bufs;
    std::vector<PlanOp> ops;
    std::vector<PlanTensor> tensors;
    std::vector<PlanOutput> outs;
    void* d_blob = nullptr;
    std::vector<DevBuf> dbufs;
    std::map<int, Program> programs;
    // staging
    float* d_input = nullptr;        // [max_batch, C, H, W] fp32
    uint8_t* d_frames = nullptr;     // [max_batch * frame_bytes]
    const uint8_t* last_dfr = nullptr; int last_fb = 0, last_fh = 0, last_fw = 0;      // frames of the last detect call, on the device
    uint8_t* d_warp = nullptr; size_t warp_cap = 0; double* d_warpM = nullptr;          // adas_engine_warp_perspective scratch
    size_t frames_cap = 0;
    float* d_raw = nullptr;          // decoded head tensor (YOLO) [max_batch, ...]
    size_t raw_per_img = 0;
    // yolo post scratch
    YoloPostBufs yp{};
    int yp_max_det = 0;
    // ufld
    float* d_lut = nullptr;          // 3*256 fp32
    double* d_row_anchor = nullptr;
    double* d_col_anchor = nullptr;
    int32_t* d_pts = nullptr; int32_t* d_npts = nullptr; uint8_t* d_status = nullptr; double* d_coords = nullptr;
    // lane geometry downstream of the lane decode (lane_geom.cu), allocated on first use
    int32_t* d_area = nullptr; int32_t* d_bird = nullptr; adas_lane_geom* d_geom = nullptr; double* d_M = nullptr; int geom_cap_area = 0; int ufld_last_batch = 0;
    int ufld_max_pts = 0;
    double ufld_crop = 0.6;       // crop ratio of the plan's dataset (ModelConfig.crop_ratio)
    std::vector<int32_t> h_ncand;
    cudaEvent_t ev_frames = nullptr;
    cudaEvent_t events[4] = {nullptr, nullptr, nullptr, nullptr};
};

namespace adas {

static size_t elem_size(uint32_t dtype) { return dtype == 1 ? 4 : 2; }

// ADAS_B200_TRACE=1: per-phase device time (CUDA events on the handle's stream) + host wall time of each detect call
static inline bool is_ufld(uint32_t kind) { return kind == ADAS_MODEL_UFLDV2 || kind == ADAS_MODEL_UFLDV1; }

struct PhaseTrace {
    static bool enabled() { static int v = -1; if (v < 0) { const char* t = getenv("ADAS_B200_TRACE"); v = (t && t[0] == '1') ? 1 : 0; } return v == 1; }
    cudaStream_t st; const char* name; cudaEvent_t ev[10]; const char* names[10]; int n = 0; double t0 = 0;
    static double now() { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6; }
    PhaseTrace(cudaStream_t s, const char* nm) : st(s), name(nm) { if (enabled()) { t0 = now(); mark("start"); } }
    void mark(const char* nm) { if (!enabled() || n >= 10) return; cudaEventCreate(&ev[n]); cudaEventRecord(ev[n], st); names[n] = nm; ++n; }
    void report() {
        if (!enabled()) return;
        cudaEventSynchronize(ev[n - 1]);
        fprintf(stderr, "[trace] %s host %.3f ms |", name, now() - t0);
        for (int i = 1; i < n; ++i) { float ms = 0; cudaEventElapsedTime(&ms, ev[i - 1], ev[i]); fprintf(stderr, " %s %.3f", names[i], ms); }
        fprintf(stderr, "\n");
        for (int i = 0; i < n; ++i) cudaEventDestroy(ev[i]);
    }
};

static const void* tensor_ptr(const adas_engine* e, int idx) {
    if (idx < 0) return nullptr;
    return static_cast<const uint8_t*>(e->d_blob) + e->tensors[idx].offset;
}

// one v3 GEMM step as the chain builder sees it (gemm_chain.cu)
struct GemmRec {
    size_t step;                       // index into Program::steps
    GemmParams g;                      // with the tile shape that was finally chosen
    int a_buf, a_coff, out_buf, out_coff, res_buf, res_coff;
    bool eligible;
    std::function<int(const GemmParams&, void**)> prep;
};

static bool chain_edge_ok(const GemmRec& a, const GemmRec& b) {
    if (!a.eligible || !b.eligible || b.step != a.step + 1) return false;
    const GemmParams &x = a.g, &y = b.g;
    if (x.M != y.M || x.N != y.N || x.Kc != y.Kc || x.ntaps != y.ntaps || x.act != y.act || x.Wp != y.Wp || x.mask_H != y.mask_H || x.mask_W != y.mask_W) return false;
    if (b.a_buf != a.out_buf || b.a_coff != a.out_coff || y.Kc != x.N) return false;        // b reads exactly what a wrote
    if (b.res_buf >= 0 && !(b.res_buf == a.a_buf && b.res_coff == a.a_coff)) return false;     // residual = the previous layer's input
    return true;
}

static int build_chains(adas_engine* e, Program* prog, std::vector<GemmRec>& recs) {
    if (!e->use_chain) return 0;
    size_t i = 0;
    while (i < recs.size()) {
        size_t j = i;
        while (j + 1 < recs.size() && chain_edge_ok(recs[j], recs[j + 1])) {
            // no layer may write a view an earlier layer of the chain still reads
            bool clash = false;
            const GemmRec& w = recs[j + 1];
            for (size_t k = i; k <= j && !clash; ++k) {
                const GemmRec& r = recs[k];
                auto overlap = [&](int buf, int coff, int C) { return buf == w.out_buf && coff < w.out_coff + w.g.N && w.out_coff < coff + C; };
                clash = overlap(r.a_buf, r.a_coff, r.g.Kc) || (r.res_buf >= 0 && overlap(r.res_buf, r.res_coff, r.g.N));
            }
            if (clash) break;
            ++j;
        }
        if (j > i) {
            static const bool chain_log = getenv("ADAS_B200_CHAIN_LOG") != nullptr;
            // tile shapes worth trying for the chain: the ones the member layers chose for themselves
            std::vector<std::pair<int, int>> shapes;
            for (size_t k = i; k <= j; ++k) {
                const std::pair<int, int> sh(recs[k].g.BN, recs[k].g.mt_hint);
                if (std::find(shapes.begin(), shapes.end(), sh) == shapes.end()) shapes.push_back(sh);
            }
            const bool timed = e->use_chain == 2 && e->autotune;
            if (!timed) shapes.resize(1);
            cudaEvent_t ev0 = nullptr, ev1 = nullptr;
            float best_ms = 1e30f;
            if (timed) {
                // the alternative: the per-layer launches as they stand, back to back
                ADAS_CUDA(cudaEventCreate(&ev0)); ADAS_CUDA(cudaEventCreate(&ev1));
                int rc = 0;
                for (int r = 0; r < 5 && !rc; ++r) {
                    if (r == 1) cudaEventRecord(ev0, e->stream);
                    for (size_t k = i; k <= j && !rc; ++k) rc = prog->steps[recs[k].step](e->stream);
                }
                cudaEventRecord(ev1, e->stream);
                if (rc || cudaEventSynchronize(ev1) != cudaSuccess) { cudaEventDestroy(ev0); cudaEventDestroy(ev1); ADAS_CHECK(false, "chain timing: per-layer launches failed (%s)", g_err); }
                cudaEventElapsedTime(&best_ms, ev0, ev1);
                if (chain_log) fprintf(stderr, "[chain] steps %zu..%zu per-layer launches: %.1f us\n", recs[i].step, recs[j].step, best_ms * 250.0);
            }
            void* best_chain = nullptr;
            for (const auto& sh : shapes) {
                std::vector<void*> layers;
                bool ok = true;
                for (size_t k = i; k <= j && ok; ++k) {
                    GemmParams gc = recs[k].g;
                    gc.BN = sh.first; gc.mt_hint = sh.second; gc.chain = 1;
                    void* op = nullptr;
                    if (recs[k].prep(gc, &op)) ok = false; else layers.push_back(op);
                }
                void* chain = nullptr;
                if (ok && gemm_chain_prepare(layers.data(), (int)layers.size(), &chain)) ok = false;
                for (void* op : layers) gemm_v3_free(op);                    // the chain keeps its own copies of the tensor maps
                if (!ok) {
                    if (chain_log) fprintf(stderr, "[chain] steps %zu..%zu BN=%d MT=%d not chainable: %s\n", recs[i].step, recs[j].step, sh.first, sh.second, g_err);
                    continue;
                }
                if (!timed) { best_chain = chain; break; }
                int rc = 0;
                for (int r = 0; r < 5 && !rc; ++r) {
                    if (r == 1) cudaEventRecord(ev0, e->stream);
                    rc = gemm_chain_run(chain, e->stream);
                }
                cudaEventRecord(ev1, e->stream);
                float ms = 1e30f;
                if (!rc && cudaEventSynchronize(ev1) == cudaSuccess) cudaEventElapsedTime(&ms, ev0, ev1);
                if (chain_log) fprintf(stderr, "[chain] steps %zu..%zu one launch BN=%d MT=%d: %.1f us\n", recs[i].step, recs[j].step, sh.first, sh.second, ms * 250.0);
                if (ms < best_ms * 0.98f) { best_ms = ms; if (best_chain) gemm_chain_free(best_chain); best_chain = chain; }
                else gemm_chain_free(chain);
            }
            if (ev0) { cudaEventDestroy(ev0); cudaEventDestroy(ev1); }
            if (best_chain) {
                std::shared_ptr<void> keep(best_chain, gemm_chain_free);
                char d[256];
                gemm_chain_describe(best_chain, d, sizeof(d));
                prog->step_desc.resize(prog->steps.size());
                prog->step_desc[recs[i].step] = d;
                prog->steps[recs[i].step] = [keep](cudaStream_t st) { return gemm_chain_run(keep.get(), st); };
                for (size_t k = i; k <= j; ++k) prog->step_tiles[recs[k].step].clear();      // no longer a per-layer tcgen05 GEMM launch
                for (size_t k = i + 1; k <= j; ++k) {
                    prog->steps[recs[k].step] = [](cudaStream_t) { return 0; };   // folded into the chain launch above
                    prog->step_type[recs[k].step] = 31;
                    prog->step_desc[recs[k].step] = "(in the chain above)";
                }
            }
        }
        i = j + 1;
    }
    return 0;
}

static int build_program(adas_engine* e, int batch, Program* prog) {
    std::vector<GemmRec> recs;
    for (size_t oi = 0; oi < e->ops.size(); ++oi) {
        const PlanOp& op = e->ops[oi];
        const int32_t* p = op.p;
        prog->step_type.push_back(op.type);
        switch (op.type) {
            case OP_GEMM: {
                const int a_buf = p[0], a_coff = p[1], Kc = p[2], ntaps = p[3], w_t = p[4], bias_t = p[5], N = p[6], act = p[7];
                const int res_buf = p[8], res_coff = p[9], res_pre = p[10], out_buf = p[11], out_coff = p[12], masked = p[13];
                const int transposed = p[14];
                int BN = p[15];
                const int s2 = p[16];
                const PlanBuffer& ab = e->bufs[a_buf];
                const PlanBuffer& ob = e->bufs[out_buf];
                ADAS_CHECK(ab.dtype == 0, "op %zu: GEMM input buffer must be fp16", oi);
                ADAS_CHECK(Kc % 8 == 0 && a_coff % 8 == 0 && ab.C % 8 == 0, "op %zu: K alignment", oi);
                ADAS_CHECK(ntaps == 1 || ((ntaps == 9 || ntaps == 4) && Kc % 64 == 0 && ab.W > 0), "op %zu: tap mode needs Cin %% 64 == 0", oi);
                ADAS_CHECK(!s2 || (Kc % 64 == 0 && ab.W > 0 && ob.W > 0 && !transposed), "op %zu: stride-2 mode needs Cin %% 64 == 0 on padded grids", oi);
                GemmParams g;
                memset(&g, 0, sizeof(g));
                const int Ktot = ntaps * Kc;
                const __half* wptr = static_cast<const __half*>(tensor_ptr(e, w_t));
                ADAS_CHECK((size_t)e->tensors[w_t].bytes >= (size_t)(transposed ? N : N) * Ktot * 2, "op %zu: weight tensor too small", oi);
                const __half* aptr = static_cast<const __half*>(e->dbufs[a_buf].ptr) + a_coff;
                const int a_rows = batch * (int)ab.rows_per_img;
                const void *opA, *opB;
                uint64_t a_inner, a_rows_u, a_stride, b_inner, b_rows_u, b_stride;
                if (!transposed) {
                    g.M = a_rows;
                    g.N = N;
                    if (BN <= 0 && !s2) {           // a starting point only: the v3 path ranks / times its own tile candidates below
                        if (N <= 256) BN = (N + 15) / 16 * 16;
                        else if (N % 256 == 0) BN = 256;
                        else if (N % 160 == 0) BN = 160;
                        else if (N % 128 == 0) BN = 128;
                        else BN = 256;
                    }
                    opA = aptr; a_inner = (uint64_t)Kc; a_rows_u = (uint64_t)a_rows; a_stride = (uint64_t)ab.C * 2;
                    opB = wptr; b_inner = (uint64_t)Ktot; b_rows_u = (uint64_t)N; b_stride = (uint64_t)Ktot * 2;
                    g.A = aptr; g.a_ld = (int)ab.C; g.Wt = wptr; g.w_ld = Ktot;
                    g.out_ld = (int)ob.C;
                    ADAS_CHECK(s2 || (int)ob.rows_per_img == (int)ab.rows_per_img, "op %zu: GEMM in/out row geometry differs", oi);
                    if (s2) {
                        // output-pixel patch (bw x bh <= 128) that wastes the fewest rows of the 128-row MMA tile
                        const int Ho = (int)ob.H, Wo = (int)ob.W;
                        int best_bw = 8, best_bh = 16; double best_eff = -1.0;
                        const int cands[] = {Wo, 128, 64, 32, 16, 8};
                        for (int ci = 0; ci < 6; ++ci) {
                            const int bw = cands[ci];
                            if (bw < 1 || bw > 128) continue;
                            const int bh = 128 / bw;
                            if (bh < 1) continue;
                            const int tw = (Wo + bw - 1) / bw, th = (Ho + bh - 1) / bh;
                            const double eff = (double)Wo * Ho / ((double)tw * th * 128.0);
                            if (eff > best_eff + 1e-9) { best_eff = eff; best_bw = bw; best_bh = bh; }
                        }
                        g.s2 = 1; g.s2_bw = best_bw; g.s2_bh = best_bh;
                        g.s2_tw = (Wo + best_bw - 1) / best_bw; g.s2_th = (Ho + best_bh - 1) / best_bh;
                        g.s2_Ho = Ho; g.s2_Wo = Wo; g.s2_Hp_in = (int)ab.H + 2;
                        if (e->conv_impl == 1) g.M = batch * (int)ob.rows_per_img;        // SIMT kernel walks output rows
                        else g.M = batch * g.s2_tw * g.s2_th * 128;                         // tcgen05 kernel walks patches
                        if (p[15] <= 0) BN = N <= 256 ? (N + 15) / 16 * 16 : (N % 256 == 0 ? 256 : 128);
                    }
                } else {
                    // swap-AB: rows = output features (weights stream once through the A operand), cols = batch rows
                    // FC semantics: ONE input vector per image -- the whole per-image slab of the input buffer (a dense [1, K] row, or a
                    // padded feature map read flat: its halo entries are zeros that meet zero weight columns)
                    const uint64_t x_ld = (uint64_t)ab.rows_per_img * ab.C;
                    g.M = N;
                    g.N = batch;
                    BN = (batch + 15) / 16 * 16;
                    ADAS_CHECK(BN <= 256, "op %zu: transposed GEMM supports at most 256 images per batch", oi);
                    ADAS_CHECK((uint64_t)Kc <= x_ld && a_coff == 0 && (x_ld * 2) % 16 == 0, "op %zu: FC input vector exceeds its buffer", oi);
                    opA = wptr; a_inner = (uint64_t)Ktot; a_rows_u = (uint64_t)N; a_stride = (uint64_t)Ktot * 2;
                    opB = aptr; b_inner = (uint64_t)Kc; b_rows_u = (uint64_t)batch; b_stride = x_ld * 2;
                    g.A = wptr; g.a_ld = Ktot; g.Wt = aptr; g.w_ld = (int)x_ld;
                    g.out_ld = (int)(ob.rows_per_img * ob.C);
                }
                if (p[17] > 0) g.mt_hint = p[17];       // plan-forced sub-tile count (test hook of plan.py)
                // Fully connected layers whose weight matrix stays in L2 (FC1 of the UFLD head: 20 MB) run as a weight stream on the CUDA
                // cores: the swap-AB tensor-core GEMM has only N/256 CTAs for them (profiles/r02_optable_ufld_b8: 47.8 us = 0.43 TB/s).
                static const bool fc_stream_on = !(getenv("ADAS_B200_FC_STREAM") && getenv("ADAS_B200_FC_STREAM")[0] == '0');
                if (transposed && e->conv_impl == 0 && fc_stream_on && ntaps == 1 && (size_t)N * Kc * 2 <= ((size_t)48 << 20) && Kc % 8 == 0 && ab.C % 8 == 0) {
                    const float* bias_p = static_cast<const float*>(tensor_ptr(e, bias_t));
                    void* out_p = static_cast<uint8_t*>(e->dbufs[out_buf].ptr) + (size_t)out_coff * elem_size(ob.dtype);
                    const int x_ld = (int)(ab.rows_per_img * ab.C), o_ld = (int)(ob.rows_per_img * ob.C), of32 = ob.dtype == 1 ? 1 : 0;
                    char d[128];
                    snprintf(d, sizeof(d), "M=%d N=%d K=%d fc_stream", batch, N, Kc);
                    prog->step_desc.resize(prog->step_type.size());
                    prog->step_desc.back() = d;
                    prog->steps.push_back([=](cudaStream_t st) { return launch_fc_stream(aptr, x_ld, batch, wptr, Kc, N, bias_p, act, out_p, o_ld, of32, st); });
                    break;
                }
                g.Kc = Kc; g.ntaps = ntaps; g.Wp = (int)ab.W + 2; g.kpt = (Kc + 63) / 64; g.BN = BN;
                g.act = act; g.out_f32 = ob.dtype == 1 ? 1 : 0;
                g.transposed = transposed;
                g.bias = static_cast<const float*>(tensor_ptr(e, bias_t));
                if (res_buf >= 0) {
                    const PlanBuffer& rb = e->bufs[res_buf];
                    g.res = static_cast<const __half*>(e->dbufs[res_buf].ptr) + res_coff;
                    g.res_ld = res_pre ? -(int)rb.C : (int)rb.C;
                }
                g.out = static_cast<uint8_t*>(e->dbufs[out_buf].ptr) + (size_t)out_coff * elem_size(ob.dtype);
                if (masked) { g.mask_H = (int)ob.H; g.mask_W = (int)ob.W; ADAS_CHECK(ob.H > 0, "op %zu: masked store into a dense buffer", oi); }
                if (e->conv_impl == 0) {
                    // ---- product path: gemm_v3.cu ----
                    void* opaque = nullptr;
                    std::vector<std::pair<int, int>> tiles;       // every tile that was prepared and launched (adas_engine_step_tiles)
                    int chosen = 0;
                    const uint64_t a_Wp = (uint64_t)ab.W + 2, a_Hp = (uint64_t)ab.H + 2, a_ldC = (uint64_t)ab.C;
                    std::function<int(const GemmParams&, void**)> prep = [=](const GemmParams& gc, void** out) -> int {
                        if (s2) return gemm_v3_prepare_s2(gc, aptr, (uint64_t)Kc, a_Wp, a_Hp, (uint64_t)batch, a_ldC, opB, b_inner, b_rows_u, b_stride, out);
                        return gemm_v3_prepare(gc, opA, a_inner, a_rows_u, a_stride, opB, b_inner, b_rows_u, b_stride, out);
                    };
                    if (!transposed && p[15] <= 0) {
                        // tile candidates ranked by the cost model; with autotuning the best few are timed on the device once per
                        // (op, batch).  Every candidate accumulates in the same K order, so the choice never changes results.
                        int cBN[16], cMT[16];
                        const int nc = gemm_v3_candidates(g, e->autotune ? 10 : 1, cBN, cMT);
                        float best_ms = 1e30f;
                        cudaEvent_t ev0 = nullptr, ev1 = nullptr;
                        if (nc > 1) { ADAS_CUDA(cudaEventCreate(&ev0)); ADAS_CUDA(cudaEventCreate(&ev1)); }
                        for (int ci = 0; ci < nc; ++ci) {
                            GemmParams gc = g;
                            gc.BN = cBN[ci]; gc.mt_hint = cMT[ci];
                            void* cand = nullptr;
                            if (prep(gc, &cand)) continue;
                            std::pair<int, int> tile;
                            gemm_v3_tile_of(cand, &tile.first, &tile.second);
                            if (nc == 1) { opaque = cand; tiles.push_back(tile); break; }
                            int rc = gemm_v3_run(cand, e->stream);
                            if (!rc) {
                                cudaEventRecord(ev0, e->stream);
                                for (int r = 0; r < 4 && !rc; ++r) rc = gemm_v3_run(cand, e->stream);
                                cudaEventRecord(ev1, e->stream);
                                if (cudaEventSynchronize(ev1) != cudaSuccess) rc = 1;
                            }
                            float ms = 1e30f;
                            if (!rc) cudaEventElapsedTime(&ms, ev0, ev1);
                            static const bool at_log = getenv("ADAS_B200_AT_LOG") != nullptr;
                            if (at_log) fprintf(stderr, "[autotune] op %zu M=%d N=%d K=%d taps=%d s2=%d BN=%d mt=%d : %.1f us\n", oi, g.M, g.N, Kc * ntaps, ntaps, s2,
                                                gc.BN, gc.mt_hint, rc ? -1.0 : ms * 1000.0 / 4.0);
                            if (!rc) tiles.push_back(tile);
                            if (!rc && ms < best_ms) { best_ms = ms; if (opaque) gemm_v3_free(opaque); opaque = cand; chosen = (int)tiles.size() - 1; }
                            else gemm_v3_free(cand);
                        }
                        if (ev0) { cudaEventDestroy(ev0); cudaEventDestroy(ev1); }
                        ADAS_CHECK(opaque != nullptr, "op %zu: no GEMM tile configuration could be launched (%s)", oi, g_err);
                    } else {
                        if (prep(g, &opaque)) return 1;
                        tiles.emplace_back();
                        gemm_v3_tile_of(opaque, &tiles[0].first, &tiles[0].second);
                    }
                    std::shared_ptr<void> keep(opaque, gemm_v3_free);
                    {
                        char d[256];
                        gemm_v3_describe(opaque, d, sizeof(d));
                        prog->step_desc.resize(prog->step_type.size());
                        prog->step_desc.back() = d;
                        prog->step_tiles.resize(prog->step_type.size());
                        prog->step_tiles.back() = tiles;
                        prog->step_chosen.resize(prog->step_type.size());
                        prog->step_chosen.back() = chosen;
                    }
                    {
                        GemmRec rec;
                        rec.step = prog->steps.size();
                        rec.g = g;
                        gemm_v3_tile_of(opaque, &rec.g.BN, &rec.g.mt_hint);
                        rec.a_buf = a_buf; rec.a_coff = a_coff; rec.out_buf = out_buf; rec.out_coff = out_coff; rec.res_buf = res_buf; rec.res_coff = res_coff;
                        rec.eligible = !s2 && !transposed && ob.dtype == 0 && masked && (ntaps == 1 || ntaps == 9) && N % 64 == 0 && rec.g.BN % 64 == 0 &&
                                       gemm_v3_is_staged(opaque);
                        rec.prep = prep;
                        recs.push_back(rec);
                    }
                    prog->steps.push_back([keep](cudaStream_t st) { return gemm_v3_run(keep.get(), st); });
                } else {
                    prog->steps.push_back([g](cudaStream_t st) { return gemm_simt_launch(g, st); });
                }
                break;
            }
            case OP_IM2COL: {
                const PlanBuffer& ib = e->bufs[p[0]];
                const PlanBuffer& ob = e->bufs[p[7]];
                const __half* in = static_cast<const __half*>(e->dbufs[p[0]].ptr);
                __half* out = static_cast<__half*>(e->dbufs[p[7]].ptr);
                const int in_ld = (int)ib.C, in_coff = p[1], H = (int)ib.H, W = (int)ib.W, Cin = p[2], kh = p[3], kw = p[4], s = p[5], pad = p[6];
                const int Ho = (int)ob.H, Wo = (int)ob.W, Kpad = (int)ob.C;
                ADAS_CHECK(kh * kw * Cin <= Kpad, "op %zu: im2col K exceeds the patch buffer width", oi);
                prog->steps.push_back([=](cudaStream_t st) {
                    return launch_im2col(in, in_ld, in_coff, batch, H, W, Cin, kh, kw, s, pad, Ho, Wo, out, Kpad, st);
                });
                break;
            }
            case OP_MAXPOOL: {
                const PlanBuffer& ib = e->bufs[p[0]];
                const PlanBuffer& ob = e->bufs[p[6]];
                const __half* in = static_cast<const __half*>(e->dbufs[p[0]].ptr) + p[1];
                __half* out = static_cast<__half*>(e->dbufs[p[6]].ptr) + p[7];
                const int in_ld = (int)ib.C, H = (int)ib.H, W = (int)ib.W, C = p[2], k = p[3], s = p[4], pad = p[5];
                const int out_ld = (int)ob.C, Ho = (int)ob.H, Wo = (int)ob.W;
                prog->steps.push_back([=](cudaStream_t st) { return launch_maxpool(in, in_ld, batch, H, W, C, k, s, pad, out, out_ld, Ho, Wo, st); });
                break;
            }
            case OP_UPSAMPLE2X: {
                const PlanBuffer& ib = e->bufs[p[0]];
                const PlanBuffer& ob = e->bufs[p[3]];
                const __half* in = static_cast<const __half*>(e->dbufs[p[0]].ptr) + p[1];
                __half* out = static_cast<__half*>(e->dbufs[p[3]].ptr) + p[4];
                const int in_ld = (int)ib.C, H = (int)ib.H, W = (int)ib.W, C = p[2], out_ld = (int)ob.C;
                ADAS_CHECK((int)ob.H == 2 * H && (int)ob.W == 2 * W, "op %zu: upsample geometry", oi);
                prog->steps.push_back([=](cudaStream_t st) { return launch_upsample2x(in, in_ld, batch, H, W, C, out, out_ld, st); });
                break;
            }
            case OP_STEMPACK: {
                const PlanBuffer& ib = e->bufs[p[0]];
                const PlanBuffer& ob = e->bufs[p[1]];
                ADAS_CHECK(ib.C == 4 && ob.C == 64 && ob.H * 2 == ib.H && ob.W * 2 == ib.W, "op %zu: stem pack geometry", oi);
                const __half* in = static_cast<const __half*>(e->dbufs[p[0]].ptr);
                __half* out = static_cast<__half*>(e->dbufs[p[1]].ptr);
                const int H = (int)ib.H, W = (int)ib.W;
                prog->steps.push_back([=](cudaStream_t st) { return launch_stempack(in, batch, H, W, out, st); });
                break;
            }
            case OP_STEMCONV: {
                const PlanBuffer& ib = e->bufs[p[0]];
                const PlanBuffer& ob = e->bufs[p[7]];
                const int Cout = p[3], k = p[4], pad = p[5], act = p[6], out_coff = p[8];
                ADAS_CHECK(ib.C == 4 && ib.dtype == 0 && ob.dtype == 0 && stem_conv_supported(Cout, k, pad) && out_coff % 8 == 0 && ob.C % 8 == 0, "op %zu: stem conv geometry", oi);
                const __half* in = static_cast<const __half*>(e->dbufs[p[0]].ptr);
                const __half* wq = static_cast<const __half*>(tensor_ptr(e, p[1]));
                const float* bias = static_cast<const float*>(tensor_ptr(e, p[2]));
                __half* out = static_cast<__half*>(e->dbufs[p[7]].ptr) + out_coff;
                const int H = (int)ib.H, W = (int)ib.W, Ho = (int)ob.H, Wo = (int)ob.W, out_ld = (int)ob.C;
                char d[128];
                snprintf(d, sizeof(d), "stem %dx%d s2 p%d 3->%d, %dx%d -> %dx%d, warp MMA from the image", k, k, pad, Cout, H, W, Ho, Wo);
                prog->step_desc.resize(prog->step_type.size());
                prog->step_desc.back() = d;
                prog->steps.push_back([=](cudaStream_t st) { return launch_stem_conv_s2(in, batch, H, W, wq, bias, Cout, k, pad, act, out, out_ld, Ho, Wo, st); });
                break;
            }
            case OP_LAYERNORM: {
                // each image's whole slab (rows_per_img * C elements) is one LayerNorm row
                const PlanBuffer& ib = e->bufs[p[0]];
                const PlanBuffer& ob = e->bufs[p[4]];
                const __half* in = static_cast<const __half*>(e->dbufs[p[0]].ptr);
                __half* out = static_cast<__half*>(e->dbufs[p[4]].ptr);
                const int in_ld = (int)(ib.rows_per_img * ib.C), d_len = p[1], d_norm = p[5], out_ld = (int)(ob.rows_per_img * ob.C);
                ADAS_CHECK(d_len <= in_ld && d_len <= out_ld && d_norm > 0, "op %zu: layernorm extent", oi);
                const float* gamma = static_cast<const float*>(tensor_ptr(e, p[2]));
                const float* beta = static_cast<const float*>(tensor_ptr(e, p[3]));
                const float eps = op.f[0];
                prog->steps.push_back([=](cudaStream_t st) { return launch_layernorm(in, in_ld, batch, d_len, d_norm, gamma, beta, eps, out, out_ld, st); });
                break;
            }
            default:
                ADAS_CHECK(false, "plan op %zu has unknown type %u", oi, op.type);
        }
    }
    prog->step_desc.resize(prog->steps.size());
    prog->step_tiles.resize(prog->steps.size());
    prog->step_chosen.resize(prog->steps.size());
    return build_chains(e, prog, recs);
}

// run the network for `batch` images already staged in buffer 0 (fp16 padded NHWC image)
static int run_plan(adas_engine* e, int batch) {
    NvtxRange nv(is_ufld(e->hdr.model_kind) ? "plan:ufld" : "plan:yolo");
    auto it = e->programs.find(batch);
    if (it == e->programs.end()) {
        Program prog;
        if (build_program(e, batch, &prog)) return 1;
        it = e->programs.emplace(batch, std::move(prog)).first;
    }
    Program& pg = it->second;
    if (pg.graph != nullptr) {
        ADAS_CUDA(cudaGraphLaunch(pg.graph, e->stream));
        count_launch(pg.n_launch());
        return 0;
    }
    if (e->use_graph && pg.runs >= 1) {
        // second run: capture the launch list once, replay it from then on
        cudaGraph_t graph = nullptr;
        ADAS_CUDA(cudaStreamBeginCapture(e->stream, cudaStreamCaptureModeThreadLocal));
        int rc = 0;
        for (auto& s : pg.steps) { rc = s(e->stream); if (rc) break; }
        cudaError_t ce = cudaStreamEndCapture(e->stream, &graph);
        if (rc) { if (graph) cudaGraphDestroy(graph); return 1; }
        ADAS_CUDA(ce);
        ADAS_CUDA(cudaGraphInstantiate(&pg.graph, graph, 0));
        ADAS_CUDA(cudaGraphDestroy(graph));
        ADAS_CUDA(cudaGraphLaunch(pg.graph, e->stream));
        pg.runs++;
        return 0;
    }
    for (auto& s : pg.steps) if (s(e->stream)) return 1;
    pg.runs++;
    return 0;
}

static int head_decode(adas_engine* e, int batch) {
    if (is_ufld(e->hdr.model_kind)) return 0;   // heads are the raw FC output buffer
    YoloLevel lv[3];
    ADAS_CHECK(e->outs.size() == 3, "YOLO plan must declare 3 output levels");
    for (int i = 0; i < 3; ++i) {
        const PlanOutput& o = e->outs[i];
        const PlanBuffer& b = e->bufs[o.buffer];
        lv[i].ptr = static_cast<const float*>(e->dbufs[o.buffer].ptr) + o.coff;
        lv[i].ld = (int)b.C; lv[i].H = (int)b.H; lv[i].W = (int)b.W; lv[i].stride = (int)o.stride;
        lv[i].rows_per_img = (int)b.rows_per_img;
    }
    const int nc = (int)e->hdr.meta[0], A = (int)e->hdr.meta[1];
    if (e->hdr.model_kind == ADAS_MODEL_YOLOV8) return launch_yolov8_head_decode(lv, batch, nc, e->d_raw, A, e->stream);
    return launch_yolov5_head_decode(lv, batch, nc, e->d_raw, A, (int)e->hdr.meta[2], e->stream);
}
// YOLOV5_LITE plans (meta[2] != 0): the network output is the sigmoid-only head; the fused detect calls apply
// YoloLiteParameters.lite_postprocess (yoloDetector.py:36-50) on the device before candidate selection.
static int lite_post(adas_engine* e, int batch) {
    if (e->hdr.model_kind != ADAS_MODEL_YOLOV5 || e->hdr.meta[2] == 0) return 0;
    return launch_yolov5_lite_post(e->d_raw, batch, (int)e->hdr.meta[1], (int)e->hdr.meta[0], (int)e->hdr.in_h, (int)e->hdr.in_w, e->stream);
}

static int alloc_yolo_post(YoloPostBufs* w, int B, int A, int max_det) {
    w->cap = A;        // every anchor may become a candidate: no limit the reference does not have
    ADAS_CUDA(cudaMalloc(&w->nms_work, (size_t)B * A * 7 * sizeof(double)));
    ADAS_CUDA(cudaMalloc(&w->flags, (size_t)B * A * 4));
    ADAS_CUDA(cudaMalloc(&w->cls, (size_t)B * A * 4));
    ADAS_CUDA(cudaMalloc(&w->conf, (size_t)B * A * 4));
    ADAS_CUDA(cudaMalloc(&w->n_cand, (size_t)B * 4));
    ADAS_CUDA(cudaMalloc(&w->cand_box, (size_t)B * w->cap * 16));
    ADAS_CUDA(cudaMalloc(&w->cand_conf, (size_t)B * w->cap * 4));
    ADAS_CUDA(cudaMalloc(&w->cand_cls, (size_t)B * w->cap * 4));
    ADAS_CUDA(cudaMalloc(&w->out_box, (size_t)B * max_det * 16));
    ADAS_CUDA(cudaMalloc(&w->out_score, (size_t)B * max_det * 4));
    ADAS_CUDA(cudaMalloc(&w->out_cls, (size_t)B * max_det * 4));
    ADAS_CUDA(cudaMalloc(&w->out_idx, (size_t)B * max_det * 4));
    ADAS_CUDA(cudaMalloc(&w->out_count, (size_t)B * 4));
    return 0;
}
static void free_yolo_post(YoloPostBufs* w) {
    cudaFree(w->nms_work); cudaFree(w->flags); cudaFree(w->cls); cudaFree(w->conf); cudaFree(w->n_cand); cudaFree(w->cand_box); cudaFree(w->cand_conf);
    cudaFree(w->cand_cls); cudaFree(w->out_box); cudaFree(w->out_score); cudaFree(w->out_cls); cudaFree(w->out_idx); cudaFree(w->out_count);
    memset(w, 0, sizeof(*w));
}

static int copy_yolo_results_enqueue(const YoloPostBufs& w, int batch, int max_det, float* boxes, float* scores, int32_t* cls, int32_t* idx,
                                     int32_t* counts, int32_t* nc_host, cudaStream_t st) {
    ADAS_CUDA(cudaMemcpyAsync(boxes, w.out_box, (size_t)batch * max_det * 16, cudaMemcpyDeviceToHost, st));
    ADAS_CUDA(cudaMemcpyAsync(scores, w.out_score, (size_t)batch * max_det * 4, cudaMemcpyDeviceToHost, st));
    ADAS_CUDA(cudaMemcpyAsync(cls, w.out_cls, (size_t)batch * max_det * 4, cudaMemcpyDeviceToHost, st));
    ADAS_CUDA(cudaMemcpyAsync(idx, w.out_idx, (size_t)batch * max_det * 4, cudaMemcpyDeviceToHost, st));
    ADAS_CUDA(cudaMemcpyAsync(counts, w.out_count, (size_t)batch * 4, cudaMemcpyDeviceToHost, st));
    ADAS_CUDA(cudaMemcpyAsync(nc_host, w.n_cand, (size_t)batch * 4, cudaMemcpyDeviceToHost, st));
    return 0;
}
static int copy_yolo_results_finish(const YoloPostBufs& w, int batch, int max_det, int32_t* counts, int32_t* n_cand, const int32_t* nc_host,
                                    cudaStream_t st) {
    ADAS_CUDA(cudaStreamSynchronize(st));
    for (int b = 0; b < batch; ++b) {
        if (n_cand) n_cand[b] = nc_host[b];
        // the reference returns every survivor; the caller-sized output arrays hold max_det per frame -- fail loudly instead of
        // dropping detections silently (advisor finding, r01)
        ADAS_CHECK(counts[b] <= max_det, "frame %d: %d detections survive the NMS but the output arrays hold %d (raise max_det)", b, counts[b], max_det);
    }
    return 0;
}
static int copy_yolo_results(const YoloPostBufs& w, int batch, int max_det, float* boxes, float* scores, int32_t* cls, int32_t* idx,
                             int32_t* counts, int32_t* n_cand, cudaStream_t st) {
    std::vector<int32_t> nc(batch);
    if (copy_yolo_results_enqueue(w, batch, max_det, boxes, scores, cls, idx, counts, nc.data(), st)) return 1;
    return copy_yolo_results_finish(w, batch, max_det, counts, n_cand, nc.data(), st);
}
static void ufld_lut_host(float* lut) {
    // ultrafastLaneDetectorV2.py:105-108,112 under numpy promotion rules: `img / 255.0` stays float32 (python scalar is
    // weak), `- mean` / `/ std` with python lists promote to float64, the final astype rounds once to float32.
    const double mean[3] = {0.485, 0.456, 0.406}, stdv[3] = {0.229, 0.224, 0.225};
    for (int c = 0; c < 3; ++c)
        for (int v = 0; v < 256; ++v) {
            const float q = (float)v / 255.0f;
            lut[c * 256 + v] = (float)(((double)q - mean[c]) / stdv[c]);
        }
}

}  // namespace adas

// =====================================================================================================
//                                            C ABI
// =====================================================================================================
extern "C" {

const char* adas_last_error(void) { return adas::g_err; }
int adas_version(void) { return 100; }
int64_t adas_launch_count(void) { return (int64_t)adas::g_launches.load(); }

// UFLDv2 dataset geometry (ModelConfig, ultrafastLaneDetectorV2.py:20-55).  The plan header names the dataset (meta[6]); crop ratio and
// anchors follow from it exactly as in the reference's ModelConfig -- they are not free parameters of a plan.
struct UfldDataset { int id; const char* name; int in_h, in_w, ngr, ncr, ngc, ncc; double crop, r0, r1, rdiv, c0, c1; };
static const UfldDataset kUfldDatasets[] = {
    {0, "CULane",   320, 1600, 200, 72, 100, 81, 0.6, 0.42, 1.0, 1.0, 0.0, 1.0},        // init_culane_config (47-55)
    {1, "TuSimple", 320,  800, 100, 56, 100, 41, 0.8, 160.0, 710.0, 720.0, 0.0, 1.0},   // init_tusimple_config (31-37): linspace(160,710,56)/720
};
// UFLD v1 dataset geometry (ModelConfig, ultrafastLaneDetector.py:15-37): source size the points are expressed in, grid cells, rows,
// row anchors in 288-row input coordinates (TuSimple: np.linspace(64, 284, 56); CULane: [round(v) for v in np.linspace(121, 287, 18)])
struct UfldV1Dataset { int id; const char* name; int img_w, img_h, G, R; double r0, r1; bool rounded; };
static const UfldV1Dataset kUfldV1Datasets[] = {
    {0, "CULane", 1640, 590, 200, 18, 121.0, 287.0, true},
    {1, "TuSimple", 1280, 720, 100, 56, 64.0, 284.0, false},
};
static const UfldV1Dataset* ufld_v1_dataset(const PlanHeader& h) {
    for (const UfldV1Dataset& d : kUfldV1Datasets)
        if ((int)h.meta[6] == d.id) return &d;
    return nullptr;
}

static const UfldDataset* ufld_dataset(const PlanHeader& h) {
    for (const UfldDataset& d : kUfldDatasets)
        if ((int)h.meta[6] == d.id) return &d;
    return nullptr;
}

// Every index, offset and size of a plan file is checked before anything is allocated or launched: a plan is input data (the
// reference trusts its .trt / .onnx files to TensorRT / ONNXRuntime, which validate them; here that job is ours).
static int validate_plan(const adas_engine* e, uint64_t file_bytes, const char* path) {
    const PlanHeader& h = e->hdr;
    const uint64_t rec_bytes = sizeof(PlanHeader) + (uint64_t)h.n_buffers * sizeof(PlanBuffer) + (uint64_t)h.n_ops * sizeof(PlanOp) +
                               (uint64_t)h.n_tensors * sizeof(PlanTensor) + (uint64_t)h.n_outputs * sizeof(PlanOutput);
    ADAS_CHECK(h.blob_offset >= rec_bytes && h.blob_offset <= file_bytes && h.blob_bytes <= file_bytes - h.blob_offset,
               "plan %s: weight blob [%llu, +%llu) lies outside the file (%llu bytes)", path, (unsigned long long)h.blob_offset,
               (unsigned long long)h.blob_bytes, (unsigned long long)file_bytes);
    ADAS_CHECK(h.in_c >= 1 && h.in_c <= 4 && h.in_h >= 1 && h.in_h <= 8192 && h.in_w >= 1 && h.in_w <= 8192, "plan %s: bad input binding %ux%ux%u", path, h.in_c, h.in_h, h.in_w);
    const int nb = (int)h.n_buffers, nt = (int)h.n_tensors;
    for (int i = 0; i < nb; ++i) {
        const PlanBuffer& b = e->bufs[i];
        ADAS_CHECK(b.rows_per_img >= 1 && b.C >= 1 && b.C <= (1u << 20) && b.dtype <= 1 && (uint64_t)b.rows_per_img * b.C <= (1ull << 31), "plan %s: buffer %d has a bad shape", path, i);
        ADAS_CHECK((b.H == 0 && b.W == 0) || (b.H >= 1 && b.W >= 1 && (uint64_t)(b.H + 2) * (b.W + 2) == b.rows_per_img), "plan %s: buffer %d: rows_per_img != (H+2)*(W+2)", path, i);
    }
    for (int i = 0; i < nt; ++i) {
        const PlanTensor& t = e->tensors[i];
        ADAS_CHECK(t.offset <= h.blob_bytes && t.bytes <= h.blob_bytes - t.offset && t.offset % 16 == 0 && t.dtype <= 1, "plan %s: tensor %d lies outside the weight blob", path, i);
    }
    auto buf_ok = [&](int b) { return b >= 0 && b < nb; };
    auto view_ok = [&](int b, int coff, int C) { return buf_ok(b) && coff >= 0 && C >= 1 && (uint64_t)coff + (uint64_t)C <= e->bufs[b].C; };
    auto tensor_ok = [&](int t, uint64_t min_bytes) { return t >= 0 && t < nt && e->tensors[t].bytes >= min_bytes; };
    for (size_t oi = 0; oi < e->ops.size(); ++oi) {
        const PlanOp& op = e->ops[oi];
        const int32_t* p = op.p;
        switch (op.type) {
            case OP_GEMM: {
                const int Kc = p[2], ntaps = p[3], N = p[6], transposed = p[14];
                ADAS_CHECK(Kc >= 8 && Kc <= (1 << 20) && N >= 1 && N <= (1 << 20) && (ntaps == 1 || ntaps == 4 || ntaps == 9), "plan %s: op %zu: bad GEMM shape", path, oi);
                ADAS_CHECK(buf_ok(p[0]) && buf_ok(p[11]) && p[1] >= 0 && p[12] >= 0, "plan %s: op %zu: GEMM buffer index out of range", path, oi);
                if (!transposed) {
                    ADAS_CHECK(view_ok(p[0], p[1], Kc) && view_ok(p[11], p[12], N), "plan %s: op %zu: GEMM channel slice exceeds its buffer", path, oi);
                } else {
                    const PlanBuffer &ab = e->bufs[p[0]], &ob = e->bufs[p[11]];
                    ADAS_CHECK(p[1] == 0 && p[12] == 0 && (uint64_t)Kc <= (uint64_t)ab.rows_per_img * ab.C && (uint64_t)N <= (uint64_t)ob.rows_per_img * ob.C,
                               "plan %s: op %zu: FC vector exceeds its buffer", path, oi);
                }
                ADAS_CHECK(tensor_ok(p[4], (uint64_t)N * Kc * ntaps * 2) && e->tensors[p[4]].dtype == 0, "plan %s: op %zu: weight tensor missing or too small", path, oi);
                ADAS_CHECK(p[5] < 0 || (tensor_ok(p[5], (uint64_t)N * 4) && e->tensors[p[5]].dtype == 1), "plan %s: op %zu: bias tensor missing or too small", path, oi);
                ADAS_CHECK(p[8] < 0 || (!transposed && view_ok(p[8], p[9], N) && e->bufs[p[8]].dtype == 0), "plan %s: op %zu: residual slice exceeds its buffer", path, oi);
                ADAS_CHECK(p[15] >= 0 && p[15] <= 256 && p[17] >= 0 && p[17] <= 4, "plan %s: op %zu: bad forced tile shape", path, oi);
                break;
            }
            case OP_IM2COL:
                ADAS_CHECK(buf_ok(p[0]) && buf_ok(p[7]) && view_ok(p[0], p[1], p[2]) && e->bufs[p[0]].H > 0 && e->bufs[p[7]].H > 0 && p[3] >= 1 && p[3] <= 7 && p[4] >= 1 && p[4] <= 7 &&
                           p[5] >= 1 && p[5] <= 4 && p[6] >= 0 && p[6] <= 3 && (uint64_t)p[2] * p[3] * p[4] <= e->bufs[p[7]].C,
                           "plan %s: op %zu: bad im2col", path, oi);
                break;
            case OP_MAXPOOL:
                ADAS_CHECK(view_ok(p[0], p[1], p[2]) && view_ok(p[6], p[7], p[2]) && e->bufs[p[0]].H > 0 && e->bufs[p[6]].H > 0 && p[3] >= 1 && p[3] <= 7 && p[4] >= 1 && p[4] <= 4 && p[5] >= 0 && p[5] <= 3,
                           "plan %s: op %zu: bad maxpool", path, oi);
                break;
            case OP_UPSAMPLE2X:
                ADAS_CHECK(view_ok(p[0], p[1], p[2]) && view_ok(p[3], p[4], p[2]) && e->bufs[p[0]].H > 0 && e->bufs[p[3]].H == 2 * e->bufs[p[0]].H && e->bufs[p[3]].W == 2 * e->bufs[p[0]].W,
                           "plan %s: op %zu: bad upsample", path, oi);
                break;
            case OP_STEMPACK:
                ADAS_CHECK(buf_ok(p[0]) && buf_ok(p[1]) && e->bufs[p[0]].H > 0 && e->bufs[p[1]].H > 0 && e->bufs[p[0]].C == 4 && e->bufs[p[1]].C == 64, "plan %s: op %zu: bad stem re-layout", path, oi);
                break;
            case OP_STEMCONV: {
                const int Cout = p[3], k = p[4];
                ADAS_CHECK(buf_ok(p[0]) && e->bufs[p[0]].H > 0 && e->bufs[p[0]].C == 4 && Cout >= 8 && Cout <= 64 && k >= 3 && k <= 7 && p[5] >= 0 && p[5] <= 3 &&
                           view_ok(p[7], p[8], Cout) && e->bufs[p[7]].H > 0 && tensor_ok(p[1], (uint64_t)Cout * k * ((4 * k + 15) / 16 * 16) * 2) &&
                           (p[2] < 0 || tensor_ok(p[2], (uint64_t)Cout * 4)) &&
                           e->bufs[p[7]].H == (e->bufs[p[0]].H + 2 * p[5] - k) / 2 + 1 && e->bufs[p[7]].W == (e->bufs[p[0]].W + 2 * p[5] - k) / 2 + 1,
                           "plan %s: op %zu: bad stem conv", path, oi);
                break;
            }
            case OP_LAYERNORM: {
                ADAS_CHECK(buf_ok(p[0]) && buf_ok(p[4]) && p[1] >= 1 && p[5] >= 1 && p[5] <= p[1], "plan %s: op %zu: bad layernorm", path, oi);
                const PlanBuffer &ib = e->bufs[p[0]], &ob = e->bufs[p[4]];
                ADAS_CHECK((uint64_t)p[1] <= (uint64_t)ib.rows_per_img * ib.C && (uint64_t)p[1] <= (uint64_t)ob.rows_per_img * ob.C && tensor_ok(p[2], (uint64_t)p[1] * 4) && tensor_ok(p[3], (uint64_t)p[1] * 4),
                           "plan %s: op %zu: layernorm vector exceeds its buffers", path, oi);
                break;
            }
            default:
                ADAS_CHECK(false, "plan %s: op %zu has unknown type %u", path, oi, op.type);
        }
    }
    for (size_t i = 0; i < e->outs.size(); ++i) {
        const PlanOutput& o = e->outs[i];
        ADAS_CHECK(buf_ok((int)o.buffer) && (uint64_t)o.coff + o.C <= (uint64_t)e->bufs[o.buffer].C * (e->bufs[o.buffer].H > 0 ? 1u : e->bufs[o.buffer].rows_per_img) && o.C >= 1,
                   "plan %s: output %zu exceeds its buffer", path, i);
    }
    if (h.n_outputs == 0) return 0;          // single-layer plans of the kernel tests: no network outputs, no head geometry
    if (h.model_kind == ADAS_MODEL_UFLDV2) {
        const uint64_t ngr = h.meta[0], ncr = h.meta[1], ngc = h.meta[2], ncc = h.meta[3], nl = h.meta[4];
        ADAS_CHECK(nl == 4 && ngr >= 2 && ncr >= 1 && ngc >= 2 && ncc >= 1 && ngr <= 1024 && ngc <= 1024 && ncr <= 1024 && ncc <= 1024, "plan %s: bad UFLD head dimensions", path);
        ADAS_CHECK(h.meta[5] == ngr * ncr * nl + ngc * ncc * nl + 2 * ncr * nl + 2 * ncc * nl, "plan %s: UFLD total_dim does not match the head dimensions", path);
        const UfldDataset* ds = ufld_dataset(h);
        ADAS_CHECK(ds != nullptr, "plan %s: unknown UFLD dataset id %u (0 = CULane, 1 = TuSimple; CurveLanes is rejected like the reference does)", path, h.meta[6]);
        ADAS_CHECK((int)ngr == ds->ngr && (int)ncr == ds->ncr && (int)ngc == ds->ngc && (int)ncc == ds->ncc && (int)h.in_h == ds->in_h && (int)h.in_w == ds->in_w,
                   "plan %s: head %llux%llu / %llux%llu at %ux%u is not the %s geometry its header names", path, (unsigned long long)ngr, (unsigned long long)ncr,
                   (unsigned long long)ngc, (unsigned long long)ncc, h.in_h, h.in_w, ds->name);
    } else if (h.model_kind == ADAS_MODEL_UFLDV1) {
        const UfldV1Dataset* ds = ufld_v1_dataset(h);
        ADAS_CHECK(ds != nullptr, "plan %s: unknown UFLD v1 dataset id %u (0 = CULane, 1 = TuSimple)", path, h.meta[6]);
        ADAS_CHECK((int)h.meta[0] == ds->G && (int)h.meta[1] == ds->R && h.meta[4] == 4 && h.meta[5] == (uint64_t)(ds->G + 1) * ds->R * 4 && h.in_h == 288 && h.in_w == 800,
                   "plan %s: head %ux%u at %ux%u is not the UFLD v1 %s geometry its header names", path, h.meta[0], h.meta[1], h.in_h, h.in_w, ds->name);
    } else {
        ADAS_CHECK(h.model_kind == ADAS_MODEL_YOLOV8 || h.model_kind == ADAS_MODEL_YOLOV5, "plan %s: unknown model kind %u", path, h.model_kind);
        ADAS_CHECK(h.meta[0] >= 1 && h.meta[0] <= 1024 && h.meta[1] >= 1 && h.meta[1] <= (1u << 22), "plan %s: bad class / anchor counts", path);
    }
    return 0;
}

int adas_engine_create(const char* plan_path, int device, int max_batch, int conv_impl, adas_engine** out) {
    ADAS_CHECK(out != nullptr && plan_path != nullptr, "adas_engine_create: null argument");
    *out = nullptr;
    FILE* f = fopen(plan_path, "rb");
    // same wording class as EngineBase.__init__ (coreEngine.py:12-13)
    ADAS_CHECK(f != nullptr, "The model path [%s] can't not found!", plan_path);
    std::unique_ptr<adas_engine> e(new adas_engine());
    e->device = device; e->max_batch = max_batch; e->conv_impl = conv_impl;
    const char* ng = getenv("ADAS_B200_NO_GRAPH");
    e->use_graph = !(ng && ng[0] == '1');
    const char* ch = getenv("ADAS_B200_CHAIN");
    e->use_chain = !ch ? 0 : ch[0] == '0' ? 0 : ch[0] == '1' ? 1 : 2;
    const char* at = getenv("ADAS_B200_AUTOTUNE");
    e->autotune = !(at && at[0] == '0');
    bool ok = fread(&e->hdr, sizeof(PlanHeader), 1, f) == 1 && memcmp(e->hdr.magic, kPlanMagic, 8) == 0 && e->hdr.version == kPlanVersion;
    if (!ok) { fclose(f); ADAS_CHECK(false, "Parameters must be a .b200w plan file (bad magic/version): %s", plan_path); }
    if (e->hdr.n_buffers > 65536 || e->hdr.n_ops > 65536 || e->hdr.n_tensors > 65536 || e->hdr.n_outputs > 64) { fclose(f); ADAS_CHECK(false, "plan %s: implausible record counts", plan_path); }
    e->bufs.resize(e->hdr.n_buffers); e->ops.resize(e->hdr.n_ops); e->tensors.resize(e->hdr.n_tensors); e->outs.resize(e->hdr.n_outputs);
    ok = fread(e->bufs.data(), sizeof(PlanBuffer), e->bufs.size(), f) == e->bufs.size() &&
         fread(e->ops.data(), sizeof(PlanOp), e->ops.size(), f) == e->ops.size() &&
         fread(e->tensors.data(), sizeof(PlanTensor), e->tensors.size(), f) == e->tensors.size() &&
         fread(e->outs.data(), sizeof(PlanOutput), e->outs.size(), f) == e->outs.size();
    if (!ok) { fclose(f); ADAS_CHECK(false, "truncated plan file %s", plan_path); }
    fseek(f, 0, SEEK_END);
    const uint64_t file_bytes = (uint64_t)ftell(f);
    if (validate_plan(e.get(), file_bytes, plan_path)) { fclose(f); return 1; }
    std::vector<uint8_t> blob(e->hdr.blob_bytes);
    fseek(f, (long)e->hdr.blob_offset, SEEK_SET);
    ok = fread(blob.data(), 1, blob.size(), f) == blob.size();
    fclose(f);
    ADAS_CHECK(ok, "truncated plan blob in %s", plan_path);

    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    ADAS_CHECK(ce == cudaSuccess && ndev > 0, "no CUDA device available: libadas_b200 has no CPU fallback (%s)", cudaGetErrorString(ce));
    ADAS_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    ADAS_CUDA(cudaGetDeviceProperties(&prop, device));
    ADAS_CHECK(prop.major == 10, "device %d is sm_%d%d; libadas_b200 is built for sm_100a only", device, prop.major, prop.minor);
    ADAS_CUDA(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
    ADAS_CUDA(cudaMalloc(&e->d_blob, blob.size() + 256));
    ADAS_CUDA(cudaMemcpy(e->d_blob, blob.data(), blob.size(), cudaMemcpyHostToDevice));
    e->dbufs.resize(e->bufs.size());
    for (size_t i = 0; i < e->bufs.size(); ++i) {
        const PlanBuffer& b = e->bufs[i];
        const size_t bytes = (size_t)max_batch * b.rows_per_img * b.C * elem_size(b.dtype) + 256;
        ADAS_CUDA(cudaMalloc(&e->dbufs[i].ptr, bytes));
        ADAS_CUDA(cudaMemset(e->dbufs[i].ptr, 0, bytes));
        e->dbufs[i].bytes = bytes;
    }
    const size_t in_elems = (size_t)e->hdr.in_c * e->hdr.in_h * e->hdr.in_w;
    ADAS_CUDA(cudaMalloc(&e->d_input, (size_t)max_batch * in_elems * 4));
    if (e->hdr.model_kind == ADAS_MODEL_UFLDV1) {
        float lut[768];
        ufld_lut_host(lut);
        ADAS_CUDA(cudaMalloc(&e->d_lut, sizeof(lut)));
        ADAS_CUDA(cudaMemcpy(e->d_lut, lut, sizeof(lut), cudaMemcpyHostToDevice));
        const UfldV1Dataset* ds = ufld_v1_dataset(e->hdr);
        const int R = ds->R;
        e->ufld_max_pts = R;
        e->ufld_crop = 1.0;                        // v1 resizes the whole frame to 800x288 (ultrafastLaneDetector.py:86)
        std::vector<double> ra(R);
        for (int i = 0; i < R; ++i) {
            const double v = (i == R - 1) ? ds->r1 : ds->r0 + (double)i * ((ds->r1 - ds->r0) / (double)(R - 1));
            ra[i] = ds->rounded ? nearbyint(v) : v;      // Python round(): half to even
        }
        ADAS_CUDA(cudaMalloc(&e->d_row_anchor, R * 8));
        ADAS_CUDA(cudaMemcpy(e->d_row_anchor, ra.data(), R * 8, cudaMemcpyHostToDevice));
        ADAS_CUDA(cudaMalloc(&e->d_pts, (size_t)max_batch * 4 * R * 2 * 4));
        ADAS_CUDA(cudaMalloc(&e->d_npts, (size_t)max_batch * 4 * 4));
        ADAS_CUDA(cudaMalloc(&e->d_status, (size_t)max_batch * 4));
        ADAS_CUDA(cudaMalloc(&e->d_coords, (size_t)max_batch * 4 * R * 8));
    } else if (e->hdr.model_kind == ADAS_MODEL_UFLDV2) {
        float lut[768];
        ufld_lut_host(lut);
        ADAS_CUDA(cudaMalloc(&e->d_lut, sizeof(lut)));
        ADAS_CUDA(cudaMemcpy(e->d_lut, lut, sizeof(lut), cudaMemcpyHostToDevice));
        const int ncr = (int)e->hdr.meta[1], ncc = (int)e->hdr.meta[3];
        e->ufld_max_pts = ncr > ncc ? ncr : ncc;
        // anchors of the plan's dataset (ModelConfig, ultrafastLaneDetectorV2.py:31-55) with np.linspace semantics:
        // start + i*step, step = (stop-start)/(n-1), last element forced to stop; TuSimple divides the row anchors by 720 afterwards
        const UfldDataset* ds = ufld_dataset(e->hdr);
        e->ufld_crop = ds->crop;
        std::vector<double> ra(ncr), ca(ncc);
        for (int i = 0; i < ncr; ++i) ra[i] = ((i == ncr - 1) ? ds->r1 : ds->r0 + (double)i * ((ds->r1 - ds->r0) / (double)(ncr - 1))) / ds->rdiv;
        for (int i = 0; i < ncc; ++i) ca[i] = (i == ncc - 1) ? ds->c1 : ds->c0 + (double)i * ((ds->c1 - ds->c0) / (double)(ncc - 1));
        ADAS_CUDA(cudaMalloc(&e->d_row_anchor, ncr * 8));
        ADAS_CUDA(cudaMalloc(&e->d_col_anchor, ncc * 8));
        ADAS_CUDA(cudaMemcpy(e->d_row_anchor, ra.data(), ncr * 8, cudaMemcpyHostToDevice));
        ADAS_CUDA(cudaMemcpy(e->d_col_anchor, ca.data(), ncc * 8, cudaMemcpyHostToDevice));
        ADAS_CUDA(cudaMalloc(&e->d_pts, (size_t)max_batch * 4 * e->ufld_max_pts * 2 * 4));
        ADAS_CUDA(cudaMalloc(&e->d_npts, (size_t)max_batch * 4 * 4));
        ADAS_CUDA(cudaMalloc(&e->d_status, (size_t)max_batch * 4));
        ADAS_CUDA(cudaMalloc(&e->d_coords, (size_t)max_batch * 4 * e->ufld_max_pts * 8));
    } else {
        const int nc = (int)e->hdr.meta[0], A = (int)e->hdr.meta[1];
        e->raw_per_img = e->hdr.model_kind == ADAS_MODEL_YOLOV8 ? (size_t)(4 + nc) * A : (size_t)A * (5 + nc);
        ADAS_CUDA(cudaMalloc(&e->d_raw, (size_t)max_batch * e->raw_per_img * 4));
    }
    *out = e.release();
    return 0;
}

int adas_engine_destroy(adas_engine* e) {
    if (!e) return 0;
    cudaSetDevice(e->device);
    if (e->stream) cudaStreamSynchronize(e->stream);
    for (auto& kv : e->programs) if (kv.second.graph) cudaGraphExecDestroy(kv.second.graph);
    for (auto& b : e->dbufs) cudaFree(b.ptr);
    cudaFree(e->d_blob); cudaFree(e->d_input); cudaFree(e->d_frames); cudaFree(e->d_raw); cudaFree(e->d_lut);
    cudaFree(e->d_warp); cudaFree(e->d_warpM);
    cudaFree(e->d_area); cudaFree(e->d_bird); cudaFree(e->d_geom); cudaFree(e->d_M);
    cudaFree(e->d_row_anchor); cudaFree(e->d_col_anchor); cudaFree(e->d_pts); cudaFree(e->d_npts); cudaFree(e->d_status); cudaFree(e->d_coords);
    if (e->ev_frames) cudaEventDestroy(e->ev_frames);
    if (e->yp.flags) free_yolo_post(&e->yp);
    if (e->stream) cudaStreamDestroy(e->stream);
    delete e;
    return 0;
}

int adas_engine_model_kind(const adas_engine* e, int* kind) { *kind = (int)e->hdr.model_kind; return 0; }
int adas_engine_meta(const adas_engine* e, int idx, int* value) {
    ADAS_CHECK(e != nullptr && idx >= 0 && idx < 16 && value != nullptr, "adas_engine_meta: bad index %d", idx);
    *value = (int)e->hdr.meta[idx];
    return 0;
}
int adas_engine_input_shape(const adas_engine* e, int64_t s[4]) {
    s[0] = 1; s[1] = e->hdr.in_c; s[2] = e->hdr.in_h; s[3] = e->hdr.in_w;
    return 0;
}
int adas_engine_num_outputs(const adas_engine* e, int* n) { *n = e->hdr.model_kind == ADAS_MODEL_UFLDV2 ? 4 : 1; return 0; }     // UFLD v1: one tensor
int adas_engine_output_shape(const adas_engine* e, int idx, int64_t s[4], int* rank) {
    const uint32_t* m = e->hdr.meta;
    s[0] = 1; s[1] = s[2] = s[3] = 0;
    if (e->hdr.model_kind == ADAS_MODEL_YOLOV8) { ADAS_CHECK(idx == 0, "bad output index"); s[1] = 4 + m[0]; s[2] = m[1]; *rank = 3; }
    else if (e->hdr.model_kind == ADAS_MODEL_YOLOV5) { ADAS_CHECK(idx == 0, "bad output index"); s[1] = m[1]; s[2] = 5 + m[0]; *rank = 3; }
    else if (e->hdr.model_kind == ADAS_MODEL_UFLDV1) { ADAS_CHECK(idx == 0, "bad output index"); s[1] = m[0] + 1; s[2] = m[1]; s[3] = m[4]; *rank = 4; }   // [griding_num + 1, rows, lanes]
    else {
        ADAS_CHECK(idx >= 0 && idx < 4, "bad output index");
        *rank = 4;
        if (idx == 0) { s[1] = m[0]; s[2] = m[1]; s[3] = m[4]; }        // loc_row  [ngr, ncr, nl]
        else if (idx == 1) { s[1] = m[2]; s[2] = m[3]; s[3] = m[4]; }   // loc_col  [ngc, ncc, nl]
        else if (idx == 2) { s[1] = 2; s[2] = m[1]; s[3] = m[4]; }      // exist_row
        else { s[1] = 2; s[2] = m[3]; s[3] = m[4]; }                    // exist_col
    }
    return 0;
}
int adas_engine_stream(const adas_engine* e, void** st) { *st = (void*)e->stream; return 0; }

static int infer_common(adas_engine* e, const float* input, int batch, float* const* outs, bool on_device) {
    ADAS_CHECK(e != nullptr, "null engine");
    ADAS_CHECK(batch >= 1 && batch <= e->max_batch, "batch %d outside [1, %d]", batch, e->max_batch);
    ADAS_CUDA(cudaSetDevice(e->device));
    const size_t in_elems = (size_t)e->hdr.in_c * e->hdr.in_h * e->hdr.in_w;
    const float* din = input;
    if (!on_device) {
        ADAS_CUDA(cudaMemcpyAsync(e->d_input, input, (size_t)batch * in_elems * 4, cudaMemcpyHostToDevice, e->stream));
        din = e->d_input;
    }
    const PlanBuffer& ib = e->bufs[0];
    if (launch_nchw_to_padded(din, batch, (int)e->hdr.in_c, (int)e->hdr.in_h, (int)e->hdr.in_w, static_cast<__half*>(e->dbufs[0].ptr),
                              (int)ib.C, e->stream)) return 1;
    if (run_plan(e, batch)) return 1;
    if (head_decode(e, batch)) return 1;
    const cudaMemcpyKind kind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
    if (e->hdr.model_kind == ADAS_MODEL_UFLDV2) {
        const uint32_t* m = e->hdr.meta;
        const size_t total = m[5];
        const size_t sz[4] = {(size_t)m[0] * m[1] * m[4], (size_t)m[2] * m[3] * m[4], (size_t)2 * m[1] * m[4], (size_t)2 * m[3] * m[4]};
        const PlanOutput& o = e->outs[0];
        const float* src = static_cast<const float*>(e->dbufs[o.buffer].ptr) + o.coff;
        const size_t ld = e->bufs[o.buffer].C;
        size_t off = 0;
        for (int k = 0; k < 4; ++k) {
            ADAS_CUDA(cudaMemcpy2DAsync(outs[k], sz[k] * 4, src + off, ld * 4, sz[k] * 4, batch, kind, e->stream));
            off += sz[k];
        }
        (void)total;
    } else if (e->hdr.model_kind == ADAS_MODEL_UFLDV1) {
        const PlanOutput& o = e->outs[0];
        const float* src = static_cast<const float*>(e->dbufs[o.buffer].ptr) + o.coff;
        const size_t total = e->hdr.meta[5], ld = e->bufs[o.buffer].C;
        ADAS_CUDA(cudaMemcpy2DAsync(outs[0], total * 4, src, ld * 4, total * 4, batch, kind, e->stream));
    } else {
        ADAS_CUDA(cudaMemcpyAsync(outs[0], e->d_raw, (size_t)batch * e->raw_per_img * 4, kind, e->stream));
    }
    ADAS_CUDA(cudaStreamSynchronize(e->stream));
    return 0;
}

int adas_engine_infer(adas_engine* e, const float* input, int batch, float* const* outs) { return infer_common(e, input, batch, outs, false); }
int adas_engine_infer_dev(adas_engine* e, const float* input, int batch, float* const* outs) { return infer_common(e, input, batch, outs, true); }

static int stage_frames(adas_engine* e, const uint8_t* frames, int on_device, int batch, int H, int W, const uint8_t** dptr) {
    e->last_fb = batch; e->last_fh = H; e->last_fw = W;
    if (on_device) { *dptr = frames; e->last_dfr = frames; return 0; }
    const size_t bytes = (size_t)batch * H * W * 3;
    if (bytes > e->frames_cap) {
        if (e->d_frames) ADAS_CUDA(cudaFree(e->d_frames));
        e->d_frames = nullptr;
        const size_t cap = (size_t)e->max_batch * H * W * 3;
        ADAS_CUDA(cudaMalloc(&e->d_frames, cap));
        e->frames_cap = cap;
    }
    ADAS_CUDA(cudaMemcpyAsync(e->d_frames, frames, bytes, cudaMemcpyHostToDevice, e->stream));
    *dptr = e->d_frames;
    e->last_dfr = e->d_frames;
    return 0;
}

int adas_yolo_detect(adas_engine* e, const uint8_t* frames, int frames_on_device, int batch, int H, int W, double box_score,
                     double nms_iou, int max_det, float* boxes_xywh, float* scores, int32_t* class_ids, int32_t* cand_index,
                     int32_t* counts, int32_t* n_candidates) {
    ADAS_CHECK(e != nullptr, "null engine");
    ADAS_CHECK(!is_ufld(e->hdr.model_kind), "adas_yolo_detect on a UFLD plan");
    ADAS_CHECK(batch >= 1 && batch <= e->max_batch, "batch %d outside [1, %d]", batch, e->max_batch);
    ADAS_CUDA(cudaSetDevice(e->device));
    const int nc = (int)e->hdr.meta[0], A = (int)e->hdr.meta[1];
    if (e->yp.flags == nullptr || e->yp_max_det != max_det) {
        if (e->yp.flags) free_yolo_post(&e->yp);
        if (alloc_yolo_post(&e->yp, e->max_batch, A, max_det)) return 1;
        e->yp_max_det = max_det;
    }
    const uint8_t* dfr = nullptr;
    NvtxRange nv("adas_yolo_detect");
    PhaseTrace tr(e->stream, "yolo_detect");
    if (stage_frames(e, frames, frames_on_device, batch, H, W, &dfr)) return 1;
    tr.mark("h2d");
    const LetterboxGeom g = letterbox_geom(H, W, (int)e->hdr.in_h, (int)e->hdr.in_w);
    if (launch_yolo_pre(dfr, batch, g, static_cast<__half*>(e->dbufs[0].ptr), (int)e->bufs[0].C, nullptr, e->stream)) return 1;
    tr.mark("pre");
    if (run_plan(e, batch)) return 1;
    tr.mark("plan");
    if (head_decode(e, batch)) return 1;
    if (lite_post(e, batch)) return 1;
    tr.mark("decode");
    if (launch_yolo_post(e->d_raw, (int)e->hdr.model_kind, batch, A, nc, g, box_score, nms_iou, max_det, e->yp, e->stream)) return 1;
    tr.mark("select+nms");
    const int rc = copy_yolo_results(e->yp, batch, max_det, boxes_xywh, scores, class_ids, cand_index, counts, n_candidates, e->stream);
    tr.mark("d2h");
    tr.report();
    return rc;
}

int adas_yolo_postprocess(int device, const float* raw_host, int model_kind, int batch, int n_anchors, int n_classes, int in_h,
                          int in_w, int src_h, int src_w, double box_score, double nms_iou, int max_det, float* boxes_xywh,
                          float* scores, int32_t* class_ids, int32_t* cand_index, int32_t* counts, int32_t* n_candidates) {
    ADAS_CUDA(cudaSetDevice(device));
    ADAS_CHECK(model_kind == ADAS_MODEL_YOLOV8 || model_kind == ADAS_MODEL_YOLOV5 || model_kind == ADAS_MODEL_YOLOV5_LITE, "adas_yolo_postprocess: bad model kind %d", model_kind);
    const size_t per = model_kind == ADAS_MODEL_YOLOV8 ? (size_t)(4 + n_classes) * n_anchors : (size_t)n_anchors * (5 + n_classes);
    float* d_raw = nullptr;
    ADAS_CUDA(cudaMalloc(&d_raw, (size_t)batch * per * 4));
    ADAS_CUDA(cudaMemcpy(d_raw, raw_host, (size_t)batch * per * 4, cudaMemcpyHostToDevice));
    YoloPostBufs w{};
    int rc = alloc_yolo_post(&w, batch, n_anchors, max_det);
    const LetterboxGeom g = letterbox_geom(src_h, src_w, in_h, in_w);
    if (!rc && model_kind == ADAS_MODEL_YOLOV5_LITE) {       // raw is the sigmoid-only head of a lite export: lite_postprocess first
        rc = launch_yolov5_lite_post(d_raw, batch, n_anchors, n_classes, in_h, in_w, 0);
        model_kind = ADAS_MODEL_YOLOV5;
    }
    if (!rc) rc = launch_yolo_post(d_raw, model_kind, batch, n_anchors, n_classes, g, box_score, nms_iou, max_det, w, 0);
    if (!rc) rc = copy_yolo_results(w, batch, max_det, boxes_xywh, scores, class_ids, cand_index, counts, n_candidates, 0);
    free_yolo_post(&w);
    cudaFree(d_raw);
    return rc;
}

int adas_yolo_preprocess(int device, const uint8_t* frames_host, int batch, int H, int W, int in_h, int in_w, float* blob) {
    ADAS_CUDA(cudaSetDevice(device));
    uint8_t* d_fr = nullptr; float* d_blob = nullptr;
    const size_t fb = (size_t)batch * H * W * 3, bb = (size_t)batch * 3 * in_h * in_w * 4;
    ADAS_CUDA(cudaMalloc(&d_fr, fb));
    ADAS_CUDA(cudaMalloc(&d_blob, bb));
    ADAS_CUDA(cudaMemcpy(d_fr, frames_host, fb, cudaMemcpyHostToDevice));
    const LetterboxGeom g = letterbox_geom(H, W, in_h, in_w);
    int rc = launch_yolo_pre(d_fr, batch, g, nullptr, 0, d_blob, 0);
    if (!rc) { cudaError_t ce = cudaMemcpy(blob, d_blob, bb, cudaMemcpyDeviceToHost); if (ce != cudaSuccess) { set_error("D2H failed: %s", cudaGetErrorString(ce)); rc = 1; } }
    cudaFree(d_fr); cudaFree(d_blob);
    return rc;
}

// lane decode of the head tensor(s) the plan just produced: v2 row / column anchors or the v1 grid expectation
static int ufld_post_dispatch(adas_engine* e, int batch, int W, int H, bool want_coords) {
    const uint32_t* m = e->hdr.meta;
    const PlanOutput& o = e->outs[0];
    const float* heads = static_cast<const float*>(e->dbufs[o.buffer].ptr) + o.coff;
    const int mp = e->ufld_max_pts;
    if (e->hdr.model_kind == ADAS_MODEL_UFLDV1) {
        const UfldV1Dataset* ds = ufld_v1_dataset(e->hdr);
        return launch_ufld_v1_post(heads, (int)e->bufs[o.buffer].C, batch, ds->G, ds->R, (int)e->hdr.in_w, (int)e->hdr.in_h, ds->img_w, ds->img_h, W, H,
                                   e->d_row_anchor, e->d_pts, e->d_npts, e->d_status, want_coords ? e->d_coords : nullptr, mp, e->stream);
    }
    UfldDims d{(int)m[0], (int)m[1], (int)m[2], (int)m[3], (int)m[4]};
    return launch_ufld_post(heads, (int)e->bufs[o.buffer].C, batch, d, W, H, e->d_row_anchor, e->d_col_anchor, e->d_pts, e->d_npts, e->d_status,
                            want_coords ? e->d_coords : nullptr, mp, e->stream);
}

int adas_ufld_detect(adas_engine* e, const uint8_t* frames, int frames_on_device, int batch, int H, int W, int32_t* pts, int32_t* npts,
                     uint8_t* status, double* coords_f) {
    ADAS_CHECK(e != nullptr, "null engine");
    ADAS_CHECK(is_ufld(e->hdr.model_kind), "adas_ufld_detect on a YOLO plan");
    ADAS_CHECK(batch >= 1 && batch <= e->max_batch, "batch %d outside [1, %d]", batch, e->max_batch);
    ADAS_CUDA(cudaSetDevice(e->device));
    const uint8_t* dfr = nullptr;
    NvtxRange nv("adas_ufld_detect");
    PhaseTrace tr(e->stream, "ufld_detect");
    if (stage_frames(e, frames, frames_on_device, batch, H, W, &dfr)) return 1;
    tr.mark("h2d");
    const int in_h = (int)e->hdr.in_h, in_w = (int)e->hdr.in_w;
    const int resize_h = (int)((double)in_h / e->ufld_crop);   // int(self.input_height / cfg.crop_ratio)
    if (launch_ufld_pre(dfr, batch, H, W, in_h, in_w, resize_h, e->d_lut, static_cast<__half*>(e->dbufs[0].ptr), (int)e->bufs[0].C, nullptr,
                        e->stream)) return 1;
    tr.mark("pre");
    if (run_plan(e, batch)) return 1;
    tr.mark("plan");
    const int mp = e->ufld_max_pts;
    if (ufld_post_dispatch(e, batch, W, H, coords_f != nullptr)) return 1;
    ADAS_CUDA(cudaMemcpyAsync(pts, e->d_pts, (size_t)batch * 4 * mp * 2 * 4, cudaMemcpyDeviceToHost, e->stream));
    ADAS_CUDA(cudaMemcpyAsync(npts, e->d_npts, (size_t)batch * 4 * 4, cudaMemcpyDeviceToHost, e->stream));
    ADAS_CUDA(cudaMemcpyAsync(status, e->d_status, (size_t)batch * 4, cudaMemcpyDeviceToHost, e->stream));
    if (coords_f) ADAS_CUDA(cudaMemcpyAsync(coords_f, e->d_coords, (size_t)batch * 4 * mp * 8, cudaMemcpyDeviceToHost, e->stream));
    ADAS_CUDA(cudaStreamSynchronize(e->stream));
    e->ufld_last_batch = batch;
    tr.mark("post+d2h");
    tr.report();
    return 0;
}

int adas_engine_warp_perspective(adas_engine* e, int batch, const double* M, int out_h, int out_w, uint8_t* out_host) {
    ADAS_CHECK(e != nullptr && M != nullptr && out_host != nullptr, "adas_engine_warp_perspective: null argument");
    ADAS_CHECK(e->last_dfr != nullptr && batch >= 1 && batch <= e->last_fb, "adas_engine_warp_perspective: batch %d, but the last detect call on this engine processed %d frames",
               batch, e->last_fb);
    ADAS_CUDA(cudaSetDevice(e->device));
    const size_t bytes = (size_t)batch * out_h * out_w * 3;
    if (bytes > e->warp_cap || e->d_warpM == nullptr) {
        cudaFree(e->d_warp); cudaFree(e->d_warpM);
        e->d_warp = nullptr; e->d_warpM = nullptr;
        e->warp_cap = (size_t)e->max_batch * out_h * out_w * 3;
        ADAS_CUDA(cudaMalloc(&e->d_warp, e->warp_cap));
        ADAS_CUDA(cudaMalloc(&e->d_warpM, (size_t)e->max_batch * 72));
    }
    if (launch_warp_perspective(e->last_dfr, batch, e->last_fh, e->last_fw, M, e->d_warpM, e->d_warp, out_h, out_w, e->stream)) return 1;
    ADAS_CUDA(cudaMemcpyAsync(out_host, e->d_warp, bytes, cudaMemcpyDeviceToHost, e->stream));
    ADAS_CUDA(cudaStreamSynchronize(e->stream));
    return 0;
}

int adas_ufld_lane_geometry(adas_engine* e, int batch, int img_w, int img_h, int adjust_lanes, const double* M, int bird_w, int bird_h, int32_t* area,
                            int cap_area, int32_t* bird, adas_lane_geom* out) {
    ADAS_CHECK(e != nullptr && is_ufld(e->hdr.model_kind), "adas_ufld_lane_geometry needs a UFLD engine");
    ADAS_CHECK(batch >= 1 && batch <= e->ufld_last_batch, "adas_ufld_lane_geometry: batch %d, but the last lane detect on this engine decoded %d frames", batch, e->ufld_last_batch);
    ADAS_CHECK(area != nullptr && out != nullptr && (M == nullptr || bird != nullptr), "adas_ufld_lane_geometry: null argument");
    ADAS_CUDA(cudaSetDevice(e->device));
    const int mp = e->ufld_max_pts;
    if (e->d_geom == nullptr || e->geom_cap_area < cap_area) {
        cudaFree(e->d_warp); cudaFree(e->d_warpM);
    cudaFree(e->d_area); cudaFree(e->d_bird); cudaFree(e->d_geom); cudaFree(e->d_M);
        e->d_area = nullptr; e->d_bird = nullptr; e->d_geom = nullptr; e->d_M = nullptr;
        ADAS_CUDA(cudaMalloc(&e->d_area, (size_t)e->max_batch * cap_area * 8));
        ADAS_CUDA(cudaMalloc(&e->d_bird, (size_t)e->max_batch * 4 * mp * 8));
        ADAS_CUDA(cudaMalloc(&e->d_geom, (size_t)e->max_batch * sizeof(adas_lane_geom)));
        ADAS_CUDA(cudaMalloc(&e->d_M, (size_t)e->max_batch * 72));
        e->geom_cap_area = cap_area;
    }
    // the decoded points of the last adas_ufld_detect / adas_detect_pair are still resident (d_pts, d_npts, d_status): no re-upload
    if (M) ADAS_CUDA(cudaMemcpyAsync(e->d_M, M, (size_t)batch * 72, cudaMemcpyHostToDevice, e->stream));
    if (launch_lane_geom(e->d_pts, e->d_npts, e->d_status, M ? e->d_M : nullptr, batch, mp, img_w, img_h, adjust_lanes, bird_w, bird_h, e->d_area, cap_area,
                         e->d_bird, e->d_geom, e->stream)) return 1;
    ADAS_CUDA(cudaMemcpyAsync(area, e->d_area, (size_t)batch * cap_area * 8, cudaMemcpyDeviceToHost, e->stream));
    ADAS_CUDA(cudaMemcpyAsync(out, e->d_geom, (size_t)batch * sizeof(adas_lane_geom), cudaMemcpyDeviceToHost, e->stream));
    if (M) ADAS_CUDA(cudaMemcpyAsync(bird, e->d_bird, (size_t)batch * 4 * mp * 8, cudaMemcpyDeviceToHost, e->stream));
    ADAS_CUDA(cudaStreamSynchronize(e->stream));
    return 0;
}

int adas_detect_pair(adas_engine* yolo, adas_engine* ufld, const uint8_t* frames, int frames_on_device, int batch, int H, int W, double box_score,
                     double nms_iou, int max_det, float* boxes_xywh, float* scores, int32_t* class_ids, int32_t* cand_index, int32_t* counts,
                     int32_t* n_candidates, int32_t* pts, int32_t* npts, uint8_t* status) {
    NvtxRange nv("adas_detect_pair");
    static int conc = -1;
    if (conc < 0) { const char* c = getenv("ADAS_B200_CONCURRENT"); conc = (c && c[0] == '0') ? 0 : 1; }
    if (!conc || yolo->device != ufld->device) {
        if (adas_yolo_detect(yolo, frames, frames_on_device, batch, H, W, box_score, nms_iou, max_det, boxes_xywh, scores, class_ids, cand_index, counts,
                             n_candidates)) return 1;
        return adas_ufld_detect(ufld, frames, frames_on_device, batch, H, W, pts, npts, status, nullptr);
    }
    // concurrent variant: both networks are enqueued on their own streams before either is waited for, so the tail waves of one
    // network's kernels can be back-filled by the other's
    adas_engine* e = yolo;
    ADAS_CHECK(batch >= 1 && batch <= e->max_batch && batch <= ufld->max_batch, "batch out of range");
    ADAS_CUDA(cudaSetDevice(e->device));
    const int nc = (int)e->hdr.meta[0], A = (int)e->hdr.meta[1];
    if (e->yp.flags == nullptr || e->yp_max_det != max_det) {
        if (e->yp.flags) free_yolo_post(&e->yp);
        if (alloc_yolo_post(&e->yp, e->max_batch, A, max_det)) return 1;
        e->yp_max_det = max_det;
    }
    e->h_ncand.resize(batch);
    if (!frames_on_device) {      // one upload on the object stream; the lane stream waits for it
        const uint8_t* dfr = nullptr;
        if (stage_frames(e, frames, 0, batch, H, W, &dfr)) return 1;
        if (!e->ev_frames) ADAS_CUDA(cudaEventCreateWithFlags(&e->ev_frames, cudaEventDisableTiming));
        ADAS_CUDA(cudaEventRecord(e->ev_frames, e->stream));
        ADAS_CUDA(cudaStreamWaitEvent(ufld->stream, e->ev_frames, 0));
        frames = dfr;
    }
    e->last_dfr = ufld->last_dfr = frames;
    e->last_fb = ufld->last_fb = batch; e->last_fh = ufld->last_fh = H; e->last_fw = ufld->last_fw = W;
    const LetterboxGeom g = letterbox_geom(H, W, (int)e->hdr.in_h, (int)e->hdr.in_w);
    if (launch_yolo_pre(frames, batch, g, static_cast<__half*>(e->dbufs[0].ptr), (int)e->bufs[0].C, nullptr, e->stream)) return 1;
    {
        adas_engine* u = ufld;
        const int in_h = (int)u->hdr.in_h, in_w = (int)u->hdr.in_w;
        const int resize_h = (int)((double)in_h / u->ufld_crop);
        if (launch_ufld_pre(frames, batch, H, W, in_h, in_w, resize_h, u->d_lut, static_cast<__half*>(u->dbufs[0].ptr), (int)u->bufs[0].C, nullptr,
                            u->stream)) return 1;
    }
    if (run_plan(e, batch)) return 1;
    if (run_plan(ufld, batch)) return 1;
    if (head_decode(e, batch)) return 1;
    if (lite_post(e, batch)) return 1;
    if (launch_yolo_post(e->d_raw, (int)e->hdr.model_kind, batch, A, nc, g, box_score, nms_iou, max_det, e->yp, e->stream)) return 1;
    if (copy_yolo_results_enqueue(e->yp, batch, max_det, boxes_xywh, scores, class_ids, cand_index, counts, e->h_ncand.data(), e->stream)) return 1;
    {
        adas_engine* u = ufld;
        const int mp = u->ufld_max_pts;
        if (ufld_post_dispatch(u, batch, W, H, false)) return 1;
        ADAS_CUDA(cudaMemcpyAsync(pts, u->d_pts, (size_t)batch * 4 * mp * 2 * 4, cudaMemcpyDeviceToHost, u->stream));
        ADAS_CUDA(cudaMemcpyAsync(npts, u->d_npts, (size_t)batch * 4 * 4, cudaMemcpyDeviceToHost, u->stream));
        ADAS_CUDA(cudaMemcpyAsync(status, u->d_status, (size_t)batch * 4, cudaMemcpyDeviceToHost, u->stream));
        u->ufld_last_batch = batch;
    }
    if (copy_yolo_results_finish(e->yp, batch, max_det, counts, n_candidates, e->h_ncand.data(), e->stream)) return 1;
    ADAS_CUDA(cudaStreamSynchronize(ufld->stream));
    return 0;
}

int adas_ufld_postprocess(int device, const float* heads_host, int batch, int ngr, int ncr, int ngc, int ncc, int nl, int img_w, int img_h,
                          const double* row_anchor, const double* col_anchor, int32_t* pts, int32_t* npts, uint8_t* status, double* coords_f) {
    ADAS_CUDA(cudaSetDevice(device));
    const size_t total = (size_t)ngr * ncr * nl + (size_t)ngc * ncc * nl + 2 * (size_t)ncr * nl + 2 * (size_t)ncc * nl;
    const int mp = ncr > ncc ? ncr : ncc;
    float* d_h = nullptr; double *d_ra = nullptr, *d_ca = nullptr, *d_co = nullptr; int32_t *d_p = nullptr, *d_n = nullptr; uint8_t* d_s = nullptr;
    ADAS_CUDA(cudaMalloc(&d_h, (size_t)batch * total * 4));
    ADAS_CUDA(cudaMalloc(&d_ra, ncr * 8)); ADAS_CUDA(cudaMalloc(&d_ca, ncc * 8));
    ADAS_CUDA(cudaMalloc(&d_p, (size_t)batch * 4 * mp * 8)); ADAS_CUDA(cudaMalloc(&d_n, (size_t)batch * 16)); ADAS_CUDA(cudaMalloc(&d_s, (size_t)batch * 4));
    ADAS_CUDA(cudaMalloc(&d_co, (size_t)batch * 4 * mp * 8));
    ADAS_CUDA(cudaMemcpy(d_h, heads_host, (size_t)batch * total * 4, cudaMemcpyHostToDevice));
    ADAS_CUDA(cudaMemcpy(d_ra, row_anchor, ncr * 8, cudaMemcpyHostToDevice));
    ADAS_CUDA(cudaMemcpy(d_ca, col_anchor, ncc * 8, cudaMemcpyHostToDevice));
    UfldDims d{ngr, ncr, ngc, ncc, nl};
    int rc = launch_ufld_post(d_h, (int)total, batch, d, img_w, img_h, d_ra, d_ca, d_p, d_n, d_s, d_co, mp, 0);
    if (!rc) {
        cudaError_t ce = cudaMemcpy(pts, d_p, (size_t)batch * 4 * mp * 8, cudaMemcpyDeviceToHost);
        if (ce == cudaSuccess) ce = cudaMemcpy(npts, d_n, (size_t)batch * 16, cudaMemcpyDeviceToHost);
        if (ce == cudaSuccess) ce = cudaMemcpy(status, d_s, (size_t)batch * 4, cudaMemcpyDeviceToHost);
        if (ce == cudaSuccess && coords_f) ce = cudaMemcpy(coords_f, d_co, (size_t)batch * 4 * mp * 8, cudaMemcpyDeviceToHost);
        if (ce != cudaSuccess) { set_error("ufld_postprocess D2H: %s", cudaGetErrorString(ce)); rc = 1; }
    }
    cudaFree(d_h); cudaFree(d_ra); cudaFree(d_ca); cudaFree(d_p); cudaFree(d_n); cudaFree(d_s); cudaFree(d_co);
    return rc;
}

int adas_ufld_v1_postprocess(int device, const float* head_host, int batch, int griding_num, int rows, int in_w, int in_h, int cfg_w, int cfg_h, int img_w,
                             int img_h, const double* row_anchor, int32_t* pts, int32_t* npts, uint8_t* status, double* coords_f) {
    ADAS_CUDA(cudaSetDevice(device));
    const size_t total = (size_t)(griding_num + 1) * rows * 4;
    float* d_h = nullptr; double *d_ra = nullptr, *d_co = nullptr; int32_t *d_p = nullptr, *d_n = nullptr; uint8_t* d_s = nullptr;
    ADAS_CUDA(cudaMalloc(&d_h, (size_t)batch * total * 4)); ADAS_CUDA(cudaMalloc(&d_ra, rows * 8));
    ADAS_CUDA(cudaMalloc(&d_p, (size_t)batch * 4 * rows * 8)); ADAS_CUDA(cudaMalloc(&d_n, (size_t)batch * 16)); ADAS_CUDA(cudaMalloc(&d_s, (size_t)batch * 4));
    ADAS_CUDA(cudaMalloc(&d_co, (size_t)batch * 4 * rows * 8));
    ADAS_CUDA(cudaMemcpy(d_h, head_host, (size_t)batch * total * 4, cudaMemcpyHostToDevice));
    ADAS_CUDA(cudaMemcpy(d_ra, row_anchor, rows * 8, cudaMemcpyHostToDevice));
    int rc = launch_ufld_v1_post(d_h, (int)total, batch, griding_num, rows, in_w, in_h, cfg_w, cfg_h, img_w, img_h, d_ra, d_p, d_n, d_s, d_co, rows, 0);
    if (!rc) {
        cudaError_t ce = cudaMemcpy(pts, d_p, (size_t)batch * 4 * rows * 8, cudaMemcpyDeviceToHost);
        if (ce == cudaSuccess) ce = cudaMemcpy(npts, d_n, (size_t)batch * 16, cudaMemcpyDeviceToHost);
        if (ce == cudaSuccess) ce = cudaMemcpy(status, d_s, (size_t)batch * 4, cudaMemcpyDeviceToHost);
        if (ce == cudaSuccess && coords_f) ce = cudaMemcpy(coords_f, d_co, (size_t)batch * 4 * rows * 8, cudaMemcpyDeviceToHost);
        if (ce != cudaSuccess) { set_error("ufld_v1_postprocess D2H: %s", cudaGetErrorString(ce)); rc = 1; }
    }
    cudaFree(d_h); cudaFree(d_ra); cudaFree(d_p); cudaFree(d_n); cudaFree(d_s); cudaFree(d_co);
    return rc;
}

int adas_ufld_preprocess(int device, const uint8_t* frames_host, int batch, int H, int W, int in_h, int in_w, double crop_ratio, float* blob) {
    ADAS_CUDA(cudaSetDevice(device));
    uint8_t* d_fr = nullptr; float* d_blob = nullptr; float* d_lut = nullptr;
    const size_t fb = (size_t)batch * H * W * 3, bb = (size_t)batch * 3 * in_h * in_w * 4;
    float lut[768];
    ufld_lut_host(lut);
    ADAS_CUDA(cudaMalloc(&d_fr, fb)); ADAS_CUDA(cudaMalloc(&d_blob, bb)); ADAS_CUDA(cudaMalloc(&d_lut, sizeof(lut)));
    ADAS_CUDA(cudaMemcpy(d_fr, frames_host, fb, cudaMemcpyHostToDevice));
    ADAS_CUDA(cudaMemcpy(d_lut, lut, sizeof(lut), cudaMemcpyHostToDevice));
    const int resize_h = (int)((double)in_h / crop_ratio);
    int rc = launch_ufld_pre(d_fr, batch, H, W, in_h, in_w, resize_h, d_lut, nullptr, 0, d_blob, 0);
    if (!rc) { cudaError_t ce = cudaMemcpy(blob, d_blob, bb, cudaMemcpyDeviceToHost); if (ce != cudaSuccess) { set_error("D2H failed: %s", cudaGetErrorString(ce)); rc = 1; } }
    cudaFree(d_fr); cudaFree(d_blob); cudaFree(d_lut);
    return rc;
}

int adas_iou_cost(int device, int problems, const double* a_tlbr, const int32_t* a_off, const double* b_tlbr, const int32_t* b_off,
                  const double* det_scores, int fuse, double* cost, const int64_t* cost_off) {
    if (problems <= 0) return 0;
    ADAS_CUDA(cudaSetDevice(device));
    const int na = a_off[problems], nb = b_off[problems];
    const int64_t ncost = cost_off[problems];
    if (ncost == 0) return 0;
    double *d_a = nullptr, *d_b = nullptr, *d_s = nullptr, *d_c = nullptr; int32_t *d_ao = nullptr, *d_bo = nullptr; int64_t* d_co = nullptr;
    ADAS_CUDA(cudaMalloc(&d_a, (size_t)(na > 0 ? na : 1) * 32)); ADAS_CUDA(cudaMalloc(&d_b, (size_t)(nb > 0 ? nb : 1) * 32));
    ADAS_CUDA(cudaMalloc(&d_s, (size_t)(nb > 0 ? nb : 1) * 8)); ADAS_CUDA(cudaMalloc(&d_c, (size_t)ncost * 8));
    ADAS_CUDA(cudaMalloc(&d_ao, (problems + 1) * 4)); ADAS_CUDA(cudaMalloc(&d_bo, (problems + 1) * 4)); ADAS_CUDA(cudaMalloc(&d_co, (problems + 1) * 8));
    ADAS_CUDA(cudaMemcpy(d_a, a_tlbr, (size_t)na * 32, cudaMemcpyHostToDevice));
    ADAS_CUDA(cudaMemcpy(d_b, b_tlbr, (size_t)nb * 32, cudaMemcpyHostToDevice));
    if (fuse) ADAS_CUDA(cudaMemcpy(d_s, det_scores, (size_t)nb * 8, cudaMemcpyHostToDevice));
    ADAS_CUDA(cudaMemcpy(d_ao, a_off, (problems + 1) * 4, cudaMemcpyHostToDevice));
    ADAS_CUDA(cudaMemcpy(d_bo, b_off, (problems + 1) * 4, cudaMemcpyHostToDevice));
    ADAS_CUDA(cudaMemcpy(d_co, cost_off, (problems + 1) * 8, cudaMemcpyHostToDevice));
    int rc = launch_iou_cost(problems, d_a, d_ao, d_b, d_bo, fuse ? d_s : nullptr, fuse, d_c, d_co, 0);
    if (!rc) { cudaError_t ce = cudaMemcpy(cost, d_c, (size_t)ncost * 8, cudaMemcpyDeviceToHost); if (ce != cudaSuccess) { set_error("iou_cost D2H: %s", cudaGetErrorString(ce)); rc = 1; } }
    cudaFree(d_a); cudaFree(d_b); cudaFree(d_s); cudaFree(d_c); cudaFree(d_ao); cudaFree(d_bo); cudaFree(d_co);
    return rc;
}

int adas_lap(int device, int problems, const double* cost, const int64_t* cost_off, const int32_t* T, const int32_t* D, const double* thresh,
             int32_t* x, const int32_t* x_off, int32_t* y, const int32_t* y_off) {
    if (problems <= 0) return 0;
    ADAS_CUDA(cudaSetDevice(device));
    const int64_t ncost = cost_off[problems];
    const int nx = x_off[problems], ny = y_off[problems];
    for (int i = 0; i < problems; ++i) ADAS_CHECK(T[i] + D[i] <= lap_max_cols() && T[i] <= lap_max_cols() / 2, "adas_lap: problem %d too large (T=%d D=%d)", i, T[i], D[i]);
    double *d_c = nullptr, *d_th = nullptr, *d_v = nullptr, *d_mv = nullptr; int64_t* d_co = nullptr;
    int32_t *d_T = nullptr, *d_D = nullptr, *d_x = nullptr, *d_y = nullptr, *d_xo = nullptr, *d_yo = nullptr, *d_wi = nullptr;
    const size_t wc = (size_t)lap_max_cols() + 1;
    ADAS_CUDA(cudaMalloc(&d_c, (size_t)(ncost > 0 ? ncost : 1) * 8)); ADAS_CUDA(cudaMalloc(&d_th, problems * 8));
    ADAS_CUDA(cudaMalloc(&d_v, problems * wc * 8)); ADAS_CUDA(cudaMalloc(&d_mv, problems * wc * 8)); ADAS_CUDA(cudaMalloc(&d_wi, problems * wc * 12));
    ADAS_CUDA(cudaMalloc(&d_co, (problems + 1) * 8)); ADAS_CUDA(cudaMalloc(&d_T, problems * 4)); ADAS_CUDA(cudaMalloc(&d_D, problems * 4));
    ADAS_CUDA(cudaMalloc(&d_x, (size_t)(nx > 0 ? nx : 1) * 4)); ADAS_CUDA(cudaMalloc(&d_y, (size_t)(ny > 0 ? ny : 1) * 4));
    ADAS_CUDA(cudaMalloc(&d_xo, (problems + 1) * 4)); ADAS_CUDA(cudaMalloc(&d_yo, (problems + 1) * 4));
    ADAS_CUDA(cudaMemcpy(d_c, cost, (size_t)ncost * 8, cudaMemcpyHostToDevice));
    ADAS_CUDA(cudaMemcpy(d_th, thresh, problems * 8, cudaMemcpyHostToDevice));
    ADAS_CUDA(cudaMemcpy(d_co, cost_off, (problems + 1) * 8, cudaMemcpyHostToDevice));
    ADAS_CUDA(cudaMemcpy(d_T, T, problems * 4, cudaMemcpyHostToDevice)); ADAS_CUDA(cudaMemcpy(d_D, D, problems * 4, cudaMemcpyHostToDevice));
    ADAS_CUDA(cudaMemcpy(d_xo, x_off, (problems + 1) * 4, cudaMemcpyHostToDevice)); ADAS_CUDA(cudaMemcpy(d_yo, y_off, (problems + 1) * 4, cudaMemcpyHostToDevice));
    int rc = launch_lap(problems, d_c, d_co, d_T, d_D, d_th, d_x, d_xo, d_y, d_yo, d_v, d_mv, d_wi, 0);
    if (!rc) {
        cudaError_t ce = cudaMemcpy(x, d_x, (size_t)nx * 4, cudaMemcpyDeviceToHost);
        if (ce == cudaSuccess) ce = cudaMemcpy(y, d_y, (size_t)ny * 4, cudaMemcpyDeviceToHost);
        if (ce != cudaSuccess) { set_error("adas_lap D2H: %s", cudaGetErrorString(ce)); rc = 1; }
    }
    cudaFree(d_c); cudaFree(d_th); cudaFree(d_v); cudaFree(d_mv); cudaFree(d_wi); cudaFree(d_co); cudaFree(d_T); cudaFree(d_D);
    cudaFree(d_x); cudaFree(d_y); cudaFree(d_xo); cudaFree(d_yo);
    return rc;
}

int adas_engine_num_buffers(const adas_engine* e, int* n) { *n = (int)e->bufs.size(); return 0; }
int adas_engine_buffer_info(const adas_engine* e, int idx, int64_t info[5]) {
    ADAS_CHECK(idx >= 0 && idx < (int)e->bufs.size(), "bad buffer index %d", idx);
    const PlanBuffer& b = e->bufs[idx];
    info[0] = b.rows_per_img; info[1] = b.C; info[2] = b.dtype; info[3] = b.H; info[4] = b.W;
    return 0;
}
int adas_engine_write_buffer(adas_engine* e, int idx, const void* host, int64_t bytes) {
    ADAS_CHECK(idx >= 0 && idx < (int)e->bufs.size() && (size_t)bytes <= e->dbufs[idx].bytes, "bad buffer write (idx %d, %lld bytes)", idx, (long long)bytes);
    ADAS_CUDA(cudaSetDevice(e->device));
    ADAS_CUDA(cudaMemcpyAsync(e->dbufs[idx].ptr, host, (size_t)bytes, cudaMemcpyHostToDevice, e->stream));
    ADAS_CUDA(cudaStreamSynchronize(e->stream));
    return 0;
}
int adas_engine_read_buffer(adas_engine* e, int idx, void* host, int64_t bytes) {
    ADAS_CHECK(idx >= 0 && idx < (int)e->bufs.size() && (size_t)bytes <= e->dbufs[idx].bytes, "bad buffer read (idx %d, %lld bytes)", idx, (long long)bytes);
    ADAS_CUDA(cudaSetDevice(e->device));
    ADAS_CUDA(cudaMemcpyAsync(host, e->dbufs[idx].ptr, (size_t)bytes, cudaMemcpyDeviceToHost, e->stream));
    ADAS_CUDA(cudaStreamSynchronize(e->stream));
    return 0;
}
int adas_engine_run(adas_engine* e, int batch) {
    ADAS_CHECK(batch >= 1 && batch <= e->max_batch, "batch %d outside [1, %d]", batch, e->max_batch);
    ADAS_CUDA(cudaSetDevice(e->device));
    if (run_plan(e, batch)) return 1;
    ADAS_CUDA(cudaStreamSynchronize(e->stream));
    return 0;
}

int adas_engine_event_record(adas_engine* e, int slot) {
    ADAS_CHECK(e != nullptr && slot >= 0 && slot < 4, "bad event slot");
    ADAS_CUDA(cudaSetDevice(e->device));
    if (e->events[slot] == nullptr) ADAS_CUDA(cudaEventCreate(&e->events[slot]));
    ADAS_CUDA(cudaEventRecord(e->events[slot], e->stream));
    return 0;
}
int adas_event_elapsed_ms(adas_engine* ea, int slot_a, adas_engine* eb, int slot_b, float* ms) {
    ADAS_CHECK(ea && eb && ea->events[slot_a] && eb->events[slot_b], "events not recorded");
    ADAS_CUDA(cudaEventSynchronize(ea->events[slot_a]));
    ADAS_CUDA(cudaEventSynchronize(eb->events[slot_b]));
    ADAS_CUDA(cudaEventElapsedTime(ms, ea->events[slot_a], eb->events[slot_b]));
    return 0;
}
int adas_engine_time_step(adas_engine* e, int batch, int step, int iters, float* ms_per_iter, int* op_type, char* desc, int desc_cap) {
    ADAS_CHECK(e != nullptr && batch >= 1 && batch <= e->max_batch && iters >= 1, "bad arguments");
    ADAS_CUDA(cudaSetDevice(e->device));
    auto it = e->programs.find(batch);
    if (it == e->programs.end()) {
        Program prog;
        if (build_program(e, batch, &prog)) return 1;
        it = e->programs.emplace(batch, std::move(prog)).first;
    }
    Program& pg = it->second;
    ADAS_CHECK(step >= 0 && step < (int)pg.steps.size(), "step %d outside [0, %d)", step, (int)pg.steps.size());
    cudaEvent_t a, b;
    ADAS_CUDA(cudaEventCreate(&a)); ADAS_CUDA(cudaEventCreate(&b));
    if (pg.steps[step](e->stream)) return 1;
    ADAS_CUDA(cudaEventRecord(a, e->stream));
    for (int r = 0; r < iters; ++r) if (pg.steps[step](e->stream)) return 1;
    ADAS_CUDA(cudaEventRecord(b, e->stream));
    ADAS_CUDA(cudaEventSynchronize(b));
    float ms = 0.f;
    ADAS_CUDA(cudaEventElapsedTime(&ms, a, b));
    cudaEventDestroy(a); cudaEventDestroy(b);
    *ms_per_iter = ms / iters;
    if (op_type) *op_type = (int)pg.step_type[step];
    if (desc && desc_cap > 0) {
        const char* d = step < (int)pg.step_desc.size() ? pg.step_desc[step].c_str() : "";
        snprintf(desc, (size_t)desc_cap, "%s", d);
    }
    return 0;
}
int adas_engine_num_steps(adas_engine* e, int batch, int* n) {
    ADAS_CHECK(e != nullptr && batch >= 1 && batch <= e->max_batch, "bad arguments");
    ADAS_CUDA(cudaSetDevice(e->device));
    auto it = e->programs.find(batch);
    if (it == e->programs.end()) {
        Program prog;
        if (build_program(e, batch, &prog)) return 1;
        it = e->programs.emplace(batch, std::move(prog)).first;
    }
    *n = (int)it->second.steps.size();
    return 0;
}
int adas_engine_step_tiles(adas_engine* e, int batch, int step, int cap, int* bn, int* mt, int* n, int* chosen) {
    ADAS_CHECK(e != nullptr && batch >= 1 && batch <= e->max_batch && cap >= 0 && n != nullptr && chosen != nullptr, "bad arguments");
    ADAS_CUDA(cudaSetDevice(e->device));
    auto it = e->programs.find(batch);
    if (it == e->programs.end()) {
        Program prog;
        if (build_program(e, batch, &prog)) return 1;
        it = e->programs.emplace(batch, std::move(prog)).first;
    }
    const Program& pg = it->second;
    ADAS_CHECK(step >= 0 && step < (int)pg.steps.size(), "step %d outside [0, %d)", step, (int)pg.steps.size());
    const std::vector<std::pair<int, int>>& t = pg.step_tiles[step];
    for (int i = 0; i < (int)t.size() && i < cap; ++i) { bn[i] = t[i].first; mt[i] = t[i].second; }
    *n = (int)t.size();
    *chosen = t.empty() ? -1 : pg.step_chosen[step];
    return 0;
}

int adas_engine_time_ops(adas_engine* e, int batch, unsigned type_mask, int iters, float* ms_per_iter, int* launches) {
    ADAS_CHECK(e != nullptr && batch >= 1 && batch <= e->max_batch && iters >= 1, "bad arguments");
    ADAS_CUDA(cudaSetDevice(e->device));
    auto it = e->programs.find(batch);
    if (it == e->programs.end()) {
        Program prog;
        if (build_program(e, batch, &prog)) return 1;
        it = e->programs.emplace(batch, std::move(prog)).first;
    }
    Program& pg = it->second;
    cudaEvent_t a, b;
    ADAS_CUDA(cudaEventCreate(&a)); ADAS_CUDA(cudaEventCreate(&b));
    int n = 0;
    for (int warm = 0; warm < 2; ++warm) {
        if (warm == 1) ADAS_CUDA(cudaEventRecord(a, e->stream));
        const int reps = warm == 0 ? 1 : iters;
        for (int r = 0; r < reps; ++r) {
            n = 0;
            for (size_t i = 0; i < pg.steps.size(); ++i)
                if (pg.step_type[i] != 31 && (type_mask & (1u << pg.step_type[i]))) { if (pg.steps[i](e->stream)) return 1; ++n; }
        }
    }
    ADAS_CUDA(cudaEventRecord(b, e->stream));
    ADAS_CUDA(cudaEventSynchronize(b));
    float ms = 0.f;
    ADAS_CUDA(cudaEventElapsedTime(&ms, a, b));
    cudaEventDestroy(a); cudaEventDestroy(b);
    *ms_per_iter = ms / iters;
    if (launches) *launches = n;
    return 0;
}

// persistent per-thread scratch for the single-problem association path (tracker hot loop)
struct AssocScratch {
    int device = -1; size_t cap_boxes = 0; size_t cap_cost = 0;
    double *d_a = nullptr, *d_b = nullptr, *d_s = nullptr, *d_c = nullptr, *d_th = nullptr, *d_v = nullptr, *d_mv = nullptr;
    int32_t *d_meta = nullptr, *d_x = nullptr, *d_y = nullptr, *d_wi = nullptr; int64_t* d_co = nullptr;
    cudaStream_t st = nullptr;
};
static thread_local AssocScratch g_as;

int adas_associate(int device, int T, int D, const double* a_tlbr, const double* b_tlbr, const double* det_scores, int fuse, double thresh,
                   int32_t* x, int32_t* y, double* cost_out) {
    for (int i = 0; i < T; ++i) x[i] = -1;
    for (int j = 0; j < D; ++j) y[j] = -1;
    if (T == 0 || D == 0) return 0;   // matching.linear_assignment's empty-matrix short circuit (matching.py:21-22)
    ADAS_CHECK(T + D <= lap_max_cols() && T <= lap_max_cols() / 2, "adas_associate: problem too large (T=%d D=%d)", T, D);
    ADAS_CUDA(cudaSetDevice(device));
    AssocScratch& s = g_as;
    const size_t nb = (size_t)(T > D ? T : D), nc = (size_t)T * D;
    if (s.device != device || nb > s.cap_boxes || nc > s.cap_cost) {
        if (s.st == nullptr || s.device != device) { int lo = 0, hi = 0; cudaDeviceGetStreamPriorityRange(&lo, &hi); ADAS_CUDA(cudaStreamCreateWithPriority(&s.st, cudaStreamNonBlocking, hi)); }
        cudaFree(s.d_a); cudaFree(s.d_b); cudaFree(s.d_s); cudaFree(s.d_c); cudaFree(s.d_x); cudaFree(s.d_y);
        s.cap_boxes = nb < 256 ? 256 : nb * 2; s.cap_cost = nc < 65536 ? 65536 : nc * 2;
        ADAS_CUDA(cudaMalloc(&s.d_a, s.cap_boxes * 32)); ADAS_CUDA(cudaMalloc(&s.d_b, s.cap_boxes * 32)); ADAS_CUDA(cudaMalloc(&s.d_s, s.cap_boxes * 8));
        ADAS_CUDA(cudaMalloc(&s.d_c, s.cap_cost * 8)); ADAS_CUDA(cudaMalloc(&s.d_x, s.cap_boxes * 4)); ADAS_CUDA(cudaMalloc(&s.d_y, s.cap_boxes * 4));
        if (s.d_th == nullptr || s.device != device) {
            const size_t wc = (size_t)lap_max_cols() + 1;
            ADAS_CUDA(cudaMalloc(&s.d_th, 8)); ADAS_CUDA(cudaMalloc(&s.d_v, wc * 8)); ADAS_CUDA(cudaMalloc(&s.d_mv, wc * 8)); ADAS_CUDA(cudaMalloc(&s.d_wi, wc * 12));
            ADAS_CUDA(cudaMalloc(&s.d_meta, 8 * 4)); ADAS_CUDA(cudaMalloc(&s.d_co, 2 * 8));
        }
        s.device = device;
    }
    // meta: [a_off0,a_off1,b_off0,b_off1,T,D,x_off0,-]  (x_off/y_off are both {0,..})
    const int32_t meta[8] = {0, T, 0, D, T, D, 0, 0};
    const int64_t co[2] = {0, (int64_t)nc};
    ADAS_CUDA(cudaMemcpyAsync(s.d_meta, meta, sizeof(meta), cudaMemcpyHostToDevice, s.st));
    ADAS_CUDA(cudaMemcpyAsync(s.d_co, co, sizeof(co), cudaMemcpyHostToDevice, s.st));
    ADAS_CUDA(cudaMemcpyAsync(s.d_a, a_tlbr, (size_t)T * 32, cudaMemcpyHostToDevice, s.st));
    ADAS_CUDA(cudaMemcpyAsync(s.d_b, b_tlbr, (size_t)D * 32, cudaMemcpyHostToDevice, s.st));
    if (fuse) ADAS_CUDA(cudaMemcpyAsync(s.d_s, det_scores, (size_t)D * 8, cudaMemcpyHostToDevice, s.st));
    ADAS_CUDA(cudaMemcpyAsync(s.d_th, &thresh, 8, cudaMemcpyHostToDevice, s.st));
    if (launch_iou_cost(1, s.d_a, s.d_meta, s.d_b, s.d_meta + 2, fuse ? s.d_s : nullptr, fuse, s.d_c, s.d_co, s.st)) return 1;
    if (launch_lap(1, s.d_c, s.d_co, s.d_meta + 4, s.d_meta + 5, s.d_th, s.d_x, s.d_meta + 6, s.d_y, s.d_meta + 6, s.d_v, s.d_mv, s.d_wi, s.st)) return 1;
    ADAS_CUDA(cudaMemcpyAsync(x, s.d_x, (size_t)T * 4, cudaMemcpyDeviceToHost, s.st));
    ADAS_CUDA(cudaMemcpyAsync(y, s.d_y, (size_t)D * 4, cudaMemcpyDeviceToHost, s.st));
    if (cost_out) ADAS_CUDA(cudaMemcpyAsync(cost_out, s.d_c, nc * 8, cudaMemcpyDeviceToHost, s.st));
    ADAS_CUDA(cudaStreamSynchronize(s.st));
    return 0;
}

}  // extern "C"
