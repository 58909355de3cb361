// C ABI of libppn_decode (declared in include/ppn_decode.h): argument checking, workspace
// carving, the launch chain of ppn_parse (decode+NMS | limb arg-max -> tree parse), the dense
// entry packing, and the host-memory entry with overlapped copies.
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <mutex>

#include "ppn_decode.h"
#include "ppn_decode_bench.h"
#include "ppn_kernels.h"

namespace {

// Tuning table (ppn_tune, declared in include/ppn_decode_bench.h).  Written under a lock; every entry point takes
// ONE snapshot when it starts (a local named g_tuning), so a call never sees a half-updated table and concurrent
// calls on other threads are unaffected by a writer.
ppn::Tuning g_tuning_shared;
std::mutex g_tune_mu;
ppn::Tuning tuning_now() {
    std::lock_guard<std::mutex> lock(g_tune_mu);
    return g_tuning_shared;
}

// ---- optional per-stage timing of ppn_parse (ppn_profile_*) --------------------------------
// When enabled, ppn_parse runs its kernels back to back and brackets each with a (start, stop)
// pair of CUDA events on the caller's stream; ppn_profile_read() sums the elapsed times.  Used by
// bench.py for the per-kernel durations behind `roofline`.  Not thread-safe: one thread only.
constexpr int kStages = 4;
constexpr int kMaxProfiled = 4096;
struct Profile {
    bool on = false;
    int used = 0;
    cudaEvent_t* ev = nullptr;          // [kMaxProfiled][2 * kStages]: (start, stop) per stage
} g_prof;

inline cudaEvent_t* profile_slot() {
    if (!g_prof.on || g_prof.used >= kMaxProfiled) return nullptr;
    return g_prof.ev + (size_t)(g_prof.used++) * (2 * kStages);
}

// ---- side lane: decode + NMS run beside the limb arg-max ---------------------------------
// parse.overlap = 1 (the alternative to the default PDL chain): decode+NMS is forked onto a private
// non-blocking stream and joined before the tree parse.  One lane per host thread and device;
// event record/wait pairs are also legal under stream capture (CUDA graphs).
struct SideLane {
    cudaStream_t stream = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
};
thread_local SideLane t_side[64];

cudaError_t side_lane(SideLane** out) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
    SideLane& l = t_side[dev];
    if (!l.stream) {
        if ((e = cudaStreamCreateWithFlags(&l.stream, cudaStreamNonBlocking)) != cudaSuccess) return e;
        if ((e = cudaEventCreateWithFlags(&l.fork, cudaEventDisableTiming)) != cudaSuccess) return e;
        if ((e = cudaEventCreateWithFlags(&l.join, cudaEventDisableTiming)) != cudaSuccess) return e;
    }
    *out = &l;
    return cudaSuccess;
}

inline int cuda_rc(cudaError_t e) { return e == cudaSuccess ? PPN_OK : (int)e; }

// ---- optional device timeline of ppn_parse's kernels (ppn_timeline, include/ppn_decode_bench.h) ------------
// Every kernel of a call gets one 4 x uint64 record {first CTA start, last CTA end, first CTA past its dependency
// wait, kind} in %globaltimer nanoseconds, written with atomicMin / atomicMax.  One benchmark thread.
struct Timeline { unsigned long long* buf = nullptr; int cap = 0, used = 0, phase = 0; } g_timeline;
inline ppn::Geom timeline_slot(ppn::Geom g) {
    if (g_timeline.buf && g_timeline.used < g_timeline.cap) { g.tl = g_timeline.buf; g.tl_slot = g_timeline.used++; g.tl_phase = g_timeline.phase; }
    else g.tl = nullptr;
    return g;
}

int check_shape(const PPNShape* s) {
    if (!s) return PPN_E_BADARG;
    if (s->B < 0 || s->K < 1 || s->E < 0 || s->H < 1 || s->W < 1 || s->sH < 1 || s->sW < 1) return PPN_E_BADARG;
    if (s->inW < 1 || s->inH < 1 || s->gridW < 0 || s->gridH < 0) return PPN_E_BADARG;   // gridW/H = int(in/out) may be 0 for the parser
    if ((long long)s->sH * s->sW > 65535) return PPN_E_UNSUPPORTED;            // arg-max map is uint16
    if (s->K > 255 || s->E > 255) return PPN_E_UNSUPPORTED;                    // chain tables are uint8
    const long long per_img = ((long long)6 * s->K + (long long)s->sH * s->sW * s->E) * s->H * s->W;
    if (per_img > 0x7fffffffLL) return PPN_E_UNSUPPORTED;
    if (s->head_dtype < PPN_HEAD_F32 || s->head_dtype > PPN_HEAD_BF16) return PPN_E_BADARG;
    return PPN_OK;
}

ppn::Geom make_geom(const PPNShape* s) {
    ppn::Geom g;
    g.B = s->B; g.K = s->K; g.E = s->E; g.H = s->H; g.W = s->W; g.HW = s->H * s->W;
    g.sH = s->sH; g.sW = s->sW; g.S = s->sH * s->sW; g.C = 6 * s->K + g.S * s->E;
    g.off_h = s->off_h; g.off_w = s->off_w;
    g.gridW = (float)s->gridW; g.gridH = (float)s->gridH; g.inW = (float)s->inW; g.inH = (float)s->inH;
    g.img_stride = (size_t)g.C * g.HW;
    g.limb_off = (size_t)6 * g.K * g.HW;
    g.tl = nullptr;
    g.tl_slot = 0;
    g.tl_phase = 0;
    auto magic = [](int d) -> uint32_t { return d <= 1 ? 0u : (uint32_t)(((1ull << 32) + d - 1) / d); };
    g.magic_W = magic(g.W);
    g.magic_K = magic(g.K);
    g.dtype = s->head_dtype;
    return g;
}

int make_chains(const PPNShape* s, const PPNParams* p, ppn::ChainTable* ch) {
    if (!p) return PPN_E_BADARG;
    if (p->n_chains < 0 || p->n_chains > PPN_MAX_CHAINS) return PPN_E_CHAINS;
    if (p->n_chains > 0 && (!p->chain_off || !p->chain_limb || !p->chain_part)) return PPN_E_BADARG;
    std::memset(ch, 0, sizeof(*ch));
    ch->n_chains = p->n_chains;
    if (p->n_chains == 0) return PPN_OK;
    if (p->chain_off[0] != 0) return PPN_E_CHAINS;
    for (int c = 0; c < p->n_chains; ++c)
        if (p->chain_off[c + 1] < p->chain_off[c]) return PPN_E_CHAINS;
    const int total = p->chain_off[p->n_chains];
    if (total > PPN_MAX_CHAIN_STEPS) return PPN_E_CHAINS;
    for (int c = 0; c <= p->n_chains; ++c) ch->off[c] = (uint8_t)p->chain_off[c];
    for (int q = 0; q < total; ++q) {
        if (p->chain_limb[q] < 0 || p->chain_limb[q] >= s->E || p->chain_part[q] < 0 || p->chain_part[q] >= s->K)
            return PPN_E_CHAINS;
        ch->limb[q] = (uint8_t)p->chain_limb[q];
        ch->part[q] = (uint8_t)p->chain_part[q];
    }
    // Do the track orders form a tree?  Then a part's cell does not depend on which chain reaches
    // it, and the kernel may walk the chains of one root concurrently (config.py:67-80 does).
    int limb_of[256], pred_of[256];
    for (int t = 0; t < 256; ++t) limb_of[t] = pred_of[t] = -1;
    ch->parallel_ok = 1;
    for (int c = 0; c < p->n_chains && ch->parallel_ok; ++c)
        for (int q = p->chain_off[c]; q < p->chain_off[c + 1]; ++q) {
            const int t = p->chain_part[q], e = p->chain_limb[q];
            const int pred = q == p->chain_off[c] ? 0 : p->chain_part[q - 1];
            if (t == 0) { ch->parallel_ok = 0; break; }
            if (limb_of[t] < 0) { limb_of[t] = e; pred_of[t] = pred; }
            else if (limb_of[t] != e || pred_of[t] != pred) { ch->parallel_ok = 0; break; }
        }
    return PPN_OK;
}

inline size_t elem_bytes(const PPNShape* s) { return s->head_dtype == PPN_HEAD_F32 ? 4 : 2; }
inline bool misaligned(const void* p, const PPNShape* s) { return (reinterpret_cast<uintptr_t>(p) & (elem_bytes(s) - 1)) != 0; }

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Workspace layout of ppn_parse (arg-max map, surviving root cells per (image, part), their
// counts), every block 256-byte aligned.
struct Workspace {
    size_t amax, keep_idx, keep_count, total;
};

Workspace carve(const PPNShape* s, int n_parts) {
    Workspace w;
    const size_t B = (size_t)s->B, HW = (size_t)s->H * s->W, P = (size_t)n_parts;
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t at = off; off = align_up(off + bytes, 256); return at; };
    w.amax = take(B * s->E * HW * sizeof(uint16_t));
    w.keep_idx = take(B * P * HW * sizeof(int32_t));
    w.keep_count = take(B * P * sizeof(int32_t));
    w.total = off;
    return w;
}

// ppn_parse alternates between the two halves of the caller's workspace from call to call on a stream
// (ppn::next_call_parity), so that a call may overlap the previous one (PPN_FLAG_INPUT_COMPLETE) without
// sharing scratch with it.

int check_params(const PPNShape* s, const PPNParams* p) {
    if (!p) return PPN_E_BADARG;
    if (p->n_nms_parts < 1 || p->n_nms_parts > s->K) return PPN_E_BADARG;
    return PPN_OK;
}

int check_humans(const PPNHumans* h) {
    if (!h || !h->count || !h->root_cell || !h->part_cell || !h->part_score || !h->part_box || h->R < 1) return PPN_E_BADARG;
    return PPN_OK;
}

}  // namespace

// ---- dense pose entries ----------------------------------------------------------------------
namespace {
struct PackedLayout { size_t header, idcell, score, box, total; };
PackedLayout packed_layout(int B, int cap) {
    PackedLayout l;
    l.header = 0;
    l.idcell = align_up((size_t)(2 + 3 * (size_t)B) * sizeof(int32_t), 256);
    l.score = l.idcell + align_up((size_t)cap * sizeof(uint32_t), 256);
    l.box = l.score + align_up((size_t)cap * sizeof(float), 256);
    l.total = l.box + align_up((size_t)cap * 4 * sizeof(float), 256);
    return l;
}
}  // namespace

namespace {
// dense entries from the fixed-stride result (paths on which the fused kernel did not write them)
int pack_after(const PPNHumans* out, const PPNShape* shape, const ppn::DenseTarget* d, cudaStream_t st) {
    if (out->R > 65536) return PPN_E_UNSUPPORTED;
    return cuda_rc(ppn::launch_pack_humans(out->count, out->part_cell, out->part_score, out->part_box, shape->B, out->R,
                                           shape->K, d->cap, d->header, d->idcell, d->score, d->box, st));
}
}  // namespace

extern "C" {

int ppn_abi_version(void) { return PPN_ABI_VERSION; }

const char* ppn_strerror(int code) {
    switch (code) {
        case PPN_OK: return "ok";
        case PPN_E_BADARG: return "ppn: bad argument (null pointer, non-positive size or misaligned base)";
        case PPN_E_UNSUPPORTED: return "ppn: shape not supported by the kernels";
        case PPN_E_WORKSPACE: return "ppn: workspace smaller than ppn_workspace_bytes()";
        case PPN_E_CHAINS: return "ppn: track orders too long or indexing outside K/E";
        case PPN_E_NO_DEVICE: return "ppn: no usable CUDA device";
        default: break;
    }
    if (code > 0) return cudaGetErrorString((cudaError_t)code);
    return "ppn: unknown error";
}

int ppn_tune(const char* key, int32_t value) {
    if (!key) return PPN_E_BADARG;
    std::lock_guard<std::mutex> lock(g_tune_mu);
    ppn::Tuning& t = g_tuning_shared;
    if (!std::strcmp(key, "argmax.variant")) t.argmax_variant = value;
    else if (!std::strcmp(key, "argmax.stage_bytes")) t.argmax_stage_bytes = value <= 0 ? 0 : (value < 1024 ? 1024 : value);
    else if (!std::strcmp(key, "argmax.stages")) t.argmax_stages = value < 2 ? 2 : (value > 32 ? 32 : value);
    else if (!std::strcmp(key, "argmax.threads")) t.argmax_threads = value < 32 ? 32 : (value > 992 ? 992 : value);
    else if (!std::strcmp(key, "argmax.ctas_per_sm")) t.argmax_ctas_per_sm = value < 1 ? 1 : (value > 8 ? 8 : value);
    else if (!std::strcmp(key, "argmax.split")) t.argmax_split = value;
    else if (!std::strcmp(key, "argmax.cluster")) t.argmax_cluster = value;
    else if (!std::strcmp(key, "argmax.cluster_ring")) t.argmax_cluster_ring = value != 0;
    else if (!std::strcmp(key, "argmax.smem_cap")) t.argmax_smem_cap = value < 0 ? 0 : value;
    else if (!std::strcmp(key, "parse.overlap")) t.parse_overlap = value < 0 ? 0 : (value > 2 ? 2 : value);
    else if (!std::strcmp(key, "argmax.tail_opt")) t.argmax_tail_opt = value < 0 ? 0 : (value > 8 ? 8 : value);
    else if (!std::strcmp(key, "argmax16.threads")) t.argmax16_threads = value < 32 ? 32 : (value > 992 ? 992 : value);
    else if (!std::strcmp(key, "argmax16.stage_bytes")) t.argmax16_stage_bytes = value < 1024 ? 1024 : value;
    else if (!std::strcmp(key, "argmax.dynamic")) t.argmax_dynamic = value != 0;
    else if (!std::strcmp(key, "parse.stage_all")) t.parse_stage_all = value;
    else if (!std::strcmp(key, "parse.chain_calls")) t.parse_chain_calls = value != 0;
    else if (!std::strcmp(key, "parse.persist")) t.parse_persist = value < 0 ? 0 : (value > 4 ? 4 : value);
    else if (!std::strcmp(key, "parse.k12_threads")) t.parse_k12_threads = value < 0 ? 0 : value;
    else if (!std::strcmp(key, "parse.fused")) t.parse_fused = value < 0 ? -1 : (value != 0);
    else if (!std::strcmp(key, "parse.threads")) t.parse_threads = value;
    else if (!std::strcmp(key, "head.subs")) t.head_subs = (t.head_subs & 0x1300) | (value < 1 ? 0 : (value > 7 ? 7 : value));   // 0 = auto
    else if (!std::strcmp(key, "head.dry")) t.head_subs = (t.head_subs & 0x10ff) | ((value & 3) << 8);   // benchmarks: epilogue skipped, results invalid
    else if (!std::strcmp(key, "head.acc")) t.head_subs = (t.head_subs & 0x3ff) | (value == 128 ? 0x1000 : 0);   // 16-bit path: 128 = four accumulators of 128 channels (default two of 256)
    else if (!std::strcmp(key, "host.chunk_images")) t.host_chunk_images = value < 1 ? 1 : value;
    else if (!std::strcmp(key, "encode.sweep")) t.encode_sweep = value != 0;
    else if (!std::strcmp(key, "encode.ctas_per_sm")) t.encode_ctas_per_sm = value < 1 ? 1 : (value > 8 ? 8 : value);
    else if (!std::strcmp(key, "nms.blockwise")) ppn::set_nms_blockwise(value);   // NMS phase 3 block by block (round 1/2) instead of the warp wavefront
    else if (!std::strcmp(key, "timeline.phase")) g_timeline.phase = value;      // which in-kernel phase boundary ppn_timeline records
    else return PPN_E_BADARG;
    return PPN_OK;
}

int ppn_tune_get(const char* key, int32_t* value) {
    if (!key || !value) return PPN_E_BADARG;
    const ppn::Tuning t = tuning_now();
    if (!std::strcmp(key, "argmax.variant")) *value = t.argmax_variant;
    else if (!std::strcmp(key, "argmax.stage_bytes")) *value = t.argmax_stage_bytes;
    else if (!std::strcmp(key, "argmax.stages")) *value = t.argmax_stages;
    else if (!std::strcmp(key, "argmax.threads")) *value = t.argmax_threads;
    else if (!std::strcmp(key, "argmax.ctas_per_sm")) *value = t.argmax_ctas_per_sm;
    else if (!std::strcmp(key, "argmax.split")) *value = t.argmax_split;
    else if (!std::strcmp(key, "argmax.cluster")) *value = t.argmax_cluster;
    else if (!std::strcmp(key, "argmax.cluster_ring")) *value = t.argmax_cluster_ring;
    else if (!std::strcmp(key, "argmax.smem_cap")) *value = t.argmax_smem_cap;
    else if (!std::strcmp(key, "parse.overlap")) *value = t.parse_overlap;
    else if (!std::strcmp(key, "argmax.tail_opt")) *value = t.argmax_tail_opt;
    else if (!std::strcmp(key, "argmax16.threads")) *value = t.argmax16_threads;
    else if (!std::strcmp(key, "argmax16.stage_bytes")) *value = t.argmax16_stage_bytes;
    else if (!std::strcmp(key, "argmax.dynamic")) *value = t.argmax_dynamic;
    else if (!std::strcmp(key, "parse.stage_all")) *value = t.parse_stage_all;
    else if (!std::strcmp(key, "parse.chain_calls")) *value = t.parse_chain_calls;
    else if (!std::strcmp(key, "parse.persist")) *value = t.parse_persist;
    else if (!std::strcmp(key, "parse.k12_threads")) *value = t.parse_k12_threads;
    else if (!std::strcmp(key, "parse.fused")) *value = t.parse_fused;
    else if (!std::strcmp(key, "parse.threads")) *value = t.parse_threads;
    else if (!std::strcmp(key, "host.chunk_images")) *value = t.host_chunk_images;
    else if (!std::strcmp(key, "encode.sweep")) *value = t.encode_sweep;
    else if (!std::strcmp(key, "encode.ctas_per_sm")) *value = t.encode_ctas_per_sm;
    else if (!std::strcmp(key, "nms.blockwise")) *value = ppn::get_nms_blockwise();
    else return PPN_E_BADARG;
    return PPN_OK;
}

int ppn_workspace_bytes(const PPNShape* shape, const PPNParams* params, size_t* bytes) {
    int rc = check_shape(shape);
    if (rc) return rc;
    if ((rc = check_params(shape, params))) return rc;
    if (!bytes) return PPN_E_BADARG;
    *bytes = 2 * carve(shape, params->n_nms_parts).total;         // two sets, used alternately
    return PPN_OK;
}

int ppn_parse_launches(const PPNShape* shape, const PPNParams* params) {
    const ppn::Tuning g_tuning = tuning_now();
    if (check_shape(shape) || check_params(shape, params)) return 0;
    if (shape->B <= 0) return 0;
    const ppn::Geom g = make_geom(shape);
    ppn::FusedSplit split;
    const bool P1 = params->n_nms_parts == 1 && g_tuning.parse_overlap != 1;
    const bool fits = P1 && ppn::parse_fused_split(g, g_tuning.parse_stage_all, g_tuning, &split);
    const bool fused = P1 && (g_tuning.parse_fused < 0 ? (fits && split.n_sub == 1) : (g_tuning.parse_fused != 0 && ppn::parse_fused_supported(g, g_tuning.parse_stage_all)));
    if (fused) return 2 * (fits ? split.n_sub : 1);
    return 3;
}

int ppn_parse_plan(const PPNShape* shape, const PPNParams* params, int32_t* info) {
    const ppn::Tuning g_tuning = tuning_now();
    if (!info) return PPN_E_BADARG;
    int rc = check_shape(shape);
    if (rc) return rc;
    if ((rc = check_params(shape, params))) return rc;
    info[0] = ppn_parse_launches(shape, params);
    info[1] = 1; info[2] = 0; info[3] = 0;
    if (shape->B <= 0) return PPN_OK;
    ppn::FusedSplit split;
    if (params->n_nms_parts == 1 && ppn::parse_fused_split(make_geom(shape), g_tuning.parse_stage_all, g_tuning, &split)) {
        info[1] = split.n_sub;
        info[2] = (int32_t)split.ring_cap;
        info[3] = split.staged ? 1 : 0;
    }
    return PPN_OK;
}

int ppn_limb_argmax(const void* head, const PPNShape* shape, uint16_t* amax, void* stream) {
    const ppn::Tuning g_tuning = tuning_now();
    int rc = check_shape(shape);
    if (rc) return rc;
    if (shape->B == 0 || shape->E == 0) return PPN_OK;
    if (!head || !amax) return PPN_E_BADARG;
    if (misaligned(head, shape)) return PPN_E_BADARG;
    return cuda_rc(ppn::launch_limb_argmax(head, amax, make_geom(shape), g_tuning, (cudaStream_t)stream));
}

int ppn_limb_stream_probe(const void* head, const PPNShape* shape, uint16_t* amax, int32_t smem_cap, void* stream) {
    const ppn::Tuning g_tuning = tuning_now();
    int rc = check_shape(shape);
    if (rc) return rc;
    if (shape->B == 0 || shape->E == 0) return PPN_OK;
    if (!head || !amax) return PPN_E_BADARG;
    if (misaligned(head, shape)) return PPN_E_BADARG;
    ppn::Tuning t = g_tuning;
    t.argmax_dry = 1;
    t.argmax_cluster = 0;                              // the ring kernels are what is being probed
    if (smem_cap > 0) t.argmax_smem_cap = smem_cap;
    return cuda_rc(ppn::launch_limb_argmax(head, amax, make_geom(shape), t, (cudaStream_t)stream));
}

int ppn_decode_candidates(const void* head, const PPNShape* shape, int32_t n_parts, float det_thresh,
                          int32_t* cand_cell, float* cand_score, float* cand_box, int32_t* cand_count, void* stream) {
    int rc = check_shape(shape);
    if (rc) return rc;
    if (n_parts < 1 || n_parts > shape->K) return PPN_E_BADARG;
    if (shape->B == 0) return PPN_OK;
    if (!head || !cand_cell || !cand_score || !cand_box || !cand_count) return PPN_E_BADARG;
    if (reinterpret_cast<uintptr_t>(cand_box) & 15) return PPN_E_BADARG;
    return cuda_rc(ppn::launch_decode_candidates(head, make_geom(shape), n_parts, det_thresh, cand_cell, cand_score,
                                                 cand_box, cand_count, (cudaStream_t)stream));
}

int ppn_restore_xy(const float* x, const float* y, float* rx, float* ry, int64_t n_planes, const PPNShape* shape, void* stream) {
    int rc = check_shape(shape);
    if (rc) return rc;
    if (n_planes < 0) return PPN_E_BADARG;
    if (n_planes == 0) return PPN_OK;
    if (!x || !y || !rx || !ry) return PPN_E_BADARG;
    return cuda_rc(ppn::launch_restore_xy(x, y, rx, ry, (size_t)n_planes * shape->H * shape->W, shape->H, shape->W,
                                          (float)shape->gridW, (float)shape->gridH, (cudaStream_t)stream));
}

int ppn_restore_size(const float* w, const float* h, float* rw, float* rh, int64_t n_planes, const PPNShape* shape, void* stream) {
    int rc = check_shape(shape);
    if (rc) return rc;
    if (n_planes < 0) return PPN_E_BADARG;
    if (n_planes == 0) return PPN_OK;
    if (!w || !h || !rw || !rh) return PPN_E_BADARG;
    return cuda_rc(ppn::launch_restore_size(w, h, rw, rh, (size_t)n_planes * shape->H * shape->W, (float)shape->inW,
                                            (float)shape->inH, (cudaStream_t)stream));
}

int ppn_nms(const float* box, const float* score, const int32_t* count, int32_t n_problems, int32_t stride,
            float nms_thresh, int32_t limit, int32_t* keep_idx, int32_t* keep_count, void* stream) {
    if (n_problems < 0 || stride < 1) return PPN_E_BADARG;
    if (n_problems == 0) return PPN_OK;
    if (!box || !count || !keep_idx || !keep_count) return PPN_E_BADARG;
    if (reinterpret_cast<uintptr_t>(box) & 15) return PPN_E_BADARG;
    return cuda_rc(ppn::launch_nms(box, score, count, n_problems, stride, nms_thresh, limit, keep_idx, keep_count,
                                   (cudaStream_t)stream));
}

int ppn_tree_parse(const void* head, const PPNShape* shape, const PPNParams* params, const uint16_t* amax,
                   const int32_t* cand_cell, const int32_t* keep_idx, const int32_t* keep_count,
                   const PPNHumans* out, void* stream) {
    int rc = check_shape(shape);
    if (rc) return rc;
    if ((rc = check_params(shape, params))) return rc;
    if ((rc = check_humans(out))) return rc;
    ppn::ChainTable ch;
    if ((rc = make_chains(shape, params, &ch))) return rc;
    if (shape->B == 0) return PPN_OK;
    if (!head || !keep_idx || !keep_count || (!amax && shape->E > 0)) return PPN_E_BADARG;   // cand_cell may be NULL
    if ((long long)shape->H * shape->W > PPN_MAX_CELLS) return PPN_E_UNSUPPORTED;
    if (reinterpret_cast<uintptr_t>(out->part_box) & 15) return PPN_E_BADARG;
    return cuda_rc(ppn::launch_tree_parse(head, make_geom(shape), ch, params->det_thresh, params->min_num_keypoints,
                                          params->n_nms_parts, amax, cand_cell, keep_idx, keep_count, out->count,
                                          out->root_cell, out->part_cell, out->part_score, out->part_box, out->R,
                                          (cudaStream_t)stream));
}

// ---- landing flags of the peer gather: a counter per rank in the ROOT's memory -----------------------------
namespace {
// One thread; launched WITHOUT the programmatic attribute, so every kernel before it in the stream (the parse
// kernels whose stores crossed NVLink) has completed and its writes are performed before the flag is released.
__global__ void peer_post_kernel(long long* counter, long long value) {
    __threadfence_system();
    asm volatile("st.release.sys.global.u64 [%0], %1;" :: "l"(counter), "l"(value) : "memory");
}
// Lane r polls counter r until it has reached `target`; gives up after timeout_ns (a dead peer must not hang the
// stream) and then raises *timed_out.
__global__ void peer_wait_kernel(const long long* counters, int n, long long target, unsigned long long timeout_ns, int* timed_out) {
    const int r = threadIdx.x;
    if (r >= n) return;
    unsigned long long t0, t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (;;) {
        long long v;
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(counters + r) : "memory");
        if (v >= target) return;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        if (t - t0 > timeout_ns) { if (timed_out) *timed_out = 1; return; }
        __nanosleep(200);
    }
}
}  // namespace

int ppn_peer_post(void* counter, long long value, void* stream) {
    if (!counter || (reinterpret_cast<uintptr_t>(counter) & 7)) return PPN_E_BADARG;
    peer_post_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(static_cast<long long*>(counter), value);
    return cuda_rc(cudaGetLastError());
}

int ppn_peer_wait(const void* counters, int32_t n, long long target, uint32_t timeout_ms, int32_t* timed_out, void* stream) {
    if (!counters || n < 1 || n > 1024 || (reinterpret_cast<uintptr_t>(counters) & 7)) return PPN_E_BADARG;
    peer_wait_kernel<<<1, (n + 31) / 32 * 32, 0, (cudaStream_t)stream>>>(static_cast<const long long*>(counters), n, target,
                                                                      (unsigned long long)timeout_ms * 1000000ull, timed_out);
    return cuda_rc(cudaGetLastError());
}

static int parse_impl(const void* head, const PPNShape* shape, const PPNParams* params, const PPNHumans* out,
                      void* workspace, size_t workspace_bytes, void* stream, const ppn::DenseTarget* dense);

int ppn_parse(const void* head, const PPNShape* shape, const PPNParams* params, const PPNHumans* out,
              void* workspace, size_t workspace_bytes, void* stream) {
    return parse_impl(head, shape, params, out, workspace, workspace_bytes, stream, nullptr);
}

int ppn_parse_dense(const void* head, const PPNShape* shape, const PPNParams* params, const PPNHumans* out,
                    void* packed, size_t packed_bytes, int32_t cap_entries, int32_t skip_slots,
                    void* workspace, size_t workspace_bytes, void* stream) {
    int rc = check_shape(shape);
    if (rc) return rc;
    if (cap_entries < 0) return PPN_E_BADARG;
    if (shape->K > 65535 || (long long)shape->H * shape->W > 65536) return PPN_E_UNSUPPORTED;   // part id and cell share 32 bits
    if (shape->B == 0) return PPN_OK;
    if (!packed || (reinterpret_cast<uintptr_t>(packed) & 255)) return PPN_E_BADARG;
    const PackedLayout l = packed_layout(shape->B, cap_entries);
    if (packed_bytes < l.total) return PPN_E_WORKSPACE;
    unsigned char* p = static_cast<unsigned char*>(packed);
    ppn::DenseTarget d;
    d.header = reinterpret_cast<int32_t*>(p + l.header);
    d.idcell = reinterpret_cast<uint32_t*>(p + l.idcell);
    d.score = reinterpret_cast<float*>(p + l.score);
    d.box = reinterpret_cast<float*>(p + l.box);
    d.cap = cap_entries;
    d.skip_slots = skip_slots != 0;
    return parse_impl(head, shape, params, out, workspace, workspace_bytes, stream, &d);
}

int ppn_parse_dense_remote(const void* head, const PPNShape* shape, const PPNParams* params, const PPNHumans* out,
                           void* local_header, size_t local_header_bytes, void* remote_packed, size_t remote_bytes,
                           int32_t cap_entries, int32_t skip_slots, void* workspace, size_t workspace_bytes, void* stream) {
    int rc = check_shape(shape);
    if (rc) return rc;
    if (cap_entries < 0) return PPN_E_BADARG;
    if (shape->K > 32 || (long long)shape->H * shape->W > PPN_MAX_CELLS) return PPN_E_UNSUPPORTED;
    if (shape->B == 0) return PPN_OK;
    if (!local_header || !remote_packed || (reinterpret_cast<uintptr_t>(local_header) & 255) ||
        (reinterpret_cast<uintptr_t>(remote_packed) & 255)) return PPN_E_BADARG;
    const PackedLayout l = packed_layout(shape->B, cap_entries);
    if (remote_bytes < l.total || local_header_bytes < (size_t)(2 + 3 * (size_t)shape->B) * sizeof(int32_t)) return PPN_E_WORKSPACE;
    unsigned char* p = static_cast<unsigned char*>(remote_packed);
    ppn::DenseTarget d;
    d.header = static_cast<int32_t*>(local_header);
    d.rheader = reinterpret_cast<int32_t*>(p + l.header);
    d.idcell = reinterpret_cast<uint32_t*>(p + l.idcell);
    d.score = reinterpret_cast<float*>(p + l.score);
    d.box = reinterpret_cast<float*>(p + l.box);
    d.cap = cap_entries;
    d.skip_slots = skip_slots != 0;
    return parse_impl(head, shape, params, out, workspace, workspace_bytes, stream, &d);
}

int ppn_peer_alloc(size_t bytes, void** dev_ptr, unsigned char* handle) {
    if (!dev_ptr || !handle || bytes == 0) return PPN_E_BADARG;
    static_assert(sizeof(cudaIpcMemHandle_t) == PPN_IPC_HANDLE_BYTES, "IPC handle size");
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) return (int)e;
    if ((e = cudaMemset(p, 0, bytes)) != cudaSuccess) { cudaFree(p); return (int)e; }
    cudaIpcMemHandle_t h;
    if ((e = cudaIpcGetMemHandle(&h, p)) != cudaSuccess) { cudaFree(p); return (int)e; }
    std::memcpy(handle, &h, sizeof(h));
    *dev_ptr = p;
    return PPN_OK;
}

int ppn_peer_open(const unsigned char* handle, void** dev_ptr) {
    if (!dev_ptr || !handle) return PPN_E_BADARG;
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, sizeof(h));
    return cuda_rc(cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
}

int ppn_peer_close(void* dev_ptr) { return dev_ptr ? cuda_rc(cudaIpcCloseMemHandle(dev_ptr)) : PPN_E_BADARG; }
int ppn_peer_free(void* dev_ptr) { return dev_ptr ? cuda_rc(cudaFree(dev_ptr)) : PPN_E_BADARG; }

int ppn_peer_copy(void* dst, const void* src, size_t bytes, void* stream) {
    if (!dst || !src) return PPN_E_BADARG;
    if (bytes == 0) return PPN_OK;
    return cuda_rc(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, (cudaStream_t)stream));
}

static int parse_impl(const void* head, const PPNShape* shape, const PPNParams* params, const PPNHumans* out,
                      void* workspace, size_t workspace_bytes, void* stream, const ppn::DenseTarget* dense) {
    const ppn::Tuning g_tuning = tuning_now();
    int rc = check_shape(shape);
    if (rc) return rc;
    if ((rc = check_params(shape, params))) return rc;
    if ((rc = check_humans(out))) return rc;
    ppn::ChainTable ch;
    if ((rc = make_chains(shape, params, &ch))) return rc;
    if (shape->B == 0) return PPN_OK;
    if (!head || !workspace) return PPN_E_BADARG;
    if (misaligned(head, shape) || (reinterpret_cast<uintptr_t>(workspace) & 255)) return PPN_E_BADARG;
    if ((long long)shape->H * shape->W > PPN_MAX_CELLS) return PPN_E_UNSUPPORTED;
    if (reinterpret_cast<uintptr_t>(out->part_box) & 15) return PPN_E_BADARG;
    const int P = params->n_nms_parts;
    const Workspace w = carve(shape, P);
    if (workspace_bytes < 2 * w.total) return PPN_E_WORKSPACE;
    unsigned char* ws = static_cast<unsigned char*>(workspace) + (ppn::next_call_parity((cudaStream_t)stream) ? w.total : 0);
    uint16_t* amax = reinterpret_cast<uint16_t*>(ws + w.amax);
    int32_t* keep_idx = reinterpret_cast<int32_t*>(ws + w.keep_idx);
    int32_t* keep_count = reinterpret_cast<int32_t*>(ws + w.keep_count);
    const ppn::Geom g = make_geom(shape);
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e;
    if ((params->flags & PPN_FLAG_CLEAR_UNUSED) && !(dense && dense->skip_slots)) {
        const size_t slots = (size_t)shape->B * out->R, SK = slots * shape->K;
        if ((e = cudaMemsetAsync(out->root_cell, 0xFF, slots * sizeof(int32_t), st)) != cudaSuccess) return (int)e;
        if ((e = cudaMemsetAsync(out->part_cell, 0xFF, SK * sizeof(int32_t), st)) != cudaSuccess) return (int)e;
        if ((e = cudaMemsetAsync(out->part_score, 0, SK * sizeof(float), st)) != cudaSuccess) return (int)e;
        if ((e = cudaMemsetAsync(out->part_box, 0, SK * 4 * sizeof(float), st)) != cudaSuccess) return (int)e;
        ppn::chain_break(st);                        // what follows the memsets starts fully ordered
    }
    // Three kernels.  The limb arg-max (K3) and decode+NMS (K12) are independent; the tree parse
    // (K4) needs both.  parse.overlap selects how they are ordered:
    //   2  one stream, programmatic dependent launches: K12 starts, K3 starts beside it at once
    //      (it reads nothing of K12's) and only waits for K12 before it completes; K4 starts its
    //      prologue (staging the decode planes) under K3's tail and waits for K3 before reading the
    //      arg-max map and the root lists.  No events, no second stream.
    //   1  K12 on a private side stream, joined before K4.
    //   0  serial: K3, K12, K4 (also used while ppn_profile_* brackets the stages with events,
    //      so that the stage times are clean).
    cudaEvent_t* ev = profile_slot();
    const int mode = ev ? 0 : g_tuning.parse_overlap;
    // Default: TWO kernels.  The limb arg-max (K3) and the fused decode + NMS + tree parse (K124), which
    // is a programmatic dependent of K3: it becomes resident beside it, does everything that does not
    // need the arg-max map (candidates, NMS, delta) while K3 streams, then waits for K3 and walks.
    //  * default flags: K3 waits for whatever precedes it in the stream (it may be producing `head`),
    //    K124 triggers after its wait — the next call's K3 only hides its launch latency;
    //  * PPN_FLAG_INPUT_COMPLETE: K3 starts at once; K124 triggers EARLY (after seeing the previous
    //    call's K124 complete), so the next call's K3 is launched while this call's K3 still runs and
    //    takes over its SMs as they free up — the limb stream never pauses between calls.  K3 waits at
    //    its end for the previous K124, K124 waits for its K3: calls complete in order.
    // Needs n_nms_parts == 1 (the reference's case) and a grid of at most 1024 cells; otherwise, or with
    // ppn_tune("parse.fused", 0), the three-kernel chain below runs.
    ppn::FusedSplit split;
    const bool fits_beside = P == 1 && ppn::parse_fused_split(g, g_tuning.parse_stage_all, g_tuning, &split);
    // auto: the two-kernel chain when the whole batch's parse CTAs fit beside the arg-max ring.  A batch that
    // would have to be cut (dense 16x16 crowds at B = 1024: two sub-batches) measured no better than the
    // three-kernel chain — there the parse work itself is as long as the arg-max — so it keeps that one.
    const bool fused = P == 1 && mode != 1 && (g_tuning.parse_fused < 0 ? (fits_beside && split.n_sub == 1) : (g_tuning.parse_fused != 0 &&
                       ppn::parse_fused_supported(g, g_tuning.parse_stage_all)));
    // the dense entry buffer: written by the fused kernel itself (its cursor, header[0..1], is cleared by
    // the arg-max kernel of the same call — nothing but kernels goes on the stream, so the overlapped
    // chain stays intact) or, on the other paths and for K > 32, by the pack kernels after the
    // fixed-stride result
    const bool dense_fused = dense && fused && shape->K <= 32;
    if (dense && dense->rheader && !dense_fused) return PPN_E_UNSUPPORTED;
    if (fused) {
        using namespace ppn;
        Tuning tuning = g_tuning;
        // A batch whose parse CTAs do not all fit on the SMs beside the arg-max ring is cut into equal
        // sub-batches that do: K3(0) K124(0) K3(1) K124(1) ... — K3(j+1) streams while sub-batch j is parsed.
        const int n_sub = fits_beside ? split.n_sub : 1;
        const int sub_B = fits_beside ? split.sub_B : g.B;
        const int staged_forced = fits_beside ? (split.staged ? 1 : 0) : -1;
        if (fits_beside) tuning.argmax_smem_cap = (int)split.ring_cap;      // leave room for every parse CTA on the SM
        const bool overlap_calls = (params->flags & PPN_FLAG_INPUT_COMPLETE) != 0;
        const bool chain = mode == 2 && g_tuning.parse_chain_calls != 0;
        cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
        if ((e = cudaStreamIsCapturing(st, &cap)) != cudaSuccess) return (int)e;
        const bool capturing = cap != cudaStreamCaptureStatusNone;
        const size_t es = elem_bytes(shape);
        const size_t K = (size_t)shape->K, R = (size_t)out->R;
        auto launch_k3 = [&](int j) -> cudaError_t {
            Geom gj = timeline_slot(g);
            const int b0 = j * sub_B;
            gj.B = std::min(sub_B, g.B - b0);
            // an overlapped K3 may only start beside a fused parse that publishes; after anything else of
            // ours it starts fully ordered (no launch attribute), which also restarts the chain cleanly.
            // Inside a call the kernel before K3(j > 0) is this call's own K124(j - 1).
            const bool attr = chain && (j > 0 || !overlap_calls || capturing || chain_clean(st));
            const int bits = mode != 2 ? 0 : ((overlap_calls || j > 0) ? (PDL_TRIGGER | PDL_WAIT_END) : (PDL_WAIT_START | PDL_TRIGGER));
            bool chained = false, zeroed = false;
            int32_t* zero2 = (dense_fused && j == 0) ? dense->header : nullptr;
            cudaError_t err = launch_limb_argmax(static_cast<const unsigned char*>(head) + (size_t)b0 * g.img_stride * es,
                                                 amax + (size_t)b0 * g.E * g.HW, gj, tuning, st, attr, &chained, bits, zero2, &zeroed);
            if (err == cudaSuccess && zero2 && !zeroed) err = cudaMemsetAsync(dense->header, 0, 2 * sizeof(int32_t), st);
            return err;
        };
        auto launch_k124 = [&](int j) -> cudaError_t {
            Geom gj = timeline_slot(g);
            const int b0 = j * sub_B;
            gj.B = std::min(sub_B, g.B - b0);
            DenseTarget dj;
            if (dense_fused) { dj = *dense; dj.B_total = g.B; dj.b0 = b0; }
            return launch_parse_fused(static_cast<const unsigned char*>(head) + (size_t)b0 * g.img_stride * es, gj, ch,
                                      params->det_thresh, params->nms_thresh, params->min_num_keypoints,
                                      amax + (size_t)b0 * g.E * g.HW, out->count + b0, out->root_cell + (size_t)b0 * R,
                                      out->part_cell + (size_t)b0 * R * K, out->part_score + (size_t)b0 * R * K,
                                      out->part_box + (size_t)b0 * R * K * 4, out->R, st,
                                      mode == 2 /* a programmatic dependent of K3 (implicit trigger if K3 is a fallback kernel) */,
                                      (overlap_calls && chain && !capturing) ? 2 : 1, g_tuning.parse_stage_all, staged_forced,
                                      dense_fused ? &dj : nullptr);
        };
        if (ev) {                                      // per-stage events: serial, all arg-max launches, then all parse launches
            cudaEventRecord(ev[0], st);
            for (int j = 0; j < n_sub; ++j) if ((e = launch_k3(j)) != cudaSuccess) return (int)e;
            cudaEventRecord(ev[1], st);
            for (int q = 2; q < 7; ++q) cudaEventRecord(ev[q], st);
            for (int j = 0; j < n_sub; ++j) if ((e = launch_k124(j)) != cudaSuccess) return (int)e;
            cudaEventRecord(ev[7], st);
        } else {
            for (int j = 0; j < n_sub; ++j) {
                if ((e = launch_k3(j)) != cudaSuccess) return (int)e;
                if ((e = launch_k124(j)) != cudaSuccess) return (int)e;
            }
        }
        if (dense && !dense_fused) return pack_after(out, shape, dense, st);
        return PPN_OK;
    }
    if (dense && dense->rheader) return PPN_E_UNSUPPORTED;     // remote entries are written by the fused parse kernel only
    if (mode == 2) {
        using namespace ppn;
        // Three kernels on one stream, chained by programmatic dependent launches, the two small ones as PERSISTENT
        // grids that are resident beside the arg-max ring (parse.persist; the ring is capped to leave them room):
        //   K12(i)  decode + NMS      needs only the head tensor; triggers at its top
        //   K3(i)   limb arg-max      starts beside K12(i) at once; waits for it only before completing
        //   K4(i)   tree parse        waits for K3(i) (hence K12(i)), then walks
        //  * default: K12 waits for whatever precedes it in the stream before reading anything (the producer of `head`
        //    may be that kernel), K4 triggers after its wait — only launch latencies are hidden between calls;
        //  * PPN_FLAG_INPUT_COMPLETE: K4(i) triggers at its very TOP, so K12(i+1) and K3(i+1) are launched while K3(i)
        //    still streams: K12(i+1) runs under K3(i) / K3(i+1), K4(i) under K3(i+1), and the limb stream never pauses.
        //    Safe because K4(i) triggers only after it has SEEN K4(i-1) complete (sequence number published by K4's
        //    last CTA — the same words the fused parse kernel uses): the kernels of call i+1 write the workspace set
        //    call i-1 read.  Completion stays transitive: K3 waits at its end for K12, K12 for the previous K4.
        //    Every kernel of the chain is fully resident when it triggers (persistent grids), so no waiting CTA can
        //    keep a CTA it waits for off the SMs.
        const bool overlap_calls = (params->flags & PPN_FLAG_INPUT_COMPLETE) != 0;
        const bool chain_calls = g_tuning.parse_chain_calls != 0;
        cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
        if ((e = cudaStreamIsCapturing(st, &cap)) != cudaSuccess) return (int)e;
        const bool capturing = cap != cudaStreamCaptureStatusNone;
        Tuning tuning = g_tuning;
        int k12_ctas = g_tuning.parse_persist, k4_ctas = g_tuning.parse_persist > 0 ? 1 : 0;
        if (k12_ctas > 0) {
            const size_t ring_cap = chain3_ring_cap(g, g_tuning.parse_stage_all, k12_ctas);
            if (ring_cap) tuning.argmax_smem_cap = (int)ring_cap;
            else k12_ctas = k4_ctas = 0;                    // no room beside a ring: the one-CTA-per-image kernels
        }
        const bool early = overlap_calls && chain_calls && !capturing && k4_ctas > 0;
        // K12 may start beside the previous call's parse only if that one publishes (ours do); after anything else it
        // starts fully ordered.  Without the flag it waits at its start, so the attribute only hides launch latency.
        const bool attr12 = chain_calls && (!overlap_calls || capturing || chain_clean(st));
        const int bits12 = PDL_TRIGGER | (!attr12 ? 0 : (overlap_calls ? PDL_WAIT_END : PDL_WAIT_START));
        bool chained = false;
        if ((e = launch_decode_nms(head, timeline_slot(g), P, params->det_thresh, params->nms_thresh, keep_idx, keep_count, st, attr12,
                                   bits12, k12_ctas, g_tuning.parse_k12_threads)) != cudaSuccess) return (int)e;
        if ((e = launch_limb_argmax(head, amax, timeline_slot(g), tuning, st, true, &chained)) != cudaSuccess) return (int)e;
        if ((e = launch_tree_parse(head, timeline_slot(g), ch, params->det_thresh, params->min_num_keypoints, P, amax, nullptr, keep_idx,
                                   keep_count, out->count, out->root_cell, out->part_cell, out->part_score, out->part_box,
                                   out->R, st, chained, chained ? (PDL_WAIT_START | PDL_TRIGGER) : 0, g_tuning.parse_stage_all,
                                   g_tuning.parse_threads, chained ? (early ? 2 : 1) : 0, k4_ctas)) != cudaSuccess) return (int)e;
        if (!chained) chain_break(st);
        if (!dense) return PPN_OK;
        rc = pack_after(out, shape, dense, st);             // plain launches: the next call starts fully ordered behind them
        chain_break(st);
        return rc;
    }
    ppn::chain_break(st);
    cudaStream_t side = st;
    SideLane* lane = nullptr;
    if (mode == 1) {
        if ((e = side_lane(&lane)) != cudaSuccess) return (int)e;
        side = lane->stream;
        if ((e = cudaEventRecord(lane->fork, st)) != cudaSuccess) return (int)e;
        if ((e = cudaStreamWaitEvent(side, lane->fork, 0)) != cudaSuccess) return (int)e;
    }
    if (ev) cudaEventRecord(ev[0], st);
    if ((e = ppn::launch_limb_argmax(head, amax, g, g_tuning, st)) != cudaSuccess) return (int)e;
    if (ev) cudaEventRecord(ev[1], st);
    // K1+K2 fused: candidates never leave shared memory (stage slot 1 = decode is inside slot 2)
    if (ev) { cudaEventRecord(ev[2], side); cudaEventRecord(ev[3], side); cudaEventRecord(ev[4], side); }
    if ((e = ppn::launch_decode_nms(head, g, P, params->det_thresh, params->nms_thresh, keep_idx, keep_count, side)) != cudaSuccess) return (int)e;
    if (ev) cudaEventRecord(ev[5], side);
    if (lane) {
        if ((e = cudaEventRecord(lane->join, side)) != cudaSuccess) return (int)e;
        if ((e = cudaStreamWaitEvent(st, lane->join, 0)) != cudaSuccess) return (int)e;
    }
    if (ev) cudaEventRecord(ev[6], st);
    if ((e = ppn::launch_tree_parse(head, g, ch, params->det_thresh, params->min_num_keypoints, P, amax, nullptr /*keep_idx holds cells*/,
                                    keep_idx, keep_count, out->count, out->root_cell, out->part_cell, out->part_score,
                                    out->part_box, out->R, st, false, 0, g_tuning.parse_stage_all, g_tuning.parse_threads)) != cudaSuccess) return (int)e;
    if (ev) cudaEventRecord(ev[7], st);
    return dense ? pack_after(out, shape, dense, st) : PPN_OK;
}

// ---- fused network head ---------------------------------------------------------------------
namespace {
struct HeadWorkspace { size_t dec, amax, keys, total; };
HeadWorkspace carve_head(const PPNShape* s) {
    HeadWorkspace w;
    const size_t B = (size_t)s->B, HW = (size_t)s->H * s->W;
    w.dec = 0;
    w.amax = align_up(B * 6 * s->K * HW * sizeof(float), 256);
    w.keys = w.amax + align_up(B * s->E * HW * sizeof(uint16_t), 256);
    w.total = w.keys + align_up(B * s->E * HW * sizeof(unsigned long long), 256);     // the epilogue's running maxima
    return w;
}
int check_head(const float* feat, const float* weight, int32_t Cin, const PPNShape* s) {
    if ((long long)s->H * s->W > 65536) return PPN_E_UNSUPPORTED;
    if (Cin < 32 || Cin % 32 != 0 || (s->H * s->W) % 4 != 0) return PPN_E_UNSUPPORTED;
    if (s->head_dtype != PPN_HEAD_F32) return PPN_E_UNSUPPORTED;
    if (!feat || !weight) return PPN_E_BADARG;
    if ((reinterpret_cast<uintptr_t>(feat) & 15) || (reinterpret_cast<uintptr_t>(weight) & 15)) return PPN_E_BADARG;
    return PPN_OK;
}
}  // namespace

int ppn_head_workspace_bytes(const PPNShape* shape, size_t* bytes) {
    int rc = check_shape(shape);
    if (rc) return rc;
    if (!bytes) return PPN_E_BADARG;
    *bytes = carve_head(shape).total;
    return PPN_OK;
}

int ppn_head_gemm_argmax(const float* feat, const float* weight, const float* bias, int32_t Cin, const PPNShape* shape,
                         float* dec, uint16_t* amax, float* emit_logits, float* emit_head, void* stream) {
    const ppn::Tuning g_tuning = tuning_now();
    int rc = check_shape(shape);
    if (rc) return rc;
    if (shape->B == 0) return PPN_OK;
    if ((rc = check_head(feat, weight, Cin, shape))) return rc;
    if (!dec || (!amax && shape->E > 0) || (reinterpret_cast<uintptr_t>(bias) & 15)) return PPN_E_BADARG;
    // no workspace in this signature: the running maxima live in a stream-ordered allocation
    const ppn::Geom g = make_geom(shape);
    cudaStream_t st = (cudaStream_t)stream;
    void* keys = nullptr;
    cudaError_t e = cudaMallocAsync(&keys, std::max<size_t>(ppn::head_keys_bytes(g), 256), st);
    if (e != cudaSuccess) return cuda_rc(e);
    e = ppn::launch_head_gemm_argmax(feat, weight, bias, Cin, g, dec, amax, static_cast<unsigned long long*>(keys), emit_logits,
                                     emit_head, st, false, 0, g_tuning.head_subs);
    const cudaError_t e2 = cudaFreeAsync(keys, st);
    return cuda_rc(e != cudaSuccess ? e : e2);
}

namespace {
struct HeadWorkspaceOpt { size_t dec, amax, keys, xt, wt, total; };
bool opt_16bit(const PPNHeadOptions* o) { return o->operand == PPN_GEMM_F16 || o->operand == PPN_GEMM_BF16; }
int check_head_opt(const void* feat, const float* weight, int32_t Cin, const PPNShape* s, const PPNHeadOptions* o) {
    if (!o) return PPN_E_BADARG;
    if (o->operand < PPN_GEMM_TF32 || o->operand > PPN_GEMM_BF16) return PPN_E_BADARG;
    if (o->feat_layout != PPN_FEAT_NCHW_F32 && o->feat_layout != PPN_FEAT_NHWC_16) return PPN_E_BADARG;
    if (!opt_16bit(o) && o->feat_layout != PPN_FEAT_NCHW_F32) return PPN_E_UNSUPPORTED;
    if (s->B == 0) return PPN_OK;
    if (!opt_16bit(o)) return check_head(static_cast<const float*>(feat), weight, Cin, s);
    if (s->head_dtype != PPN_HEAD_F32) return PPN_E_UNSUPPORTED;
    if (!ppn::head16_supported(Cin, make_geom(s))) return PPN_E_UNSUPPORTED;
    if (!feat || !weight) return PPN_E_BADARG;
    if ((reinterpret_cast<uintptr_t>(feat) & 15) || (reinterpret_cast<uintptr_t>(weight) & 15)) return PPN_E_BADARG;
    return PPN_OK;
}
HeadWorkspaceOpt carve_head_opt(const PPNShape* s, int32_t Cin, const PPNHeadOptions* o) {
    const HeadWorkspace w = carve_head(s);
    HeadWorkspaceOpt r;
    r.dec = w.dec; r.amax = w.amax; r.keys = w.keys; r.xt = r.wt = r.total = w.total;
    if (opt_16bit(o)) {
        const ppn::Geom g = make_geom(s);
        r.wt = r.xt + (o->feat_layout == PPN_FEAT_NCHW_F32 ? align_up(ppn::head16_packed_feat_bytes(Cin, g), 1024) : 0);
        r.total = r.wt + align_up(ppn::head16_packed_weight_bytes(Cin, g), 1024);
    }
    return r;
}
}  // namespace

int ppn_head_workspace_bytes_opt(const PPNShape* shape, int32_t Cin, const PPNHeadOptions* opt, size_t* bytes) {
    int rc = check_shape(shape);
    if (rc) return rc;
    if (!bytes || !opt || Cin < 1) return PPN_E_BADARG;
    *bytes = carve_head_opt(shape, Cin, opt).total;
    return PPN_OK;
}

int ppn_head_gemm_argmax_opt(const void* feat, const float* weight, const float* bias, int32_t Cin, const PPNShape* shape,
                             const PPNHeadOptions* opt, void* workspace, size_t workspace_bytes,
                             float* dec, uint16_t* amax, float* emit_logits, float* emit_head, void* stream) {
    int rc = check_shape(shape);
    if (rc) return rc;
    if ((rc = check_head_opt(feat, weight, Cin, shape, opt))) return rc;
    if (!opt_16bit(opt))
        return ppn_head_gemm_argmax(static_cast<const float*>(feat), weight, bias, Cin, shape, dec, amax, emit_logits, emit_head, stream);
    if (shape->B == 0) return PPN_OK;
    if (!dec || (!amax && shape->E > 0) || (reinterpret_cast<uintptr_t>(bias) & 15)) return PPN_E_BADARG;
    if (!workspace || (reinterpret_cast<uintptr_t>(workspace) & 255)) return PPN_E_BADARG;
    const HeadWorkspaceOpt w = carve_head_opt(shape, Cin, opt);
    if (workspace_bytes < w.total) return PPN_E_WORKSPACE;
    unsigned char* ws = static_cast<unsigned char*>(workspace);
    return cuda_rc(ppn::launch_head_gemm16_argmax(feat, opt->feat_layout == PPN_FEAT_NCHW_F32, weight, bias, Cin,
                                                  opt->operand == PPN_GEMM_BF16, make_geom(shape), ws + w.xt, ws + w.wt, dec, amax,
                                                  reinterpret_cast<unsigned long long*>(ws + w.keys), emit_logits, emit_head,
                                                  (cudaStream_t)stream, 0, tuning_now().head_subs));
}

int ppn_head_parse_opt(const void* feat, const float* weight, const float* bias, int32_t Cin, const PPNShape* shape,
                       const PPNParams* params, const PPNHeadOptions* opt, const PPNHumans* out, void* workspace,
                       size_t workspace_bytes, float* emit_logits, float* emit_head, void* stream) {
    const ppn::Tuning g_tuning = tuning_now();
    int rc = check_shape(shape);
    if (rc) return rc;
    if ((rc = check_params(shape, params))) return rc;
    if ((rc = check_humans(out))) return rc;
    ppn::ChainTable ch;
    if ((rc = make_chains(shape, params, &ch))) return rc;
    if ((rc = check_head_opt(feat, weight, Cin, shape, opt))) return rc;
    if (shape->B == 0) return PPN_OK;
    if (!workspace || (reinterpret_cast<uintptr_t>(workspace) & 255)) return PPN_E_BADARG;
    if (params->n_nms_parts != 1 || (long long)shape->H * shape->W > PPN_MAX_CELLS) return PPN_E_UNSUPPORTED;
    if ((reinterpret_cast<uintptr_t>(out->part_box) & 15) || (reinterpret_cast<uintptr_t>(bias) & 15)) return PPN_E_BADARG;
    const HeadWorkspaceOpt w = carve_head_opt(shape, Cin, opt);
    if (workspace_bytes < w.total) return PPN_E_WORKSPACE;
    unsigned char* ws = static_cast<unsigned char*>(workspace);
    float* dec = reinterpret_cast<float*>(ws + w.dec);
    uint16_t* amax = reinterpret_cast<uint16_t*>(ws + w.amax);
    const ppn::Geom g = make_geom(shape);
    // the parse kernel reads the decode planes as a head tensor that holds nothing but its 6K decode channels
    ppn::Geom gd = g;
    gd.img_stride = (size_t)6 * g.K * g.HW;
    if (!ppn::parse_fused_supported(gd, g_tuning.parse_stage_all)) return PPN_E_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e;
    if (params->flags & PPN_FLAG_CLEAR_UNUSED) {     // as ppn_parse: slots past count[b] read -1 / 0
        const size_t slots = (size_t)shape->B * out->R, SK = slots * shape->K;
        if ((e = cudaMemsetAsync(out->root_cell, 0xFF, slots * sizeof(int32_t), st)) != cudaSuccess) return (int)e;
        if ((e = cudaMemsetAsync(out->part_cell, 0xFF, SK * sizeof(int32_t), st)) != cudaSuccess) return (int)e;
        if ((e = cudaMemsetAsync(out->part_score, 0, SK * sizeof(float), st)) != cudaSuccess) return (int)e;
        if ((e = cudaMemsetAsync(out->part_box, 0, SK * 4 * sizeof(float), st)) != cudaSuccess) return (int)e;
        ppn::chain_break(st);                        // what follows the memsets starts fully ordered
    }
    // launches: clear the running maxima, [pack the operands,] GEMM + epilogue, maxima -> arg-max map, parse (a programmatic
    // dependent of the last: it becomes resident early and waits at its top)
    unsigned long long* keys = reinterpret_cast<unsigned long long*>(ws + w.keys);
    if (opt_16bit(opt))
        e = ppn::launch_head_gemm16_argmax(feat, opt->feat_layout == PPN_FEAT_NCHW_F32, weight, bias, Cin, opt->operand == PPN_GEMM_BF16,
                                           g, ws + w.xt, ws + w.wt, dec, amax, keys, emit_logits, emit_head, st, 0, g_tuning.head_subs);
    else
        e = ppn::launch_head_gemm_argmax(static_cast<const float*>(feat), weight, bias, Cin, g, dec, amax, keys, emit_logits, emit_head, st,
                                         false, 0, g_tuning.head_subs);
    if (e != cudaSuccess) return (int)e;
    e = ppn::launch_parse_fused(dec, gd, ch, params->det_thresh, params->nms_thresh, params->min_num_keypoints, amax, out->count,
                                out->root_cell, out->part_cell, out->part_score, out->part_box, out->R, st, true, 1,
                                g_tuning.parse_stage_all, -1, nullptr, true);
    ppn::chain_break(st);
    return cuda_rc(e);
}

int ppn_head_parse(const float* feat, const float* weight, const float* bias, int32_t Cin, const PPNShape* shape,
                   const PPNParams* params, const PPNHumans* out, void* workspace, size_t workspace_bytes,
                   float* emit_logits, float* emit_head, void* stream) {
    const PPNHeadOptions opt = {PPN_GEMM_TF32, PPN_FEAT_NCHW_F32};
    return ppn_head_parse_opt(feat, weight, bias, Cin, shape, params, &opt, out, workspace, workspace_bytes, emit_logits, emit_head, stream);
}

int ppn_part_centres(const PPNHumans* humans, int32_t B, int32_t K, float* centre_yx, void* stream) {
    int rc = check_humans(humans);
    if (rc) return rc;
    if (B < 0 || K < 1) return PPN_E_BADARG;
    if (B == 0) return PPN_OK;
    if (!centre_yx || (reinterpret_cast<uintptr_t>(centre_yx) & 7) || (reinterpret_cast<uintptr_t>(humans->part_box) & 15)) return PPN_E_BADARG;
    return cuda_rc(ppn::launch_part_centres(humans->count, humans->part_cell, humans->part_box, B, humans->R, K, centre_yx,
                                            (cudaStream_t)stream));
}


int ppn_skeleton(const PPNHumans* humans, int32_t B, int32_t K, int32_t E, const int32_t* edges,
                 int32_t* rect, float* keypoint_xy, float* segment, void* stream) {
    int rc = check_humans(humans);
    if (rc) return rc;
    if (B < 0 || K < 1 || E < 0 || K > 255 || E > 255) return PPN_E_BADARG;
    if (B == 0) return PPN_OK;
    if (!rect || !keypoint_xy || (E > 0 && (!segment || !edges))) return PPN_E_BADARG;
    if ((reinterpret_cast<uintptr_t>(rect) & 15) || (reinterpret_cast<uintptr_t>(keypoint_xy) & 7) ||
        (reinterpret_cast<uintptr_t>(segment) & 15) || (reinterpret_cast<uintptr_t>(humans->part_box) & 15)) return PPN_E_BADARG;
    for (int e = 0; e < E; ++e)
        if (edges[2 * e] < 0 || edges[2 * e] >= K || edges[2 * e + 1] < 0 || edges[2 * e + 1] >= K) return PPN_E_CHAINS;
    return cuda_rc(ppn::launch_skeleton(humans->count, humans->part_cell, humans->part_box, B, humans->R, K, E, edges, rect,
                                        keypoint_xy, segment, (cudaStream_t)stream));
}

int ppn_packed_bytes(int32_t B, int32_t cap_entries, size_t* bytes, size_t* offsets) {
    if (B < 0 || cap_entries < 0 || !bytes) return PPN_E_BADARG;
    const PackedLayout l = packed_layout(B, cap_entries);
    *bytes = l.total;
    if (offsets) { offsets[0] = l.header; offsets[1] = l.idcell; offsets[2] = l.score; offsets[3] = l.box; }
    return PPN_OK;
}

int ppn_pack_humans(const PPNHumans* humans, int32_t B, int32_t K, int32_t cap_entries, void* packed, size_t packed_bytes,
                    void* stream) {
    int rc = check_humans(humans);
    if (rc) return rc;
    if (B < 0 || K < 1 || cap_entries < 0) return PPN_E_BADARG;
    if (K > 65535 || humans->R > 65536) return PPN_E_UNSUPPORTED;          // part id and cell share 32 bits
    if (B == 0) return PPN_OK;
    if (!packed || (reinterpret_cast<uintptr_t>(packed) & 255)) return PPN_E_BADARG;
    const PackedLayout l = packed_layout(B, cap_entries);
    if (packed_bytes < l.total) return PPN_E_WORKSPACE;
    unsigned char* p = static_cast<unsigned char*>(packed);
    return cuda_rc(ppn::launch_pack_humans(humans->count, humans->part_cell, humans->part_score, humans->part_box, B,
                                           humans->R, K, cap_entries, reinterpret_cast<int32_t*>(p + l.header),
                                           reinterpret_cast<uint32_t*>(p + l.idcell), reinterpret_cast<float*>(p + l.score),
                                           reinterpret_cast<float*>(p + l.box), (cudaStream_t)stream));
}

int ppn_encode_targets(const PPNPeople* people, const PPNShape* shape, const int32_t* edges,
                       const PPNTargets* out, void* stream) {
    return ppn_encode_targets_opt(people, shape, edges, out, PPN_HEAD_F32, stream);
}

int ppn_encode_targets_opt(const PPNPeople* people, const PPNShape* shape, const int32_t* edges,
                           const PPNTargets* out, int32_t limb_dtype, void* stream) {
    const ppn::Tuning g_tuning = tuning_now();
    int rc = check_shape(shape);
    if (rc) return rc;
    if (!people || !out) return PPN_E_BADARG;
    if (limb_dtype < PPN_HEAD_F32 || limb_dtype > PPN_HEAD_BF16) return PPN_E_BADARG;
    if (shape->gridW < 1 || shape->gridH < 1) return PPN_E_BADARG;                     // the encoder divides by them
    if (shape->sH != shape->sW || (shape->sH & 1) == 0) return PPN_E_UNSUPPORTED;      // dataset.py:163-167
    if (shape->B == 0) return PPN_OK;
    if (!people->person_off || !out->delta || !out->weight || !out->tx || !out->ty || !out->tx_half || !out->ty_half ||
        !out->tw || !out->th) return PPN_E_BADARG;
    if (shape->E > 0 && (!edges || !out->te || !out->weight_ij)) return PPN_E_BADARG;
    if ((reinterpret_cast<uintptr_t>(out->te) & 15) || (reinterpret_cast<uintptr_t>(out->weight_ij) & 15)) return PPN_E_BADARG;
    ppn::EncodeArgs a;
    std::memset(&a, 0, sizeof(a));
    for (int e = 0; e < shape->E; ++e) {
        const int s = edges[2 * e], t = edges[2 * e + 1];
        if (s < 0 || s >= shape->K || t < 0 || t >= shape->K) return PPN_E_CHAINS;
        a.edges.src[e] = (uint8_t)s;
        a.edges.dst[e] = (uint8_t)t;
    }
    a.person_off = people->person_off; a.bbox = people->bbox; a.keypoints = people->keypoints;
    a.visible = people->visible; a.size = people->size;
    a.delta = out->delta; a.weight = out->weight; a.weight_ij = out->weight_ij; a.tx = out->tx; a.ty = out->ty;
    a.tx_half = out->tx_half; a.ty_half = out->ty_half; a.tw = out->tw; a.th = out->th; a.te = out->te;
    a.limb_dtype = limb_dtype;
    a.K = shape->K; a.E = shape->E; a.H = shape->H; a.W = shape->W; a.sH = shape->sH; a.sW = shape->sW;
    a.sweep = g_tuning.encode_sweep;
    a.sweep_ctas_per_sm = g_tuning.encode_ctas_per_sm;
    a.magic_sW = shape->sW <= 1 ? 0u : (uint32_t)(((1ull << 32) + shape->sW - 1) / shape->sW);
    a.gridW = (float)shape->gridW; a.gridH = (float)shape->gridH;
    a.inW = (double)shape->inW; a.inH = (double)shape->inH;
    int dev = 0, sms = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return (int)e;
    if ((e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return (int)e;
    return cuda_rc(ppn::launch_encode_targets(a, shape->B, sms, (cudaStream_t)stream));
}

// ---- the training loss (PPNLoss, main.py:125-216) -----------------------------------------------------
namespace {
inline bool bad_ptr(const void* p, size_t align) { return !p || (reinterpret_cast<uintptr_t>(p) & (align - 1)); }
inline bool bad_f32(const void* p) { return bad_ptr(p, 4); }
inline size_t dtype_bytes(int32_t dtype) { return dtype == PPN_HEAD_F32 ? 4 : 2; }

// the (head, limb target) element types the kernels are built for: limb targets fp32 or the head's type
int check_loss_types(const PPNShape* shape, const PPNLossOptions* opt) {
    if (!opt || opt->limb_dtype < PPN_HEAD_F32 || opt->limb_dtype > PPN_HEAD_BF16) return PPN_E_BADARG;
    if (opt->limb_dtype != PPN_HEAD_F32 && opt->limb_dtype != shape->head_dtype) return PPN_E_UNSUPPORTED;
    return PPN_OK;
}

int loss_args(const void* head, const PPNShape* shape, const PPNTargets* t, const PPNLossOptions* opt, ppn::LossArgs* a) {
    int rc = check_shape(shape);
    if (rc) return rc;
    if ((rc = check_loss_types(shape, opt))) return rc;
    if (shape->B < 1) return PPN_E_BADARG;                                   // the batch mean needs an image
    std::memset(a, 0, sizeof(*a));
    const ppn::Geom g = make_geom(shape);
    a->B = g.B; a->K = g.K; a->W = g.W; a->HW = g.HW; a->L = g.S * g.E * g.HW;
    a->img_stride = g.img_stride; a->limb_off = g.limb_off;
    a->gW = g.gridW; a->gH = g.gridH; a->inW = g.inW; a->inH = g.inH;
    a->head_dtype = shape->head_dtype;
    a->limb_dtype = opt->limb_dtype;
    ppn::loss_plan(a);
    if (!t) return PPN_E_BADARG;
    const float* small[] = {t->delta, t->weight, t->tx, t->ty, t->tx_half, t->ty_half, t->tw, t->th};
    for (const float* p : small)
        if (bad_f32(p)) return PPN_E_BADARG;
    const size_t limb_align = dtype_bytes(opt->limb_dtype);
    if (bad_ptr(head, elem_bytes(shape)) || (a->L > 0 && (bad_ptr(t->te, limb_align) || bad_ptr(t->weight_ij, limb_align))))
        return PPN_E_BADARG;
    a->head = head;
    a->delta = t->delta; a->weight = t->weight; a->weight_ij = t->weight_ij; a->tx = t->tx; a->ty = t->ty;
    a->tx_half = t->tx_half; a->ty_half = t->ty_half; a->tw = t->tw; a->th = t->th; a->te = t->te;
    return PPN_OK;
}

int sm_count(int* sms) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev);
    return cuda_rc(e);
}

// the fp32 exports: fp32 head and targets only, as before the 16-bit path existed
const PPNLossOptions kLossF32 = {PPN_HEAD_F32};
int check_f32_loss(const PPNShape* shape) {
    int rc = check_shape(shape);
    if (rc) return rc;
    return shape->head_dtype != PPN_HEAD_F32 ? PPN_E_UNSUPPORTED : PPN_OK;
}
}  // namespace

int ppn_loss_workspace_bytes_opt(const PPNShape* shape, const PPNLossOptions* opt, size_t* bytes) {
    int rc = check_shape(shape);
    if (rc) return rc;
    if (!bytes) return PPN_E_BADARG;
    if ((rc = check_loss_types(shape, opt))) return rc;
    if (shape->B < 1) return PPN_E_BADARG;
    ppn::LossArgs a;
    std::memset(&a, 0, sizeof(a));
    a.B = shape->B; a.K = shape->K; a.HW = shape->H * shape->W; a.L = shape->sH * shape->sW * shape->E * a.HW;
    ppn::loss_plan(&a);
    *bytes = ppn::loss_workspace_bytes(a);
    return PPN_OK;
}

int ppn_loss_workspace_bytes(const PPNShape* shape, size_t* bytes) {
    int rc = check_shape(shape);
    if (rc) return rc;
    if (!bytes) return PPN_E_BADARG;
    if ((rc = check_f32_loss(shape))) return rc;
    return ppn_loss_workspace_bytes_opt(shape, &kLossF32, bytes);
}

namespace {
// the forward and backward exports with the head as the sigmoid's output (from_logits false) or its input (true)
int loss_forward(const void* head, const PPNShape* shape, const PPNTargets* targets, const PPNLossOptions* opt,
                 float* loss, void* workspace, size_t workspace_bytes, void* stream, bool from_logits) {
    ppn::LossArgs a;
    int rc = loss_args(head, shape, targets, opt, &a);
    if (rc) return rc;
    if (bad_f32(loss) || !workspace || (reinterpret_cast<uintptr_t>(workspace) & 7)) return PPN_E_BADARG;
    if (workspace_bytes < ppn::loss_workspace_bytes(a)) return PPN_E_WORKSPACE;
    a.partial = static_cast<double*>(workspace);
    int sms = 0;
    if ((rc = sm_count(&sms))) return rc;
    return cuda_rc(ppn::launch_loss_forward(a, loss, sms, (cudaStream_t)stream, from_logits));
}

int loss_backward(const void* head, const PPNShape* shape, const PPNTargets* targets, const PPNLossOptions* opt,
                  const float* grad_loss, void* grad_head, void* stream, bool from_logits) {
    ppn::LossArgs a;
    int rc = loss_args(head, shape, targets, opt, &a);
    if (rc) return rc;
    if (bad_f32(grad_loss) || bad_ptr(grad_head, elem_bytes(shape))) return PPN_E_BADARG;
    a.grad_loss = grad_loss;
    a.grad = grad_head;
    int sms = 0;
    if ((rc = sm_count(&sms))) return rc;
    return cuda_rc(ppn::launch_loss_backward(a, sms, (cudaStream_t)stream, from_logits));
}
}  // namespace

// PPNLoss.forward (main.py:125-216): the five batch-mean terms into loss[5]
int ppn_loss_forward_opt(const void* head, const PPNShape* shape, const PPNTargets* targets, const PPNLossOptions* opt,
                         float* loss, void* workspace, size_t workspace_bytes, void* stream) {
    return loss_forward(head, shape, targets, opt, loss, workspace, workspace_bytes, stream, false);
}

int ppn_loss_forward(const float* head, const PPNShape* shape, const PPNTargets* targets, float* loss,
                     void* workspace, size_t workspace_bytes, void* stream) {
    const int rc = check_f32_loss(shape);
    return rc ? rc : ppn_loss_forward_opt(head, shape, targets, &kLossF32, loss, workspace, workspace_bytes, stream);
}

// PPNLoss's backward under autograd (loss.backward() in main.py's training step), with respect to the head only
int ppn_loss_backward_opt(const void* head, const PPNShape* shape, const PPNTargets* targets, const PPNLossOptions* opt,
                          const float* grad_loss, void* grad_head, void* stream) {
    return loss_backward(head, shape, targets, opt, grad_loss, grad_head, stream, false);
}

int ppn_loss_backward(const float* head, const PPNShape* shape, const PPNTargets* targets, const float* grad_loss,
                      float* grad_head, void* stream) {
    const int rc = check_f32_loss(shape);
    return rc ? rc : ppn_loss_backward_opt(head, shape, targets, &kLossF32, grad_loss, grad_head, stream);
}

// the loss on the conv output before model.py's final sigmoid (model.py:133-136), the sigmoid fused in
int ppn_loss_forward_logits(const void* logits, const PPNShape* shape, const PPNTargets* targets, const PPNLossOptions* opt,
                            float* loss, void* workspace, size_t workspace_bytes, void* stream) {
    return loss_forward(logits, shape, targets, opt, loss, workspace, workspace_bytes, stream, true);
}

int ppn_loss_backward_logits(const void* logits, const PPNShape* shape, const PPNTargets* targets, const PPNLossOptions* opt,
                             const float* grad_loss, void* grad_logits, void* stream) {
    return loss_backward(logits, shape, targets, opt, grad_loss, grad_logits, stream, true);
}

int ppn_sigmoid(const void* x, int32_t x_dtype, float* y, size_t n, void* stream) {
    if (x_dtype < PPN_HEAD_F32 || x_dtype > PPN_HEAD_BF16) return PPN_E_BADARG;
    if (n == 0) return PPN_OK;
    if (bad_ptr(x, dtype_bytes(x_dtype)) || bad_f32(y)) return PPN_E_BADARG;
    return cuda_rc(ppn::launch_sigmoid(x, x_dtype, y, n, (cudaStream_t)stream));
}

int ppn_debug_argmax_items(const PPNShape* shape, int32_t sms, int32_t* info, int32_t* first, int32_t* size, int32_t max_items) {
    int rc = check_shape(shape);
    if (rc) return rc;
    if (!info || sms < 1) return PPN_E_BADARG;
    const ppn::Tuning g_tuning = tuning_now();
    ppn::ArgmaxPlan p;
    if (!ppn::plan_argmax(make_geom(shape), g_tuning, sms, &p) || !p.split_mats) return PPN_E_UNSUPPORTED;
    struct Ctx { int32_t* first; int32_t* size; int32_t max; } ctx = {first, size, max_items};
    int n_items = 0;
    ppn::argmax_item_partition(p, shape->B * shape->E, &n_items, [](void* c, int it, int m0, int nm) -> int {
        Ctx* x = static_cast<Ctx*>(c);
        if (x->first && x->size && it < x->max) { x->first[it] = m0; x->size[it] = nm; }
        return 0;
    }, &ctx);
    info[0] = p.G; info[1] = p.n_big; info[2] = p.small_m; info[3] = n_items;
    return PPN_OK;
}

int ppn_timeline(void* dev_records, int32_t max_records) {
    g_timeline.buf = static_cast<unsigned long long*>(dev_records);
    g_timeline.cap = dev_records ? max_records : 0;
    g_timeline.used = 0;
    return PPN_OK;
}

int ppn_profile_enable(int32_t on) {
    if (on && !g_prof.ev) {
        g_prof.ev = new cudaEvent_t[(size_t)kMaxProfiled * (2 * kStages)];
        for (size_t i = 0; i < (size_t)kMaxProfiled * (2 * kStages); ++i) {
            cudaError_t e = cudaEventCreate(&g_prof.ev[i]);
            if (e != cudaSuccess) return (int)e;
        }
    }
    g_prof.on = on != 0;
    g_prof.used = 0;
    return PPN_OK;
}

int ppn_profile_read(float* stage_ms, int32_t* n_calls) {
    if (!stage_ms || !n_calls) return PPN_E_BADARG;
    for (int s = 0; s < kStages; ++s) stage_ms[s] = 0.0f;
    *n_calls = g_prof.used;
    for (int c = 0; c < g_prof.used; ++c) {
        cudaEvent_t* ev = g_prof.ev + (size_t)c * (2 * kStages);
        cudaError_t e = cudaEventSynchronize(ev[2 * kStages - 1]);
        if (e != cudaSuccess) return (int)e;
        for (int s = 0; s < kStages; ++s) {
            float ms = 0.0f;
            if ((e = cudaEventElapsedTime(&ms, ev[2 * s], ev[2 * s + 1])) != cudaSuccess) return (int)e;
            stage_ms[s] += ms;
        }
    }
    g_prof.used = 0;
    return PPN_OK;
}

// ---- host-memory entry --------------------------------------------------------------------
// Device scratch layout: [head chunk A][head chunk B][workspace A][workspace B][packed result B*R].
namespace {
struct HostPlan {
    int chunk;                 // images per chunk
    size_t head_bytes;         // per chunk buffer
    size_t ws_bytes;           // per chunk workspace
    size_t off_head[2], off_ws[2], off_count, off_root, off_cell, off_score, off_box, total;
};
HostPlan plan_host(const PPNShape* s, const PPNParams* p, int R) {
    const ppn::Tuning g_tuning = tuning_now();
    HostPlan h;
    h.chunk = g_tuning.host_chunk_images;
    if (h.chunk > s->B) h.chunk = s->B > 0 ? s->B : 1;
    PPNShape cs = *s;
    cs.B = h.chunk;
    const size_t per_img = ((size_t)6 * s->K + (size_t)s->sH * s->sW * s->E) * s->H * s->W * elem_bytes(s);
    h.head_bytes = align_up(per_img * h.chunk, 256);
    h.ws_bytes = 2 * carve(&cs, p->n_nms_parts).total;
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t at = off; off = align_up(off + bytes, 256); return at; };
    h.off_head[0] = take(h.head_bytes); h.off_head[1] = take(h.head_bytes);
    h.off_ws[0] = take(h.ws_bytes); h.off_ws[1] = take(h.ws_bytes);
    const size_t B = (size_t)s->B, K = (size_t)s->K;
    h.off_count = take(B * sizeof(int32_t));
    h.off_root = take(B * R * sizeof(int32_t));
    h.off_cell = take(B * R * K * sizeof(int32_t));
    h.off_score = take(B * R * K * sizeof(float));
    h.off_box = take(B * R * K * 4 * sizeof(float));
    h.total = off;
    return h;
}
}  // namespace

int ppn_parse_host_scratch_bytes(const PPNShape* shape, const PPNParams* params, int32_t R, size_t* bytes) {
    int rc = check_shape(shape);
    if (rc) return rc;
    if ((rc = check_params(shape, params))) return rc;
    if (!bytes || R < 1) return PPN_E_BADARG;
    *bytes = plan_host(shape, params, R).total;
    return PPN_OK;
}

int ppn_parse_host(const void* head_host, const PPNShape* shape, const PPNParams* params, const PPNHumans* out_host,
                   void* dev_scratch, size_t dev_scratch_bytes) {
    int rc = check_shape(shape);
    if (rc) return rc;
    if ((rc = check_params(shape, params))) return rc;
    if ((rc = check_humans(out_host))) return rc;
    if (shape->B == 0) return PPN_OK;
    if (!head_host || !dev_scratch || (reinterpret_cast<uintptr_t>(dev_scratch) & 255)) return PPN_E_BADARG;
    const int R = out_host->R;
    const HostPlan h = plan_host(shape, params, R);
    if (dev_scratch_bytes < h.total) return PPN_E_WORKSPACE;
    unsigned char* d = static_cast<unsigned char*>(dev_scratch);
    const size_t K = (size_t)shape->K;
    const size_t per_img_b = ((size_t)6 * shape->K + (size_t)shape->sH * shape->sW * shape->E) * shape->H * shape->W * elem_bytes(shape);

    // two streams ping-pong over two (head, workspace) buffer pairs: the upload of chunk i+1 overlaps the kernels
    // of chunk i.  Created once per (thread, device) and kept.
    struct HostLane { cudaStream_t s[2] = {nullptr, nullptr}; };
    static thread_local HostLane t_lanes[64];
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return (int)e;
    if (dev < 0 || dev >= 64) return (int)cudaErrorInvalidDevice;
    cudaStream_t* streams = t_lanes[dev].s;
    for (int i = 0; i < 2; ++i)
        if (!streams[i] && (e = cudaStreamCreateWithFlags(&streams[i], cudaStreamNonBlocking)) != cudaSuccess) return (int)e;
    // whatever happens, no copy may still be in flight over the caller's buffers when we return
    auto fail = [&](int code) { cudaStreamSynchronize(streams[0]); cudaStreamSynchronize(streams[1]); return code; };

    int32_t* d_count = reinterpret_cast<int32_t*>(d + h.off_count);
    int32_t* d_root = reinterpret_cast<int32_t*>(d + h.off_root);
    int32_t* d_cell = reinterpret_cast<int32_t*>(d + h.off_cell);
    float* d_score = reinterpret_cast<float*>(d + h.off_score);
    float* d_box = reinterpret_cast<float*>(d + h.off_box);

    PPNParams chunk_params = *params;
    chunk_params.flags &= ~PPN_FLAG_INPUT_COMPLETE;      // the chunk's head arrives by the copy just ahead of it
    int slot = 0;
    for (int b0 = 0; b0 < shape->B; b0 += h.chunk, slot ^= 1) {
        const int nb = (shape->B - b0 < h.chunk) ? shape->B - b0 : h.chunk;
        cudaStream_t st = streams[slot];
        void* d_head = d + h.off_head[slot];
        if ((e = cudaMemcpyAsync(d_head, static_cast<const unsigned char*>(head_host) + (size_t)b0 * per_img_b,
                                 (size_t)nb * per_img_b, cudaMemcpyHostToDevice, st)) != cudaSuccess) return fail((int)e);
        PPNShape cs = *shape;
        cs.B = nb;
        PPNHumans dev_out;
        dev_out.count = d_count + b0;
        dev_out.root_cell = d_root + (size_t)b0 * R;
        dev_out.part_cell = d_cell + (size_t)b0 * R * K;
        dev_out.part_score = d_score + (size_t)b0 * R * K;
        dev_out.part_box = d_box + (size_t)b0 * R * K * 4;
        dev_out.R = R;
        if ((rc = ppn_parse(d_head, &cs, &chunk_params, &dev_out, d + h.off_ws[slot], h.ws_bytes, st))) return fail(rc);
        // the counts of this chunk go home behind its kernels; the slots follow once the largest count is known
        if ((e = cudaMemcpyAsync(out_host->count + b0, dev_out.count, (size_t)nb * sizeof(int32_t), cudaMemcpyDeviceToHost, st)) != cudaSuccess) return fail((int)e);
    }
    for (int i = 0; i < 2; ++i)
        if ((e = cudaStreamSynchronize(streams[i])) != cudaSuccess) return (int)e;
    // Only slots [0, count[b]) of an image carry humans.  Copy the first m = max_b min(count[b], R) slots of every
    // image (strided copies, one per array) instead of all R: at the BASELINE shapes that is several times fewer
    // bytes over PCIe (cfg2: ~20 of 144 slots).  Slots [m, R) of the host arrays are left untouched, unless
    // PPN_FLAG_CLEAR_UNUSED asks for them to be cleared: that is done here on the host, not over PCIe.
    int m = 0;
    for (int b = 0; b < shape->B; ++b) m = std::max(m, std::min(out_host->count[b], R));
    if (m > 0) {
        cudaStream_t st = streams[0];
        const size_t B = (size_t)shape->B;
        if ((e = cudaMemcpy2DAsync(out_host->root_cell, (size_t)R * 4, d_root, (size_t)R * 4, (size_t)m * 4, B, cudaMemcpyDeviceToHost, st)) != cudaSuccess) return fail((int)e);
        if ((e = cudaMemcpy2DAsync(out_host->part_cell, (size_t)R * K * 4, d_cell, (size_t)R * K * 4, (size_t)m * K * 4, B, cudaMemcpyDeviceToHost, st)) != cudaSuccess) return fail((int)e);
        if ((e = cudaMemcpy2DAsync(out_host->part_score, (size_t)R * K * 4, d_score, (size_t)R * K * 4, (size_t)m * K * 4, B, cudaMemcpyDeviceToHost, st)) != cudaSuccess) return fail((int)e);
        if ((e = cudaMemcpy2DAsync(out_host->part_box, (size_t)R * K * 16, d_box, (size_t)R * K * 16, (size_t)m * K * 16, B, cudaMemcpyDeviceToHost, st)) != cudaSuccess) return fail((int)e);
        if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return (int)e;
    }
    if ((params->flags & PPN_FLAG_CLEAR_UNUSED) && m < R) {      // device slots [count[b], m) came back cleared already
        const size_t tail = (size_t)(R - m);
        for (size_t b = 0; b < (size_t)shape->B; ++b) {
            const size_t s = b * R + m;
            std::fill_n(out_host->root_cell + s, tail, -1);
            std::fill_n(out_host->part_cell + s * K, tail * K, -1);
            std::fill_n(out_host->part_score + s * K, tail * K, 0.0f);
            std::fill_n(out_host->part_box + s * K * 4, tail * K * 4, 0.0f);
        }
    }
    return PPN_OK;
}

}  // extern "C"
