// Internal interface between the kernels (ppn_kernels.cu) and the C ABI (ppn_capi.cu).
#pragma once
#include "ppn_device.cuh"

namespace ppn {

struct Tuning {
    int argmax_variant = 0;            // 0 = TMA bulk-copy ring (persistent), 1 = direct 128-bit loads
    int argmax_stage_bytes = 0;        // ring stage size; 0 = auto: 48 KB for small matrices (<= 64 KB: several per stage, rows of
                                       // a few hundred bytes — fewer, larger stages measured 2-4 % faster), else 32 KB
    int argmax_stages = 4;
    int argmax_threads = 320;          // target consumer threads per CTA
    int argmax_ctas_per_sm = 1;
    int argmax_split = -1;             // -1 auto, 0 = groups split rows, 1 = groups take one matrix each
    int argmax_dynamic = 1;            // ring kernels draw work from a global ticket counter (0: static round-robin)
    int argmax_tail_opt = 0;           // split-matrix mode: n > 1 hands the last ~1.5 waves of work out in items 1/n the size (more rows of
                                       // fewer matrices per stage), so that the CTAs finish within 1/n item of one another.  Measured at
                                       // cfg2 (profiles/tail_sweep_r2.txt): isolated launch 60.1 us with equal items, 60.5 / 64.1 / 74.6 us
                                       // with n = 2 / 4 / 8 — a tail item keeps 1/n of the consumer threads busy and streams slower than
                                       // the half-empty last wave costs; and inside the call chain the next launch fills that wave anyway
    int argmax_cluster = -1;           // tiny batches: a cluster of CTAs per matrix, partials merged through distributed
                                       // shared memory.  -1 auto (matrices <= half the SMs), 0 never, 2/4/8 forced
    int argmax_cluster_ring = 0;       // 1: the cluster kernel streams its rows through a 4-stage ring of bulk copies instead of
                                       // 128-bit loads (measured equal, 12.3 vs 12.5 us for one native image: fixed latencies, not the
                                       // load pattern, bound a 128 KB slab per CTA — kept as a tested option)
    int argmax_smem_cap = 0;           // > 0: the ring may use at most this much shared memory (set per call by ppn_parse
                                       // so that the fused parse kernel's CTAs fit beside it on every SM)
    int argmax16_threads = 320;        // 16-bit heads: their own ring shape (rows are half as long, so an item
    int argmax16_stage_bytes = 48 * 1024;   // of G matrices is half the bytes; measured, profiles/sweep_argmax16_*)
    int parse_stage_all = -1;          // tree parse stages: -1 auto, 0 nothing, 1 resp+conf, 2 all six groups
    int parse_threads = 0;             // tree-parse CTA size, 0 = by grid size
    int parse_fused = -1;              // whole-path call: decode+NMS+tree parse in one kernel.  -1 auto (when all of its
                                       // CTAs fit on the SMs beside the arg-max ring), 0 never (three kernels), 1 whenever supported
    int parse_chain_calls = 1;         // PDL chain: the first kernel of a call is a programmatic dependent too
    int parse_k12_threads = 0;         // decode+NMS CTA size in the whole-path call, 0 = by grid size (256 up to 256 cells, else 512)
    int parse_persist = 1;             // three-kernel chain: decode+NMS and the tree parse as persistent grids resident beside the
                                       // arg-max ring (this many decode+NMS CTAs per SM, one tree-parse CTA); 0: one CTA per list / image
    int host_chunk_images = 64;
    int encode_sweep = 1;              // target encoder: limb tensors by the address-ordered persistent sweep (0: one CTA per image part)
    int encode_ctas_per_sm = 6;
    int argmax_dry = 0;                // ring kernels only move the bytes (no compares, no stores): the read ceiling of this ring
    int head_subs = 0;                 // fused head: epilogue warps per TMEM lane quadrant (1, 2, 4 or 6; 0 = auto: 4 for TF32 operands, 6 for
                                       // 16-bit ones, where the faster MMAs leave the latency-bound epilogue warps more to hide; bits 8-9:
                                       // the head.dry probes, bit 12: head.acc = 128)
    int parse_overlap = 2;             // 0 serial; 1 decode+NMS on a side stream beside the arg-max;
                                       // 2 one stream, programmatic dependent launches (PDL chain)
};

struct ArgmaxPlan {
    int CV;               // float4 columns per row = HW / 4
    int G;                // row groups: thread (g, cv) takes rows g, g+G, ... of every chunk
    int threads;          // CV * G working consumer threads
    int threads_padded;   // rounded up to whole warps
    int rows;             // rows per ring stage
    int chunks;           // stages per matrix = ceil(S / rows)
    int split_mats;       // 1: the G groups take G different matrices (no merge), 0: they split rows
    int stages;           // ring depth
    int ctas_per_sm;
    int dry;              // 1: consumers only release the stages (bandwidth probe)
    int n_big;            // split-matrix mode: items [0, n_big) hold G matrices each, the items after them `small_m`
    int small_m;          //   (a shrinking tail: with equal items the last wave of a persistent grid is on average half empty)
    int rows_s, chunks_s; // rows per stage / stages per matrix of a tail item (more rows of fewer matrices: same bytes per stage)
    uint32_t stage_bytes;
    size_t smem_bytes;
};

bool plan_argmax(const Geom& g, const Tuning& t, int sms, ArgmaxPlan* p);
void argmax_item_partition(const ArgmaxPlan& p, int n_mats, int* n_items, int (*first_size)(void*, int, int, int), void* ctx);

// pdl: launch as a programmatic dependent of the previous kernel in `st` (starts beside it, waits
// for it only before completing); *pdl_used tells whether the chosen kernel variant honoured it.
cudaError_t launch_limb_argmax(const void* head, uint16_t* amax, const Geom& g, const Tuning& t, cudaStream_t st,
                               bool pdl = false, bool* pdl_used = nullptr, int pdl_bits = -1 /* default: trigger + end wait */,
                               int32_t* zero2 = nullptr /* two ints the ring kernel clears before anything else runs */,
                               bool* zeroed = nullptr);

cudaError_t launch_decode_candidates(const void* head, const Geom& g, int n_parts, float thr, int32_t* cand_cell,
                                     float* cand_score, float* cand_box, int32_t* cand_count, cudaStream_t st);

void set_nms_blockwise(int on);     // benchmark knob "nms.blockwise"
int get_nms_blockwise();
cudaError_t launch_nms(const float* box, const float* score, const int32_t* count, int n_problems, int stride,
                       float thr, int limit, int32_t* keep_idx, int32_t* keep_count, cudaStream_t st);

// fused K1+K2 of the whole-path call: surviving root cells per (image, part), nothing else
cudaError_t launch_decode_nms(const void* head, const Geom& g, int n_parts, float det_thr, float nms_thr,
                              int32_t* keep_cell, int32_t* keep_count, cudaStream_t st, bool pdl_attr = false,
                              int pdl_bits = 0, int ctas_per_sm = 0 /* > 0: persistent grid */, int threads_pref = 0);
// shared memory left for the arg-max ring beside k12_ctas decode+NMS CTAs and one tree-parse CTA per SM (0: no room)
size_t chain3_ring_cap(const Geom& g, int stage_all_pref, int k12_ctas);

cudaError_t launch_restore_xy(const float* x, const float* y, float* rx, float* ry, size_t n, int H, int W,
                              float gridW, float gridH, cudaStream_t st);
cudaError_t launch_restore_size(const float* w, const float* h, float* rw, float* rh, size_t n, float inW, float inH,
                                cudaStream_t st);

cudaError_t launch_part_centres(const int32_t* count, const int32_t* cell, const float* box, int B, int R, int K,
                                float* centre, cudaStream_t st);

cudaError_t launch_skeleton(const int32_t* count, const int32_t* cell, const float* box, int B, int R, int K, int E,
                            const int32_t* edges /* host [E][2] */, int32_t* rect, float* keypoint, float* segment, cudaStream_t st);

cudaError_t launch_pack_humans(const int32_t* count, const int32_t* cell, const float* score, const float* box, int B, int R,
                               int K, int cap, int32_t* header, uint32_t* e_idcell, float* e_score, float* e_box,
                               cudaStream_t st);

size_t tree_parse_smem_bytes(const Geom& g, int n_groups);

cudaError_t launch_tree_parse(const void* head, const Geom& g, const ChainTable& ch, float thr, int min_kp, int n_parts,
                              const uint16_t* amax, const int32_t* cand_cell, const int32_t* keep_idx,
                              const int32_t* keep_count, int32_t* h_count, int32_t* h_root, int32_t* h_cell,
                              float* h_score, float* h_box, int R, cudaStream_t st, bool pdl_attr = false, int pdl_bits = 0,
                              int stage_all_pref = -1, int threads_pref = 0, int chain_mode = 0 /* 1, 2: a publishing link of the
                              call chain, see the launcher */, int ctas_per_sm = 0 /* > 0: persistent grid */);

// fused decode + NMS + tree parse (n_nms_parts == 1, H*W <= 1024): the whole-path call's second kernel
bool parse_fused_supported(const Geom& g, int stage_pref);
// How the overlapped two-kernel chain runs a batch: n_sub equal sub-batches of sub_B images, each small enough
// that all of its parse CTAs are resident beside one arg-max CTA per SM; ring_cap = shared memory left for the
// arg-max ring on an SM.  false: the fused kernel cannot sit beside a ring at all for this shape.
struct FusedSplit { int n_sub, sub_B; bool staged; size_t smem, ring_cap; };
bool parse_fused_split(const Geom& g, int stage_pref, const Tuning& t, FusedSplit* out);
size_t parse_fused_smem_bytes(const Geom& g, int stage_pref);
// dense (human, part) entry buffer written by the fused kernel itself (header[0..1] cleared by the arg-max kernel)
struct DenseTarget { int32_t* header; uint32_t* idcell; float* score; float* box; int32_t cap; int32_t skip_slots;
                     int32_t B_total; int32_t b0;
                     int32_t* rheader = nullptr; };   // set: idcell/score/box belong to another buffer (e.g. a peer's), whose header this is
cudaError_t launch_parse_fused(const void* head, const Geom& g, const ChainTable& ch, float det_thr, float nms_thr, int min_kp,
                               const uint16_t* amax, int32_t* h_count, int32_t* h_root, int32_t* h_cell, float* h_score,
                               float* h_box, int R, cudaStream_t st, bool pdl_attr, int chain_mode, int stage_pref,
                               int staged_forced = -1, const DenseTarget* dense_to = nullptr, bool wait_top = false);
unsigned next_call_parity(cudaStream_t st);   // which workspace half the next whole-path call on `st` takes (alternates per stream)
bool chain_clean(cudaStream_t st);      // the stream's last whole-path launch was a (publishing) fused parse
void chain_break(cudaStream_t st);      // ... was something else: the next overlapped call starts fully ordered

// ---- fused network head (ppn_head.cu): 1x1 convolution (tcgen05 GEMM) + sigmoid + limb-window arg-max ---------
// feat [B, Cin, H, W] fp32, weight [C, Cin] fp32, bias [C] or nullptr  ->  dec [B, 6K, HW] = sigmoid of the decode
// channels, amax [B, E, HW]; optional emit_logits / emit_head [B, C, HW] for parity tests (model.py:85, 133-136).
size_t head_smem_bytes();
// keys: scratch of head_keys_bytes() (the epilogue's running maxima; the launcher clears it and converts it to amax);
// subs: epilogue warps per TMEM lane quadrant (1 .. 4).  Launches: memset, [pack,] GEMM, finalize.
size_t head_keys_bytes(const Geom& g);
cudaError_t launch_head_gemm_argmax(const float* feat, const float* weight, const float* bias, int Cin, const Geom& g,
                                    float* dec, uint16_t* amax, unsigned long long* keys, float* emit_logits, float* emit_head,
                                    cudaStream_t st, bool pdl_attr, int pdl_bits, int subs);
// The 16-bit operand path: fp16 / bf16 K-major operands.  feat = fp32 NCHW (packed into `xt` [B * HW][Cin] by a
// pre-pass) or, when !feat_nchw_f32, already [B * HW][Cin] in the operand type (channels_last) and read in place;
// wt [C][Cin] receives the converted weights.  Two launches (pack, GEMM as its programmatic dependent).
bool head16_supported(int Cin, const Geom& g);
size_t head16_packed_feat_bytes(int Cin, const Geom& g);
size_t head16_packed_weight_bytes(int Cin, const Geom& g);
cudaError_t launch_head_gemm16_argmax(const void* feat, bool feat_nchw_f32, const float* weight, const float* bias, int Cin, bool bf16,
                                      const Geom& g, void* xt, void* wt, float* dec, uint16_t* amax, unsigned long long* keys,
                                      float* emit_logits, float* emit_head, cudaStream_t st, int pdl_bits, int subs);

// ---- training-target encoder (ppn_encode.cu) ----------------------------------------------------------
struct EdgeTable { uint8_t src[256]; uint8_t dst[256]; };
struct EncodeArgs {
    const int32_t* person_off;      // [B + 1]
    const double* bbox;             // [n, 4] cx, cy, w, h
    const float* keypoints;         // [n, K - 1, 2]
    const uint8_t* visible;         // [n, K - 1]
    const double* size;             // [n]
    float *delta, *weight, *tx, *ty, *tx_half, *ty_half, *tw, *th;
    void *weight_ij, *te;           // elements of limb_dtype
    int32_t limb_dtype;             // HEAD_F32, HEAD_F16 or HEAD_BF16
    int32_t K, E, H, W, sH, sW, rows_per_cta;
    int32_t small_only, sweep, sweep_ctas_per_sm;   // launcher state / tuning (encode.sweep, encode.ctas_per_sm)
    uint32_t magic_sW;              // ceil(2^32 / sW) for exact x / sW, 0 <= x < 65536 (0 when sW == 1)
    float gridW, gridH;
    double inW, inH;
    EdgeTable edges;
};
cudaError_t launch_encode_targets(EncodeArgs a, int B, int sms, cudaStream_t st);

// ---- the training loss (ppn_loss.cu): forward sums and the head gradient of the reference's PPNLoss -------------
constexpr int kLossMaxCtas = 2048;     // CTAs of the forward grid at most: the workspace holds one partial set each
struct LossArgs {
    const void* head;                   // [B, C, H, W] of head_dtype
    void* grad;                         // [B, C, H, W] of head_dtype (backward)
    const float *delta, *weight, *tx, *ty, *tx_half, *ty_half, *tw, *th;
    const void *weight_ij, *te;         // [B, E, sH, sW, H, W] of limb_dtype
    int32_t head_dtype, limb_dtype;     // HEAD_*: (F32, F32), (F16, F32 or F16), (BF16, F32 or BF16)
    const float* grad_loss;             // [5] device (backward)
    double* partial;                    // [grid][5] workspace (forward)
    int32_t B, K, W, HW, L;             // L = E * sH * sW * H * W limb elements per image
    size_t img_stride, limb_off;        // C * HW, 6 * K * HW
    float gW, gH, inW, inH;
    long long small_items, limb_chunks, n_items;   // filled by loss_plan
};
void loss_plan(LossArgs* a);
size_t loss_workspace_bytes(const LossArgs& a);
// two launches: the streaming kernel (CTA partials into a.partial), then the fixed-order sum into loss[5].
// from_logits: a.head holds the logits; the kernels apply sigmoid_f32 to every head element and the sigmoid's
// derivative to every gradient element (ppn_loss.cu)
cudaError_t launch_loss_forward(LossArgs a, float* loss, int sms, cudaStream_t st, bool from_logits = false);
cudaError_t launch_loss_backward(LossArgs a, int sms, cudaStream_t st, bool from_logits = false);
// y[i] = sigmoid_f32(x[i]) for x of HeadDtype `dtype`, y fp32 (ppn_sigmoid)
cudaError_t launch_sigmoid(const void* x, int dtype, float* y, size_t n, cudaStream_t st);

}  // namespace ppn
