/*
 * libppn_decode — C ABI of the B200 (sm_100a) Pose Proposal Network output parser.
 *
 * The reference (noirmist/Pytorch_Pose_Proposal_Network) has no FFI or plugin layer: its
 * "operator API" for this path is four module-level Python functions plus the head-tensor
 * layout.  Each entry point below names the reference interface it stands in for
 * (paths under /root/reference):
 *
 *   ppn_limb_argmax ........ the np.argmax of every limb window, datatest.py:100,113
 *   ppn_decode_candidates .. resp*conf, restore_xy/restore_size, box assembly and
 *                            np.where(score > thresh): rt_test.py:130, datatest.py:63-71,80-92
 *   ppn_restore_xy/_size ... restore_xy(x, y) / restore_size(w, h), datatest.py:63-71
 *   ppn_nms ................ non_maximum_suppression(bbox, thresh, score, limit), datatest.py:134-160
 *   ppn_tree_parse ......... the per-root walk of get_humans_by_feature, datatest.py:103-131
 *   ppn_part_centres ....... box -> keypoint of draw_humans / evaluation, datatest.py:200-211, 314-317
 *   ppn_skeleton ........... everything draw_humans computes before it draws: root rectangles, keypoints, limb
 *                            segments, datatest.py:162-232
 *   ppn_parse .............. get_humans_by_feature end to end on a device batch: what
 *                            rt_test.py:109-133 / main.py:946-972 do per image after model(image)
 *   ppn_parse_proposals .... not the reference's parse: per-part proposals, limb scores of candidate pairs and a
 *                            greedy tree parse in which humans compete for parts (the paper's form, DESIGN.md §13)
 *   ppn_parse_host ......... the same from host memory (the reference's numpy arrays), with the
 *                            copies the reference's `.cpu()` calls stand for done here in reverse
 *   ppn_parse_dense ........ ppn_parse that also emits dense (human, part) records (what a multi-GPU job gathers)
 *   ppn_parse_dense_remote . the same with the records stored straight into a peer GPU's buffer over NVLink
 *   ppn_head_parse ......... the network's last layer fused in: conv3 (1x1) + sigmoid, model.py:85,133-136, then
 *                            the whole parse, without the head tensor ever reaching memory
 *   ppn_encode_targets ..... the inverse of the path: the "# Encode samples" half of
 *                            KeypointsDataset.__getitem__, dataset.py:89-198, for a whole batch
 *   ppn_loss_forward ....... the consumer of those targets: PPNLoss.forward, main.py:125-216 (five terms)
 *   ppn_loss_backward ...... its autograd backward with respect to the head tensor
 *   ppn_loss_*_opt ......... the same for fp16 / bf16 heads and limb targets (mixed-precision training)
 *   ppn_loss_*_logits ...... the same on the conv output before model.py's final sigmoid, the sigmoid fused in
 *   ppn_sigmoid ............ that sigmoid alone, elementwise (model.py:136 with the loss's exact values)
 *   ppn_ap_match ........... the validation pass's scoring, per image: poseval's eval_helpers.assignGTmulti
 *   ppn_ap_finalize ........ ... and over the pass: evaluateAP.computeMetrics (computeRPC, VOCap)
 *   ppn_flip_merge ......... the flip test: a head averaged with the mirrored head of its flipped input (§15)
 *
 * Conventions
 *   - plain C: pointers and sizes only; no CUDA or torch types.  `stream` is a cudaStream_t
 *     passed as void* (NULL = the legacy default stream).
 *   - every function returns int: 0 = ok, > 0 = a cudaError_t value, < 0 = a PPN_E_* code;
 *     ppn_strerror() turns either into text.  Nothing throws across the boundary.
 *   - device entry points only ENQUEUE work on `stream`; they never synchronise and never
 *     allocate (one exception: 2 KB of work counters per device on the very first launch).  The caller owns every buffer (torch tensors in the Python host layer) and
 *     selects the device (cudaSetDevice / torch.cuda.set_device) before calling.
 *   - thread-safe for distinct streams and buffers.  The only global mutable state is the benchmark tuning
 *     table of include/ppn_decode_bench.h (not part of this interface); every call works on one snapshot of it.
 *   - head tensor: fp32 (or fp16 / bf16, PPNShape.head_dtype), NCHW contiguous [B, 6K + sH*sW*E, H, W]; channel groups resp, conf,
 *     x, y, w, h (K each) then the limb block viewed as [E, sH, sW, H, W] (model.py:64,
 *     rt_test.py:109-120).  16-byte aligned base.
 *   - cells are flat indices h*W + w; boxes are (ymin, xmin, ymax, xmax) in pixels.
 *   - all floating-point results are bit-identical to numpy's fp32 evaluation of the
 *     reference's expressions (single rounding per operation, no FMA contraction).
 */
#ifndef PPN_DECODE_H_
#define PPN_DECODE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PPN_ABI_VERSION 7

/* library error codes (negative); positive return values are cudaError_t */
#define PPN_OK               0
#define PPN_E_BADARG        -1   /* NULL pointer, non-positive size, misaligned base            */
#define PPN_E_UNSUPPORTED   -2   /* shape outside what the kernels handle (see ppn_limits)      */
#define PPN_E_WORKSPACE     -3   /* workspace smaller than ppn_workspace_bytes()                */
#define PPN_E_CHAINS        -4   /* track orders too long / indexes outside K or E              */
#define PPN_E_NO_DEVICE     -5   /* no CUDA device, or not an sm_100 class device               */

#define PPN_MAX_CHAINS       32  /* track orders (config.py:67-73 has 5)                        */
#define PPN_MAX_CHAIN_STEPS 192  /* total limb steps over all track orders (reference: 25)      */
#define PPN_MAX_CELLS      1024  /* H*W handled by the in-shared-memory NMS and parse kernels   */

/* Geometry of one head tensor.  Mirrors the module globals of datatest.py:53-60 and the
 * attributes of PoseProposalNet (model.py:54-64). */
typedef struct PPNShape {
    int32_t B;              /* images in the batch                                              */
    int32_t K, E;           /* parts (incl. 'instance' = part 0), limbs                          */
    int32_t H, W;           /* grid: outH, outW                                                  */
    int32_t sH, sW;         /* limb displacement window                                          */
    int32_t inW, inH;       /* network input size in pixels                                      */
    int32_t gridW, gridH;   /* int(inW/outW), int(inH/outH)  (datatest.py:60)                    */
    int32_t off_h, off_w;   /* half-windows subtracted from row / column (datatest.py:115-116)   */
    int32_t head_dtype;     /* PPN_HEAD_F32 (the reference's), PPN_HEAD_F16 or PPN_HEAD_BF16          */
} PPNShape;

/* Element type of the head tensor.  A 16-bit head halves the HBM traffic of the path; every
 * element is widened to fp32 exactly when loaded and all arithmetic stays the reference's fp32,
 * so the result is the reference's on head.float(). */
#define PPN_HEAD_F32  0
#define PPN_HEAD_F16  1
#define PPN_HEAD_BF16 2

/* Thresholds and the track orders (config.py:67-80 DIRECTED_GRAPHS, flattened).  The three
 * chain arrays are HOST pointers; they are copied into kernel arguments at launch. */
typedef struct PPNParams {
    float   det_thresh;         /* 0.15 at rt_test.py:133; root: delta > thr, limb target: delta >= thr */
    float   nms_thresh;         /* 0.3 at datatest.py:94; IoU >= thr suppresses                  */
    int32_t min_num_keypoints;  /* datatest.py:74,129                                            */
    int32_t n_nms_parts;        /* parts 0..n-1 get a compacted candidate list and NMS; the
                                   reference uses only part 0 (datatest.py:86-94) => 1           */
    int32_t n_chains;
    int32_t flags;              /* PPN_FLAG_* , 0 = none                                         */
    const int32_t* chain_off;   /* [n_chains + 1]                                                */
    const int32_t* chain_limb;  /* [chain_off[n_chains]] limb index of each step  ("eis")        */
    const int32_t* chain_part;  /* [chain_off[n_chains]] target part of each step ("ts")         */
} PPNParams;

/* ppn_parse only.  The caller vouches that the head tensor was completely written before the call
 * was enqueued (it is resident from an earlier, already completed step, or was followed by a
 * synchronisation) — NOT merely ordered before it on the stream by a still-running producer kernel.
 * Then the call's arg-max and decode kernels may start while the previous ppn_parse on the same
 * stream is still in its tree parse; results still complete in call order. */
#define PPN_FLAG_INPUT_COMPLETE 1
/* Slots [count[b], R) of the result normally keep whatever the caller's buffers held.  With this flag the call
 * first clears the result arrays on the stream (root_cell / part_cell = -1, scores and boxes = 0), so that a
 * consumer may scan all R slots.  Costs one pass over the result arrays and orders the call after the memsets
 * (consecutive calls no longer overlap).  Honoured by ppn_parse, ppn_parse_dense (unless skip_slots), ppn_parse_host
 * (the host slots no copy reaches are cleared on the host) and ppn_head_parse[_opt]; it combines with
 * PPN_FLAG_INPUT_COMPLETE. */
#define PPN_FLAG_CLEAR_UNUSED 2

/* Packed result, device memory owned by the caller.  Humans of image b occupy slots
 * [0, min(count[b], R)) in descending root-score (NMS) order, as the reference's list is. */
typedef struct PPNHumans {
    int32_t* count;        /* [B]        humans found (may exceed R: only the first R are stored) */
    int32_t* root_cell;    /* [B, R]                                                             */
    int32_t* part_cell;    /* [B, R, K]  cell of part k, -1 = absent; part 0 = root               */
    float*   part_score;   /* [B, R, K]  delta at that cell (0 where absent)                      */
    float*   part_box;     /* [B, R, K, 4] (ymin, xmin, ymax, xmax) (0 where absent)              */
    int32_t  R;            /* slots per image; H*W can never overflow                             */
} PPNHumans;

int         ppn_abi_version(void);
const char* ppn_strerror(int code);

/* Bytes of scratch ppn_parse needs for this shape: two sets of (arg-max map, surviving root cells,
 * counts), used alternately by successive calls on the same workspace. */
int ppn_workspace_bytes(const PPNShape* shape, const PPNParams* params, size_t* bytes);

/* Number of kernel launches one ppn_parse call enqueues for this shape. */
int ppn_parse_launches(const PPNShape* shape, const PPNParams* params);

/* How ppn_parse will run this shape: info[4] = {kernel launches, sub-batches of the two-kernel chain, shared-memory
 * bytes the arg-max ring is capped to so that the parse CTAs fit beside it (0 = uncapped), 1 if delta is staged}. */
int ppn_parse_plan(const PPNShape* shape, const PPNParams* params, int32_t* info /*[4]*/);

/* amax[B, E, H*W] (uint16) = index in [0, sH*sW) of the FIRST maximum of each limb window;
 * NaN counts as the maximum (numpy argmax).  Streams the limb block once. */
int ppn_limb_argmax(const void* head, const PPNShape* shape, uint16_t* amax, void* stream);

/* Measurement aid: the SAME bulk-copy ring as ppn_limb_argmax moving the same bytes through shared memory, but
 * the consumers only release the stages — no compares, nothing written.  Its duration is the read ceiling of this
 * access pattern on this GPU (bench.py: roofline.read_peak_gbs).  smem_cap > 0 bounds the ring like ppn_parse does
 * when the parse kernel's CTAs must fit beside it.  `amax` is not written (pass the buffer a real call would get). */
int ppn_limb_stream_probe(const void* head, const PPNShape* shape, uint16_t* amax, int32_t smem_cap, void* stream);

/* For parts 0..n_parts-1 of every image: cells with resp*conf > det_thresh in ascending cell
 * order, with score and box.  Lists are [B, n_parts, H*W]; cand_count is [B, n_parts]. */
int ppn_decode_candidates(const void* head, const PPNShape* shape, int32_t n_parts, float det_thresh,
                          int32_t* cand_cell, float* cand_score, float* cand_box, int32_t* cand_count,
                          void* stream);

/* restore_xy(x, y) and restore_size(w, h) of datatest.py:63-71 as operators over n_planes
 * contiguous [H, W] planes: rx = (x + col) * gridW, ry = (y + row) * gridH; rw = inW*w, rh = inH*h. */
int ppn_restore_xy(const float* x, const float* y, float* rx, float* ry, int64_t n_planes,
                   const PPNShape* shape, void* stream);
int ppn_restore_size(const float* w, const float* h, float* rw, float* rh, int64_t n_planes,
                     const PPNShape* shape, void* stream);

/* Greedy IoU suppression of n_problems independent box lists laid out with `stride` slots
 * each: box [n_problems, stride, 4], score [n_problems, stride] or NULL (keep input order),
 * count [n_problems] (device).  keep_idx [n_problems, stride] receives indices into each list
 * in visiting order (descending score; equal scores: larger index first), keep_count
 * [n_problems] how many.  limit <= 0 means no limit.  stride <= PPN_MAX_CELLS uses the
 * shared-memory kernel; larger lists take a slower global-memory kernel. */
int ppn_nms(const float* box, const float* score, const int32_t* count, int32_t n_problems,
            int32_t stride, float nms_thresh, int32_t limit,
            int32_t* keep_idx, int32_t* keep_count, void* stream);

/* Walk the track orders from every surviving root of part 0.  cand_cell/keep_idx/keep_count
 * are the outputs of the two calls above with params->n_nms_parts lists per image; with
 * cand_cell == NULL, keep_idx holds root CELLS directly instead of indices into cand_cell. */
int ppn_tree_parse(const void* head, const PPNShape* shape, const PPNParams* params,
                   const uint16_t* amax, const int32_t* cand_cell, const int32_t* keep_idx,
                   const int32_t* keep_count, const PPNHumans* out, void* stream);

/* The whole path on a device batch in three launches on `stream`: decode+NMS fused in one kernel
 * (candidates stay in shared memory), the limb arg-max started beside it, and the tree parse,
 * chained by programmatic dependent launch so that each kernel's start-up hides under its
 * predecessor.  Results are identical to calling the four stage functions above in sequence. */
int ppn_parse(const void* head, const PPNShape* shape, const PPNParams* params,
              const PPNHumans* out, void* workspace, size_t workspace_bytes, void* stream);

/* ---- proposal-pair parse: humans compete for parts (DESIGN.md §13) -------------------------------------------
 * A second parser over the same head tensor and the same PPNHumans layout.  ppn_parse follows the reference: NMS on
 * part 0 only, then from each root the arg-max of every limb window, so several humans may hold the same part cell.
 * This one gives every part proposals and matches them greedily down the skeleton tree.  For one image:
 *   1. proposals: for EVERY part k, the cells with delta[k] > det_thresh (strict), through ppn_nms's greedy IoU
 *      suppression (IoU >= nms_thresh; equal scores: larger cell first).  The survivors P_k keep NMS order;
 *   2. human i is the i-th proposal of P_0, rooted at that cell;
 *   3. the track orders must form a tree rooted at part 0: every target part reached by one limb from one
 *      predecessor, part 0 never a target (PPN_E_CHAINS otherwise).  Parts are matched in first-reach order;
 *   4. limb e = (s -> t) pairs the part-s cell a of every human that has part s with every b in P_t whose
 *      displacement dy = row(b) - row(a) + off_h, dx = col(b) - col(a) + off_w lies in the window (0 <= dy < sH,
 *      0 <= dx < sW).  Score sc = (delta[s, a] * lv) * delta[t, b], lv = head[6K + (e*sH + dy)*sW + dx, a], each
 *      product rounded once; the pair is a candidate iff sc > 0 (NaN, zero and negative limb values never connect);
 *   5. candidates in order of sc descending, then smaller human index, then smaller cell; a pair is accepted when
 *      its human has no part t yet and b is unused;
 *   6. humans stay in root NMS order; those with at least min_num_keypoints non-root parts are kept (after the
 *      matching: a dropped human's parts go to no one).  part_score / part_box of a present part are those ppn_parse
 *      computes for that cell; count[b] may exceed R, only the first R humans are stored.
 * No part instance belongs to two humans, and every present part's parent is present.
 * params->n_nms_parts is not read (every part is NMSed).  Among the flags only PPN_FLAG_CLEAR_UNUSED is honoured;
 * calls are stream-ordered (no overlap with the previous call).  Needs K <= 64 and H*W <= PPN_MAX_CELLS
 * (PPN_E_UNSUPPORTED beyond).  Two kernels: decode + NMS of every (image, part), and the pair-scoring + matching
 * kernel as its programmatic dependent; no host synchronisation, capturable in a CUDA graph.
 *   ppn_parse_proposals_workspace_bytes: scratch for the per-part survivor lists (256-byte aligned workspace). */
int ppn_parse_proposals_workspace_bytes(const PPNShape* shape, const PPNParams* params, size_t* bytes);
int ppn_parse_proposals(const void* head, const PPNShape* shape, const PPNParams* params, const PPNHumans* out,
                        void* workspace, size_t workspace_bytes, void* stream);

/* The whole path from HOST memory (pinned for full speed): uploads `head` in chunks
 * overlapped with the kernels, runs ppn_parse, downloads the packed result into the HOST
 * arrays of `out_host`.  Synchronous.  dev_scratch/dev_scratch_bytes: device memory of at
 * least ppn_parse_host_scratch_bytes().  Of every image only the first m = max_b min(count[b], R) slots are copied
 * back: slots [count[b], m) receive the device's unused slots, and slots [m, R) keep their host bytes.  With
 * PPN_FLAG_CLEAR_UNUSED every slot from count[b] on reads -1 / 0 (slots [m, R) are cleared on the host). */
int ppn_parse_host_scratch_bytes(const PPNShape* shape, const PPNParams* params, int32_t R, size_t* bytes);
int ppn_parse_host(const void* head_host, const PPNShape* shape, const PPNParams* params,
                   const PPNHumans* out_host, void* dev_scratch, size_t dev_scratch_bytes);

/* Centre of every part's box, centre_yx[B, R, K, 2] = ((ymin + ymax) / 2, (xmin + xmax) / 2), (0, 0)
 * for absent parts and unused slots: what the code right after the path reads off the boxes — the
 * keypoints drawn by draw_humans (datatest.py:200-211) and the x / y of the AP-evaluation records
 * (datatest.py:314-317).  Same fp32 arithmetic as numpy's. */
int ppn_part_centres(const PPNHumans* humans, int32_t B, int32_t K, float* centre_yx, void* stream);

/* The drawing primitives of draw_humans (datatest.py:162-232; the webcam loop calls it right after the parser,
 * rt_test.py:138-145) for every slot of a packed result, so that the consumer draws without touching per-human
 * dicts:  rect [B, R, 4] int32 = the root box as drawn, (xmin, ymin, xmax, ymax) truncated like int()
 * (datatest.py:177-181);  keypoint_xy [B, R, K, 2] fp32 = (x, y) centre of every present part (:200-202);
 * segment [B, R, E, 4] fp32 = (bx, by, ex, ey) of every limb whose two parts are present (:213-221).  Absent
 * parts / limbs and unused slots: NaN (rect: 0).  edges: HOST [E][2] part ids (config.py:65 EDGES). */
int ppn_skeleton(const PPNHumans* humans, int32_t B, int32_t K, int32_t E, const int32_t* edges,
                 int32_t* rect, float* keypoint_xy, float* segment, void* stream);

/* Dense pose ENTRIES for shipping results (the multi-GPU gather): one contiguous device buffer
 *   int32  header[2 + 3B] = {total entries, overflow flag, count[B] humans, entries[B] per image,
 *                            start[B] first entry of each image}
 *   uint32 idcell[cap]    = part id << 16 | cell      float score[cap]      float box[cap][4]
 * (256-byte aligned blocks).  One entry per PRESENT part; a human's root (part 0) is its first
 * entry, so an entry with part id 0 starts a new human and the list needs no per-human table.
 * An image's entries are contiguous, humans in result order; ppn_pack_humans lays the images out
 * in order (start[b] = sum_{i<b} entries[i]), ppn_parse_dense in any order.  An image whose block
 * would end beyond `cap_entries` is not written and the overflow flag is set.  ppn_packed_bytes
 * gives the buffer size and, if `offsets` != NULL, the byte offsets of {header, idcell, score, box}. */
int ppn_packed_bytes(int32_t B, int32_t cap_entries, size_t* bytes, size_t* offsets /*[4] or NULL*/);
int ppn_pack_humans(const PPNHumans* humans, int32_t B, int32_t K, int32_t cap_entries,
                    void* packed, size_t packed_bytes, void* stream);

/* ppn_parse that also produces the dense entry buffer `packed` (ppn_packed_bytes(B, cap_entries)).
 * On the default two-kernel path the parse kernel writes the entries itself, straight from shared
 * memory — no pack kernel, no second pass over the fixed-stride arrays, and nothing but kernels on
 * the stream, so consecutive PPN_FLAG_INPUT_COMPLETE calls stay overlapped; otherwise (several NMS
 * parts, more than 32 parts, grids the fused kernel does not take) it is ppn_parse followed by
 * ppn_pack_humans.  `out` is always required (count[] is always written); skip_slots != 0 says the
 * caller does not need root_cell / part_cell / part_score / part_box, which the two-kernel path
 * then leaves untouched.  Consecutive overlapping calls need different `packed` buffers, like `out`. */
int ppn_parse_dense(const void* head, const PPNShape* shape, const PPNParams* params, const PPNHumans* out,
                    void* packed, size_t packed_bytes, int32_t cap_entries, int32_t skip_slots,
                    void* workspace, size_t workspace_bytes, void* stream);

/* ---- multi-GPU pose gather over peer memory (SURVEY §8e) ----------------------------------------------
 * Images are sharded over the GPUs of one box with no data-path collective; what has to travel is each rank's
 * poses.  ppn_parse_dense_remote is ppn_parse_dense whose entry stores go to ANOTHER buffer of the same layout —
 * typically the gather root's, mapped into this process over NVLink (ppn_peer_open) — straight from the parse
 * kernel: `remote_packed` receives the per-image table {count, entries, start} and the idcell / score / box
 * entries (plain stores; nothing is read back, the block cursor stays in `local_header`), so the gather costs no
 * extra kernel, copy or collective on the compute stream.  header[0..1] of the remote buffer are not written: the
 * reader derives the total as sum(entries) and overflow as any(start + entries > cap_entries).  Only where the
 * fused parse kernel writes the entries itself (n_nms_parts == 1, K <= 32, H*W <= PPN_MAX_CELLS and a batch the
 * two-kernel chain takes): PPN_E_UNSUPPORTED otherwise.  `local_header`: >= 4 * (2 + 3B) bytes, 256-byte aligned.
 *
 * ppn_peer_alloc / _open / _close / _free wrap cudaMalloc + cudaIpcGetMemHandle and cudaIpcOpenMemHandle (which
 * enables peer access) so that the host layer can exchange the 64-byte handle through its process group
 * (torch.distributed) and hand the kernels raw peer pointers; ppn_peer_copy is one cudaMemcpyAsync (direction
 * inferred from the pointers; copy engine, no SM) — between two such buffers for gather variants that ship a group
 * of steps at a time, or into pinned host memory to read the root's buffer. */
#define PPN_IPC_HANDLE_BYTES 64
int ppn_peer_alloc(size_t bytes, void** dev_ptr, unsigned char* handle /*[64]*/);
int ppn_peer_open(const unsigned char* handle /*[64]*/, void** dev_ptr);
int ppn_peer_close(void* dev_ptr);
int ppn_peer_free(void* dev_ptr);
int ppn_peer_copy(void* dst, const void* src, size_t bytes, void* stream);
/* Landing flags of the gather, without a collective: ppn_peer_post stores `value` (release, system scope) into a
 * 64-bit counter — this rank's, in the ROOT's buffer — behind everything enqueued on `stream` so far (a one-thread
 * kernel, launched fully ordered: the parse kernels before it have completed, so their records have landed);
 * ppn_peer_wait makes `stream` wait until all `n` counters have reached `target` (one polling warp per 32 counters,
 * acquire loads at system scope; after `timeout_ms` it gives up and sets *timed_out, a device int32, so that a dead
 * peer cannot hang the stream).  What the reference would do with a blocking gather after its loop
 * (main.py:240-245 is its only use of the process group) costs one 8-byte store per rank here. */
int ppn_peer_post(void* counter, long long value, void* stream);
int ppn_peer_wait(const void* counters, int32_t n, long long target, uint32_t timeout_ms, int32_t* timed_out, void* stream);
int ppn_parse_dense_remote(const void* head, const PPNShape* shape, const PPNParams* params, const PPNHumans* out,
                           void* local_header, size_t local_header_bytes, void* remote_packed, size_t remote_bytes,
                           int32_t cap_entries, int32_t skip_slots, void* workspace, size_t workspace_bytes, void* stream);

/* ---- the network head fused in (SURVEY §8f row 1) ---------------------------------------------------
 * Replaces `conv3_out = self.conv3(lRelu2); out = self.sigmoid(conv3_out)` (model.py:133-136) TOGETHER with the
 * parse of `out`: feat = lRelu2 [B, Cin, H, W] fp32 NCHW contiguous (Cin = 512, model.py:85), weight = conv3.weight
 * viewed as [C, Cin] fp32, bias = conv3.bias [C] or NULL; C = 6K + sH*sW*E.  The 1x1 convolution runs on the
 * tensor cores in TF32 with fp32 accumulation (what cuDNN does for the reference under PyTorch's defaults); the
 * sigmoid and numpy's first-maximum rule are applied to the accumulators in the GEMM epilogue, so only the 6K
 * decode planes and the uint16 arg-max map are written — never the [B, C, H, W] head tensor.
 *   ppn_head_gemm_argmax: that kernel alone.  dec [B, 6K, H*W] fp32 = sigmoid of the decode channels, amax
 *       [B, E, H*W]; emit_logits / emit_head (each NULL or [B, C, H*W] fp32) additionally receive the convolution
 *       output and its sigmoid — the reference's head tensor — for parity checks.
 *   ppn_head_parse: the kernel above, then the fused decode + NMS + tree parse on its output.  Results are
 *       bit-identical to ppn_parse on the tensor emit_head would hold, PPN_FLAG_CLEAR_UNUSED included (the
 *       result arrays are cleared before the first head kernel).  Needs Cin % 32 == 0, H*W % 4 == 0,
 *       H*W <= PPN_MAX_CELLS, n_nms_parts == 1 and 16-byte aligned feat / weight: PPN_E_UNSUPPORTED otherwise. */
int ppn_head_workspace_bytes(const PPNShape* shape, size_t* bytes);
int ppn_head_gemm_argmax(const float* feat, const float* weight, const float* bias, int32_t Cin, const PPNShape* shape,
                         float* dec, uint16_t* amax, float* emit_logits, float* emit_head, void* stream);
int ppn_head_parse(const float* feat, const float* weight, const float* bias, int32_t Cin, const PPNShape* shape,
                   const PPNParams* params, const PPNHumans* out, void* workspace, size_t workspace_bytes,
                   float* emit_logits, float* emit_head, void* stream);

/* The same with a choice of tensor-core operand type and activation layout.
 *   operand      PPN_GEMM_TF32: as above (fp32 NCHW activations read in place).
 *                PPN_GEMM_F16 / PPN_GEMM_BF16: operands rounded to fp16 / bf16 (round to nearest even), products
 *                accumulated in fp32 — what the reference's conv3 computes under its apex AMP training setup
 *                (main.py:282-289).  fp16 keeps TF32's 10 mantissa bits (activations beyond +-65504 overflow);
 *                bf16 keeps fp32's range with 7.  Twice the tensor-core rate on half the operand bytes.
 *   feat_layout  PPN_FEAT_NCHW_F32: feat is fp32 [B, Cin, H, W]; for a 16-bit operand a pre-pass kernel packs it to
 *                [B*H*W, Cin] in the workspace (one extra read of feat, one 16-bit write).
 *                PPN_FEAT_NHWC_16: feat already is [B, H, W, Cin] in the operand type (a channels_last tensor of
 *                an autocast network): read in place, no pre-pass.  16-bit operands only.
 * The 16-bit path needs 64 <= Cin <= 512, Cin % 64 == 0 (conv3 has Cin = 512): PPN_E_UNSUPPORTED otherwise.
 * Everything downstream of the logits is exact as above: results are bit-identical to ppn_parse on emit_head.
 * `workspace` (ppn_head_workspace_bytes_opt, 256-byte aligned) holds dec, amax and the packed operands;
 * ppn_head_gemm_argmax_opt writes dec / amax to the caller's buffers and uses the workspace for the packed
 * operands only (it may be NULL for PPN_GEMM_TF32). */
#define PPN_GEMM_TF32      0
#define PPN_GEMM_F16       1
#define PPN_GEMM_BF16      2
#define PPN_FEAT_NCHW_F32  0
#define PPN_FEAT_NHWC_16   1
typedef struct PPNHeadOptions {
    int32_t operand;        /* PPN_GEMM_*                                                           */
    int32_t feat_layout;    /* PPN_FEAT_*                                                           */
} PPNHeadOptions;
int ppn_head_workspace_bytes_opt(const PPNShape* shape, int32_t Cin, const PPNHeadOptions* opt, size_t* bytes);
int ppn_head_gemm_argmax_opt(const void* feat, const float* weight, const float* bias, int32_t Cin, const PPNShape* shape,
                             const PPNHeadOptions* opt, void* workspace, size_t workspace_bytes,
                             float* dec, uint16_t* amax, float* emit_logits, float* emit_head, void* stream);
int ppn_head_parse_opt(const void* feat, const float* weight, const float* bias, int32_t Cin, const PPNShape* shape,
                       const PPNParams* params, const PPNHeadOptions* opt, const PPNHumans* out, void* workspace,
                       size_t workspace_bytes, float* emit_logits, float* emit_head, void* stream);

/* ---- the inverse of the parser: training targets from annotations ------------------------------
 * Replaces the "# Encode samples" half of KeypointsDataset.__getitem__ (dataset.py:89-198) for a whole
 * batch.  People of image b are rows [person_off[b], person_off[b+1]) of the four arrays, in the
 * reference's post-transform types (aug.py:138-160): bbox float64 (cx, cy, w, h), keypoints fp32
 * (x, y) of parts 1..K-1, visible 0/1 bytes, size float64 (side of a part's box).  All DEVICE pointers. */
typedef struct PPNPeople {
    const int32_t* person_off;  /* [B + 1]                                                          */
    const double*  bbox;        /* [n, 4]                                                           */
    const float*   keypoints;   /* [n, K - 1, 2]                                                    */
    const uint8_t* visible;     /* [n, K - 1]                                                       */
    const double*  size;        /* [n]                                                              */
} PPNPeople;

/* The ten grids __getitem__ returns after the image (dataset.py:198), batched, fp32, caller-owned
 * device memory: [B, K, H, W] each, except weight_ij and te: [B, E, sH, sW, H, W]. */
typedef struct PPNTargets {
    float *delta, *weight, *weight_ij, *tx, *ty, *tx_half, *ty_half, *tw, *th, *te;
} PPNTargets;

/* edges: HOST array [E][2] of (source part, target part) (config.py:65 EDGES).  Every output element is
 * written (no pre-zeroing needed).  Same arithmetic as the reference (fp32 cell division and offsets,
 * float64 size division rounded once), people applied in order (later ones overwrite).  Like the
 * reference's window slicing (dataset.py:163-167) it needs an odd square limb window:
 * PPN_E_UNSUPPORTED otherwise. */
int ppn_encode_targets(const PPNPeople* people, const PPNShape* shape, const int32_t* edges,
                       const PPNTargets* out, void* stream);

/* ---- the training loss over the head tensor and the encoded targets --------------------------------
 * Stands in for the reference's criterion PPNLoss (main.py:125-216), called as criterion(output, delta, weight,
 * weight_ij, tx_half, ty_half, tx, ty, tw, th, te) in its training loop.  The reference tree is not part of this
 * project: the specification is the float64 restatement documented in DESIGN.md §11 (IoU differentiable in x, y, w,
 * h; eps = 1e-6 in the IoU denominator; L_resp unweighted), not bit parity with main.py.  For image b:
 *   L_resp = sum (resp - delta)^2          L_iou = sum delta (conf - iou)^2
 *   L_coor = sum weight ((x - tx_half)^2 + (y - ty_half)^2)
 *   L_size = sum weight ((sqrt(w + eps) - sqrt(tw + eps))^2 + (sqrt(h + eps) - sqrt(th + eps))^2)
 *   L_limb = sum weight_ij (e - te)^2
 * over every element of the image, then averaged over the batch (sum / B).  The five terms stay separate: the
 * reference weights them by GradNorm (main.py:704-708), so weighting is the caller's.
 * head: fp32 [B, C, H, W] (PPN_HEAD_F32 only: PPN_E_UNSUPPORTED otherwise); `targets` as ppn_encode_targets writes
 * them (read only).  Every pointer needs 4-byte alignment; the limb block is streamed with 128-bit accesses wherever
 * the tensors of an image share their phase within 16 bytes.  B >= 1.
 *   ppn_loss_workspace_bytes: scratch of ppn_loss_forward for this shape (per-CTA partial sums; 8-byte aligned).
 *   ppn_loss_forward:  loss[5] (device fp32) = (L_resp, L_iou, L_coor, L_size, L_limb).  Deterministic: fp64
 *                      partials reduced in a fixed order, no float atomics.
 *   ppn_loss_backward: grad_head [B, C, H, W] (device fp32, every element written) = sum_t grad_loss[t] * dL_t/dhead,
 *                      grad_loss[5] a DEVICE array (never read by the host).  Recomputes from the inputs; torch's
 *                      conventions at kinks: relu'(0) = 0, a tie in min / max splits the gradient evenly.  The fp32
 *                      operation order is documented in csrc/ppn_loss.cu. */
int ppn_loss_workspace_bytes(const PPNShape* shape, size_t* bytes);
int ppn_loss_forward(const float* head, const PPNShape* shape, const PPNTargets* targets, float* loss,
                     void* workspace, size_t workspace_bytes, void* stream);
int ppn_loss_backward(const float* head, const PPNShape* shape, const PPNTargets* targets, const float* grad_loss,
                      float* grad_head, void* stream);

/* ---- mixed precision: 16-bit heads and limb targets (the reference trains under apex AMP, main.py:282-289) -------
 * The same loss with shape->head_dtype selecting the element type of the head AND of grad_head, and
 * opt->limb_dtype (a PPN_HEAD_* code) that of targets->te and targets->weight_ij: with a 16-bit limb_dtype those two
 * pointers point to fp16 / bf16 elements (despite their float* type).  The eight [B, K, H, W] targets stay fp32.
 * Supported (head, limb targets): (F32, F32), (F16, F32), (F16, F16), (BF16, F32), (BF16, BF16); any other pair
 * (an fp32 head with 16-bit limb targets, limb targets in the other 16-bit type) is PPN_E_UNSUPPORTED, a limb_dtype
 * that is no PPN_HEAD_* code PPN_E_BADARG.
 * Rule: a 16-bit input is widened exactly and the fp32 loss above is applied to it, operation for operation; every
 * gradient element is rounded once (round to nearest even) to the head's type, overflow giving +-inf.  So the terms
 * equal ppn_loss_forward on the widened inputs up to the order of the fp64 sums, and grad_head equals
 * ppn_loss_backward on the widened inputs converted to the head's type, bit for bit.
 * Pointers need the alignment of their element (2 bytes for 16-bit, 4 for fp32).  The workspace is the same as for
 * the fp32 loss of the same batch.  The three fp32 exports above keep rejecting 16-bit shapes. */
typedef struct PPNLossOptions {
    int32_t limb_dtype;     /* PPN_HEAD_F32, PPN_HEAD_F16 or PPN_HEAD_BF16: element type of te and weight_ij   */
} PPNLossOptions;
int ppn_loss_workspace_bytes_opt(const PPNShape* shape, const PPNLossOptions* opt, size_t* bytes);
int ppn_loss_forward_opt(const void* head, const PPNShape* shape, const PPNTargets* targets, const PPNLossOptions* opt,
                         float* loss, void* workspace, size_t workspace_bytes, void* stream);
int ppn_loss_backward_opt(const void* head, const PPNShape* shape, const PPNTargets* targets, const PPNLossOptions* opt,
                          const float* grad_loss, void* grad_head, void* stream);

/* ppn_encode_targets writing te and weight_ij as limb_dtype (PPN_HEAD_*; PPN_E_BADARG otherwise): te in {0, 1} is
 * exact in every type; weight_ij in {1, 0.0005f} stores 0.0005f rounded to nearest even (fp16 0.000500202...,
 * bf16 0.000499725...).  The eight small grids are fp32 as above; shape->head_dtype is not used. */
int ppn_encode_targets_opt(const PPNPeople* people, const PPNShape* shape, const int32_t* edges,
                           const PPNTargets* out, int32_t limb_dtype, void* stream);

/* ---- the loss on logits: the network's final sigmoid fused into the loss (BCEWithLogitsLoss style) ----------
 * `logits` is the conv output BEFORE model.py's sigmoid (model.py:133-136), laid out like the head tensor, and every
 * one of its C channels (resp, conf, x, y, w, h and the limb block) is taken through
 *   s = 1 / (1 + expf(-x))          fp32: libdevice expf, one add, one IEEE division (-inf gives 0, +inf gives 1)
 * after a 16-bit logit is widened exactly.  The loss above is then applied to s, operation for operation; s stays
 * fp32 (it is not rounded to the head's type).  With g_s the fp32 gradient ppn_loss_backward_opt forms for s,
 *   grad_logits = (g_s * (1 - s)) * s                   (each operation rounded once: torch's sigmoid_backward)
 * rounded once (to nearest even, overflow to +-inf) to the head's type.  So in fp32 grad_logits equals
 * ppn_loss_backward(s) followed by torch's sigmoid backward, bit for bit, for s = ppn_sigmoid(logits); and a 16-bit
 * call equals the fp32 call on the widened inputs, the gradient converted to the head's type.
 * Types, alignment, workspace (ppn_loss_workspace_bytes_opt) and every PPN_E_* answer are those of the _opt exports;
 * grad_logits [B, C, H, W] has the head's type and every element is written.  The caller reads loss[5] and grad_logits
 * in place of the same results on sigmoid(logits); nothing else changes.
 *   ppn_sigmoid: y[i] = s(x[i]) for i < n, x of x_dtype (PPN_HEAD_*; PPN_E_BADARG otherwise, checked first), y fp32:
 *                the values the two loss exports use, e.g. to build from a logits model the head tensor that the
 *                parse entry points read.  n = 0 is a no-op; x and y need the alignment of their element. */
int ppn_loss_forward_logits(const void* logits, const PPNShape* shape, const PPNTargets* targets, const PPNLossOptions* opt,
                            float* loss, void* workspace, size_t workspace_bytes, void* stream);
int ppn_loss_backward_logits(const void* logits, const PPNShape* shape, const PPNTargets* targets, const PPNLossOptions* opt,
                             const float* grad_loss, void* grad_logits, void* stream);
int ppn_sigmoid(const void* x, int32_t x_dtype, float* y, size_t n, void* stream);

/* ---- multi-person pose AP over the packed result (the validation pass's scoring stage) ----------------------------
 * Stands in for the poseval fork the reference scores its validation with (main.validate / main.test_output):
 * eval_helpers.assignGTmulti per image, then evaluateAP.computeMetrics (computeRPC, VOCap) over the pass.  The fork is
 * not part of this project: the specification is the float64 restatement of DESIGN.md §12.  Joints j < J; the
 * prediction of joint j is part j + 1 of a human, at the centre of its box (ppn_part_centres), with its part score;
 * an absent part is a score-0 entry at (0, 0), as evaluation.pred_frame writes it.  Joints j >= K - 1 have no
 * prediction.
 * Ground truth, DEVICE pointers: people of image b are rows [person_off[b], person_off[b+1]) of the three arrays. */
typedef struct PPNPoseGT {
    const int32_t* person_off;  /* [B + 1]                                                          */
    const double*  head_box;    /* [n, 4] x1, y1, x2, y2 of the head rectangle                      */
    const double*  joint_xy;    /* [n, J, 2] x, y                                                   */
    const uint8_t* joint_valid; /* [n, J] 1 = joint annotated                                       */
    int32_t        n;           /* rows of the three arrays                                         */
} PPNPoseGT;

typedef struct PPNAPParams {
    int32_t n_joints;           /* J, 1..32 (PPN_E_UNSUPPORTED above 32)                             */
    double  dist_thresh;        /* PCKh threshold: a joint matches if dist / headSize <= it (0.5)    */
    double  head_scale;         /* headSize = head_scale * |(x2 - x1, y2 - y1)| (0.6)               */
} PPNAPParams;

/* Per-image match result, caller-owned device memory; slot i of image b stands for the i-th human of the result. */
typedef struct PPNAPMatch {
    float*   score;             /* [B, R, J] entry score of (slot, joint), for slots < used[b], joints < min(K - 1, J) */
    uint8_t* label;             /* [B, R, J] 1 = true positive (same entries)                        */
    int32_t* used;              /* [B] min(count[b], R of the packed result)                         */
    int32_t* flags;             /* [B] PPN_AP_* bits                                                 */
    int32_t* n_gt;              /* [B, J] annotated GT joints of the image (nGTall)                  */
    int32_t  R;                 /* slot stride of score / label, >= the packed result's R            */
} PPNAPMatch;
#define PPN_AP_OVERFLOW 1       /* count[b] > R: humans beyond the slots were never seen             */
#define PPN_AP_BAD_GT   2       /* more than 64 GT people, or person_off outside [0, n]: GT not used */

/* ppn_ap_match: assignGTmulti on B images of a packed result, one CTA per image (distances in fp64, one rounding per
 *   operation, dist = sqrt(dx*dx + dy*dy) / headSize, NaN never matches).  A prediction is labelled with its match
 *   mask against the GT person it is assigned to (the first GT person of maximal PCKh that in turn prefers it, as
 *   the two arg-max passes of assignGTmulti decide), every other prediction with 0.  Reads `humans` only during the
 *   call: the parser may overwrite it afterwards.  Up to 64 GT people per image (more: PPN_AP_BAD_GT, checked on the
 *   device); any R.
 * ppn_ap_workspace_bytes: scratch of ppn_ap_finalize for N images of R slots and J joints (N * R * J < 2^31).
 * ppn_ap_finalize: computeMetrics over N images laid out as one PPNAPMatch (images in the order the entries are
 *   appended): entries of every joint ranked by descending score, equal scores the later-appended entry first, NaN
 *   first (a CUB segmented radix sort on 64-bit keys in the workspace), then computeRPC and VOCap.  ap, precision,
 *   recall: [J + 1] fp64 in percent, the last entry the plain mean over the joints.  A joint without entries gives
 *   0, one with entries and no GT joint NaN recall and AP.  status[3] (int32): images flagged PPN_AP_OVERFLOW, images
 *   flagged PPN_AP_BAD_GT, entries per joint.  Deterministic: the result depends on the ranked entries alone. */
int ppn_ap_match(const PPNHumans* humans, int32_t B, int32_t K, const PPNPoseGT* gt, const PPNAPParams* params,
                 const PPNAPMatch* out, void* stream);
int ppn_ap_workspace_bytes(int32_t N, int32_t R, int32_t J, size_t* bytes);
int ppn_ap_finalize(const PPNAPMatch* match, int32_t N, int32_t K, int32_t J, double* ap, double* precision,
                    double* recall, int32_t* status, void* workspace, size_t workspace_bytes, void* stream);

/* ---- batch augmentation: warp, flip and normalise a ragged uint8 batch, and move its annotations -----------------
 * Stands in for the reference's per-image transform (aug.py: affine / crop / resize of the image, keypoints and boxes,
 * then ToNormalizedTensor).  The rule is DESIGN.md §14; exactness starts at the parameters.  Per image, a forward
 * affine A (2x3 fp64, source pixel coordinates -> output coordinates, pixel (row i, col j) centred at (j + .5, i + .5)),
 * M = A^-1 rounded to fp32, and a flip flag (A already mirrors; the flag swaps left_* and right_* part columns).
 *
 * ppn_augment_images: output pixel (u, v), channel c, fp32 with one rounding per operation:
 *   sx = ((m00 (u + .5) + m01 (v + .5)) + m02) - .5, sy likewise; x0 = floor(sx), ax = sx - x0, the same in y;
 *   val = (p00 (1 - ax) + p01 ax) (1 - ay) + (p10 (1 - ax) + p11 ax) ay,   p01 the tap at (x0 + 1, y0), ...
 *   out = (val * in_scale - mean[c]) / std[c]   (IEEE division), rounded once to the output dtype.
 * A tap outside the source reads fill[c]; a pixel whose four taps are all outside, or whose sx or sy is non-finite or
 * beyond +-2^30, takes val = fill[c].  One launch for the batch, any mix of sizes, no host synchronisation.
 * `pixels` is read in aligned 16-byte words that hold at least one byte of an image, so it must be readable up to the
 * next 16-byte boundary after its last image byte.  out: [B, 3, out_h, out_w] (PPN_LAYOUT_NCHW) or [B, out_h, out_w, 3]
 * (PPN_LAYOUT_NHWC, a channels_last tensor's memory) of out_dtype (PPN_HEAD_*), out_bytes exactly its size, aligned
 * to its element.  PPN_E_BADARG: a NULL pointer, B < 1, an image with h or w outside [1, 65535] or outside `bytes`,
 * an output size outside [1, 65535] or not matching out_bytes, an unknown dtype or layout, std[c] <= 0 (or NaN). */
typedef struct PPNImageBatch {
    const uint8_t* pixels;      /* DEVICE: every image, HWC RGB uint8, image b at byte offset[b] (any alignment)      */
    const int64_t* offset;      /* DEVICE [B]                                                                      */
    const int32_t* hw;          /* DEVICE [B][2] (h, w)                                                             */
    const int64_t* offset_host; /* HOST copies of offset and hw with the same values: the checks read these, the      */
    const int32_t* hw_host;     /*   kernel the device arrays                                                       */
    size_t         bytes;       /* size of `pixels`                                                                 */
    int32_t        B;
} PPNImageBatch;

typedef struct PPNImageNorm {
    float mean[3];              /* per channel, in units of val * in_scale (ImageNet: 0.485, 0.456, 0.406)         */
    float std[3];               /* > 0 (ImageNet: 0.229, 0.224, 0.225)                                              */
    float fill[3];              /* pixel value of taps outside the source, in uint8 units (0)                       */
    float in_scale;             /* fl32(1 / 255); 1 reproduces rt_test.py's 0-1 statistics on 0-255 pixels          */
} PPNImageNorm;

#define PPN_LAYOUT_NCHW 0
#define PPN_LAYOUT_NHWC 1

int ppn_augment_images(const PPNImageBatch* in, const float* M /* DEVICE [B][2][3] */, const PPNImageNorm* norm,
                       int32_t out_h, int32_t out_w, int32_t out_dtype, int32_t out_layout, void* out, size_t out_bytes,
                       void* stream);

/* ppn_augment_people: the annotations of B images (the PPNPeople layout ppn_encode_targets reads; n people, K - 1
 * parts each) through each image's A, in fp64 with one rounding per operation, written to `out` (person_off is
 * unchanged and not written):
 *   keypoints: (a00 x + a01 y) + a02, (a10 x + a11 y) + a12 rounded once to fp32; on a flipped image column i of
 *              keypoints and visible takes column perm[i] (perm: HOST [K - 1], a permutation);
 *   visible:   never changed otherwise (points that leave the output stay visible; the encoder's bounds drop them);
 *   bbox:      w > 0 and h > 0: the bounds of the four transformed corners (cx -+ w / 2, cy -+ h / 2), as
 *              ((min + max) / 2, max - min); otherwise the transformed centre with w = h = 0 (part 0 stays unlabelled);
 *   size:      size * sqrt(|a00 a11 - a01 a10|).
 * DEVICE pointers except perm.  PPN_E_BADARG: a NULL pointer, B < 1, n < 0, K outside [1, 256], perm not a
 * permutation of [0, K - 1).  n = 0 is a no-op.  The rows of `in` are only read, so out may not alias them. */
typedef struct PPNPeopleOut {
    double*  bbox;              /* [n, 4]                                                           */
    float*   keypoints;         /* [n, K - 1, 2]                                                    */
    uint8_t* visible;           /* [n, K - 1]                                                       */
    double*  size;              /* [n]                                                              */
} PPNPeopleOut;
int ppn_augment_people(const PPNPeople* in, int32_t B, int32_t n, int32_t K, const double* A /* DEVICE [B][2][3] */,
                       const uint8_t* flip /* DEVICE [B] */, const int32_t* perm, const PPNPeopleOut* out, void* stream);

/* ---- the flip test: merge a head with the mirrored head of its horizontally flipped input -------------------------
 * The standard test-time step of a bottom-up pose estimator; the reference has none, so the rule is DESIGN.md §15.
 * head is the network's head on an input x, head_flipped its head on x.flip(-1) (the exact pixel mirror), both
 * [B, C, H, W] of shape->head_dtype.  For every element, with p = part_mirror, q = limb_mirror:
 *   source plane   part group g (resp, conf, x, y, w, h), part k: g * K + p[k];
 *                  limb plane (e, a, b) of the [E, sH, sW] block: (q[e], a, sW - 1 - b)
 *   source cell    (i, j) reads head_flipped at (i, W - 1 - j)
 *   value          widened exactly, then fp32 with one rounding per operation, no FMA: b' = 1 - b in the x group
 *                  (b otherwise), out = (a + b') * 0.5, rounded once (to nearest even) to the head's dtype.
 * part_mirror (HOST [K]) maps each part to its mirror part (left_* <-> right_*, part 0 to itself); limb_mirror
 * (HOST [E]) each limb (s, t) to the limb (p[s], p[t]).  Both travel in the kernel parameters: one launch, no
 * copies, no host synchronisation, capturable in a CUDA graph.  out may be head (in place: the first half of a
 * [2B] output); it must not overlap head_flipped, nor overlap head without being it.
 * PPN_E_BADARG: a NULL pointer, B < 1, an unknown head_dtype, a pointer not aligned to the element size, part_mirror
 * or limb_mirror not a self-inverse permutation or part_mirror[0] != 0, out overlapping head_flipped (or part of head).
 * PPN_E_UNSUPPORTED: inW != W * gridW (the cell mirror is not exact), 2 * off_w != sW - 1 (nor the window mirror),
 * K > 64, H * W > PPN_MAX_CELLS. */
int ppn_flip_merge(const void* head, const void* head_flipped, void* out, const PPNShape* shape,
                   const int32_t* part_mirror /* host [K] */, const int32_t* limb_mirror /* host [E] */,
                   void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PPN_DECODE_H_ */
