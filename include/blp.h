/*
 * blp.h -- C ABI of the B200-native candidate-pair similarity scorer.
 *
 * This is the drop-in boundary for ONE path of es1985/bipartite-link-prediction: the
 * neighbourhood similarity scores of similarity.py.  The reference has no FFI of its own for this
 * path -- it crosses Python->SWIG->C++ (SNAP) four times and does the set arithmetic in Python --
 * so each entry point below names the reference call sites it replaces (file:line relative to
 * the reference checkout).  INTEGRATION.md shows the ctypes stub a maintainer adds.
 *
 * Conventions
 *   - Every function returns an int: BLP_OK (0) or a negative blp_status.  Nothing throws across
 *     the boundary and nothing calls exit().  blp_last_error() returns a thread-local message.
 *   - The caller owns every buffer.  The library owns only the graph handle (CSR arrays, degree
 *     and weight tables in HBM) and stream-ordered scratch it allocates and frees per call.
 *   - Indices are LOCAL: users 0..n_users-1, businesses 0..n_biz-1 (the host layer maps the
 *     reference's shared id space onto them).  In a pair, an index that is negative, out of range
 *     or names a node of degree 0 means "id not in graph": every output of that pair is 0
 *     (similarity.py:59-60, 104-105).
 *   - Every entry point runs on its handle's device and restores the caller's current device
 *     before it returns.
 *   - A handle's graph is immutable after creation.  Scoring calls issued by ONE host thread on
 *     several streams overlap on the device; concurrent calls from several host threads on the
 *     same handle are not supported (the handle owns a side stream, events and the accounting
 *     of the last call) -- use one handle per thread.
 *   - There is no CPU fallback: without a CUDA device every compute entry point fails with
 *     BLP_ERR_CUDA.
 */
#ifndef BLP_H_
#define BLP_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BLP_VERSION 200 /* major*10000 + minor*100 + patch */

typedef enum blp_status {
    BLP_OK = 0,
    BLP_ERR_INVALID = -1,     /* bad argument (null pointer, negative size, bad side, ...) */
    BLP_ERR_CUDA = -2,        /* CUDA runtime / driver error, or no device */
    BLP_ERR_OOM = -3,         /* host or device allocation failed */
    BLP_ERR_RANGE = -4,       /* an edge endpoint is outside [0,n_users) x [0,n_biz) */
    BLP_ERR_UNSUPPORTED = -5  /* configuration outside what this build handles */
} blp_status;

typedef enum blp_side {
    BLP_SIDE_USER = 0,     /* hop-2 set of the user, neighbours of the business (similarity.py:20-61) */
    BLP_SIDE_BUSINESS = 1  /* hop-2 set of the business, neighbours of the user (similarity.py:63-106) */
} blp_side;

typedef struct blp_graph blp_graph; /* opaque; one per device / rank */

typedef struct blp_graph_info_t {
    int32_t n_users;
    int32_t n_biz;
    int64_t n_edges_in;       /* edge lines given */
    int64_t n_edges;          /* distinct edges kept (duplicates collapse, as in SNAP's TUNGraph) */
    int32_t n_users_in_graph; /* users with degree >= 1 */
    int32_t n_biz_in_graph;
    int32_t max_user_degree;
    int32_t max_biz_degree;
    int64_t device_bytes;     /* HBM held by the handle */
    int32_t device;
    int32_t sm_count;
    int32_t n_hub_biz;        /* businesses whose user list is also kept as a bitmap (user side) */
    int32_t n_hub_users;      /* users whose business list is also kept as a bitmap (business side) */
    int32_t hub_min_biz_degree;
    int32_t hub_min_user_degree;
    int64_t biz_index_bytes;     /* business x business co-review bitmap (0 = not built: the
                                    business side groups and expands per call) */
    float biz_index_build_ms;    /* its construction time at graph creation */
} blp_graph_info_t;

/* Which kernels scored the last call of a side (blp_score_stats_t.path). */
typedef enum blp_score_path {
    BLP_PATH_GROUPED = 0,   /* pairs grouped by x, hop2(x) built per group (k_score_side / k_score_light) */
    BLP_PATH_BIZ_INDEX = 1  /* business side: one pass over the pairs against the co-review bitmap */
} blp_score_path;

/* Per-launch accounting of the last blp_score_pairs call on a handle (for bench / roofline). */
typedef struct blp_score_stats_t {
    int64_t n_pairs;
    int64_t n_groups;         /* work items = distinct hop-2 sets built (+1 for the "not in graph" bucket) */
    int32_t kernel_launches;  /* kernels launched by the call */
    int32_t ctas;             /* grid of the scoring kernel */
    int32_t threads_per_cta;
    int32_t smem_bytes;       /* dynamic shared memory per CTA */
    int32_t range_passes;     /* id-range passes over the hop-2 bitmap (1 = fits shared memory) */
    float group_ms;           /* CUDA-event time of the grouping kernels (count, scan, scatter) */
    float score_ms;           /* CUDA-event time of the scoring kernels alone, on their own stream */
    float light_ms;           /* span of the warp-per-group kernel (it runs beside the CTA kernel), 0 if not used */
    int32_t light_groups;     /* work items scored by the warp-per-group kernel */
    int32_t path;             /* blp_score_path */
} blp_score_stats_t;

int blp_version(void);
const char* blp_last_error(void);
/* 0 when a CUDA device is usable, BLP_ERR_CUDA otherwise (never touches a device buffer). */
int blp_device_count(int* count);

/*
 * Build the graph handle.  Replaces snap.LoadEdgeList(snap.PUNGraph, graph_file, 0, 1)
 * (similarity.py:16) and the node-id list of similarity.py:22,65: duplicate edges collapse, both
 * CSR directions, degree tables and the Adamic-Adar weight table 1/ln(deg) (similarity.py:121-123)
 * are made resident in HBM.  edge_u / edge_b are HOST arrays of n_edges local indices
 * (column 0 = user, column 1 = business of graph.txt, dataset_maker.py:197); they are copied to the
 * device and built as blp_graph_create_device builds, on the legacy default stream.
 * Limits of the packed row descriptors: degrees below 2^24 and at most 2^30 adjacency entries per
 * direction after padding every row to a multiple of four (about a billion distinct edges);
 * beyond that the call fails with BLP_ERR_UNSUPPORTED.
 */
int blp_graph_create(int32_t n_users, int32_t n_biz, int64_t n_edges,
                     const int32_t* edge_u, const int32_t* edge_b,
                     int device, blp_graph** out);
/*
 * The same, with the edge arrays already in DEVICE memory and the whole construction on the GPU:
 * 64-bit radix sort of the (user, business) keys, duplicate removal, both padded CSR directions,
 * bank striping of the rows, per-entry weights (SURVEY.md section 8f, the step in front of the
 * path).  `stream` is a cudaStream_t; the call returns when the handle is ready.
 */
int blp_graph_create_device(int32_t n_users, int32_t n_biz, int64_t n_edges,
                            const int32_t* edge_u_dev, const int32_t* edge_b_dev,
                            int device, void* stream, blp_graph** out);
/*
 * graph.txt on the device (SURVEY.md section 8f rank 1: parse -> sort -> de-dup).  `text_dev` holds
 * the file's bytes in DEVICE memory: one "<user_id> <business_id>\n" per review
 * (dataset_maker.py:197).  A data line is a line whose first non-blank character starts an
 * integer; blank and comment lines are skipped, columns beyond the second ignored (what
 * snap.LoadEdgeList(PUNGraph, file, 0, 1) reads, similarity.py:16).
 *   blp_edge_list_count : *n_lines_host = number of data lines
 *   blp_edge_list_parse : col0_dev / col1_dev (DEVICE, n_lines x int64) = the ids of columns 0 / 1
 *                         in file order; BLP_ERR_INVALID when a data line lacks a second integer
 * Both run on the caller's current device and return when done.  The ids are of the reference's
 * shared id space; the host layer compacts them to local indices for blp_graph_create_device.
 */
int blp_edge_list_count(const char* text_dev, int64_t n_bytes, int64_t* n_lines_host, void* stream);
int blp_edge_list_parse(const char* text_dev, int64_t n_bytes, int64_t n_lines, int64_t* col0_dev,
                        int64_t* col1_dev, void* stream);
/*
 * examples.json on the device: the reference's {"<user>": {"<business>": label}}
 * (dataset_maker.py:142-159, read by similarity.py:14).  `text_dev` holds the file's bytes in
 * DEVICE memory.  The grammar is exactly what json.dumps writes for such a dict, with any JSON
 * whitespace (space, tab, CR, LF) between tokens: keys are canonical decimal integers ("0", or an
 * optional '-' and [1-9][0-9]*, at most 18 digits, no escapes), labels are JSON integers that fit
 * int32.  Anything else -- duplicate user keys or duplicate business keys of one user (json.load
 * resolves those by "last wins, first position"), other key spellings, float / bool / null /
 * string labels, deeper nesting, truncated or trailing text, a BOM, an empty file -- fails with
 * BLP_ERR_UNSUPPORTED, and blp_last_error() names the byte offset: such files are for json.load.
 *   blp_examples_count : *n_users_host / *n_pairs_host = users and (user, business) pairs
 *   blp_examples_parse : DEVICE outputs in file order -- user_off (n_users + 1 int64: the pairs of
 *                        user i are [user_off[i], user_off[i+1])), user_ids (n_users int64),
 *                        biz_ids (n_pairs int64), labels (n_pairs int32, may be NULL)
 * Both run on the caller's current device and return when done.
 */
int blp_examples_count(const char* text_dev, int64_t n_bytes, int64_t* n_users_host, int64_t* n_pairs_host,
                       void* stream);
int blp_examples_parse(const char* text_dev, int64_t n_bytes, int64_t n_users, int64_t n_pairs,
                       int64_t* user_off_dev, int64_t* user_ids_dev, int64_t* biz_ids_dev, int32_t* labels_dev,
                       void* stream);

/* Value column of a score file (blp_json_scores_count / _fill), as similarity._emit types it. */
typedef enum blp_json_kind {
    BLP_JSON_INT32 = 0,            /* cn: int32, written as ints */
    BLP_JSON_INT64 = 1,            /* pa: int64, written as ints */
    BLP_JSON_FLOAT64 = 2,          /* jaccard: doubles, float.__repr__ */
    BLP_JSON_FLOAT64_INT_ZERO = 3  /* adamic: doubles, but 0.0 written as the int 0 (similarity.py:116-126) */
} blp_json_kind;

/*
 * Score file writer: the bytes util.write_json writes for the {"<u>": {"<b>": v}} dict of one
 * method (similarity.py:49-61, 94-106), from DEVICE arrays.  The example users in file order are
 * user_off (n_users + 1 int64, pairs of user i = [user_off[i], user_off[i+1])) and user_ids
 * (int64); biz_ids (int64) and in_graph (one byte, 0 = an id of the pair is not in the graph) are
 * per pair; `values` is the pair's column of type `kind`.  A pair not in the graph is written as
 * the int 0 whatever the column; values == NULL writes only those zeros (an unknown method name,
 * or in-graph entries the reference omits).  Keys are the decimal ids; floats are float.__repr__
 * (Ryu shortest round trip), NaN / Infinity / -Infinity as json.dumps spells them.
 * User i's text is  , "<u>": {"<b>": v, "<b>": v}  -- empty when none of its pairs is written --
 * and the document is "{" + the concatenation of all users' texts without its first two bytes + "}"
 * ("{}" when all are empty).
 *   blp_json_scores_count : lengths_dev[i] (DEVICE, n_users int64) = bytes of user i's text
 *   blp_json_scores_fill  : the texts of users [user_begin, user_end), user i's at
 *                           out_dev + text_off_dev[i] - text_off_dev[user_begin], where text_off_dev
 *                           is the caller's exclusive prefix sum of the lengths (DEVICE int64)
 * so a large file is produced in chunks cut at user boundaries.  Both are asynchronous on `stream`.
 */
int blp_json_scores_count(const int64_t* user_off_dev, const int64_t* user_ids_dev, int64_t n_users,
                          const int64_t* biz_ids_dev, const uint8_t* in_graph_dev, const void* values_dev,
                          int kind, int64_t* lengths_dev, void* stream);
int blp_json_scores_fill(const int64_t* user_off_dev, const int64_t* user_ids_dev, int64_t n_users,
                         const int64_t* biz_ids_dev, const uint8_t* in_graph_dev, const void* values_dev,
                         int kind, const int64_t* text_off_dev, int64_t user_begin, int64_t user_end,
                         char* out_dev, void* stream);
int blp_graph_destroy(blp_graph* g);
int blp_graph_info(const blp_graph* g, blp_graph_info_t* info);

/* De-duplicated degrees (G.GetNI(i).GetDeg(), similarity.py:121) copied to a HOST array of
 * n_users (side USER) or n_biz (side BUSINESS) int32. */
int blp_graph_degrees(const blp_graph* g, int side, int32_t* host_out);

/*
 * Score n candidate pairs from one side.  Replaces loops A/B/C of users() (similarity.py:24-61)
 * for side USER and loops A'/B'/C' of business() (similarity.py:67-106) for side BUSINESS,
 * together with common_neighbors / jaccard / adamic_adar (similarity.py:108-126) -- one pass
 * produces what the reference computes with three separate intersections per pair.
 *
 * pair_u / pair_b and every output are DEVICE arrays of n elements in the caller's pair order
 * (any order; the library groups pairs by the node whose hop-2 set they share).  Outputs:
 *   cn        int32   |hop2(x) & N(y)|                      (similarity.py:113-114), bit-exact
 *   uni       int32   |hop2(x) | N(y)|                      (similarity.py:110), bit-exact
 *   jaccard   double  (double)cn / (double)uni, div.rn       (similarity.py:108-111), bit-exact
 *   adamic    double  sum over matched i with deg(i)>1 of 1/ln(deg(i)) (similarity.py:116-126);
 *                     accumulated in 2^-31 fixed point so the result does not depend on
 *                     summation order, bucket or rank count (|err| <= cn*2^-32, rel <= 4e-9)
 *   pa        int64   deg(u)*deg(v)  ("Link prediction.R":400-415); may be NULL
 *   hop2_size int32   |hop2(x)| of the pair's grouping node; may be NULL (debug / tests)
 * with x = user, y = business for side USER and x = business, y = user for side BUSINESS.
 * cn, uni, jaccard, adamic may each be NULL to skip that output.
 * `stream` is a cudaStream_t (NULL = legacy default stream).  The call is asynchronous.
 */
int blp_score_pairs(blp_graph* g, int side,
                    const int32_t* pair_u, const int32_t* pair_b, int64_t n,
                    int32_t* cn, int32_t* uni, double* jaccard, double* adamic,
                    int64_t* pa, int32_t* hop2_size, void* stream);

/*
 * The whole step with HOST buffers: what similarity.main (similarity.py:11-18) does between
 * loading examples.json and dumping the six score dicts, for array-shaped callers.  pair_u / pair_b
 * and the nine result columns are HOST arrays of n elements (page-locked memory for full speed;
 * pageable memory works, slower); the pair ids are uploaded, both sides are scored and every column
 * is copied back inside the call, which returns when the results are in host memory.  The copies
 * overlap the kernels: the user side runs in `user_slices` slices, the first `lead_slices` of them
 * before the rest of the ids are up, the business side in `biz_slices` slices between them
 * (<= 0 / < 0 / <= 0 select the defaults 4 / 1 / 2).  Outputs as in blp_score_pairs; a NULL column is
 * not copied back (the link is the bottleneck of this call: 56 bytes per pair for all nine).
 * Not re-entrant on one handle (it owns the handle's staging buffers and streams).
 */
int blp_score_pairs_host(blp_graph* g, const int32_t* pair_u, const int32_t* pair_b, int64_t n,
                         int32_t* u_cn, int32_t* u_union, double* u_jaccard, double* u_adamic,
                         int32_t* b_cn, int32_t* b_union, double* b_jaccard, double* b_adamic,
                         int64_t* pa, int user_slices, int lead_slices, int biz_slices);

/*
 * Candidate generation (SURVEY.md section 8f, rank 2): the businesses at BFS distance exactly 3
 * of each given user -- snap.GetNodesAtHop(G, u, 3, ...) of make_examples (dataset_maker.py:137-139),
 * i.e. N(hop2(u)) minus N(u).  Variable-length output, two calls:
 *   blp_hop3_count : counts[i] = |hop3(users[i])|                      (0 for ids not in the graph)
 *   blp_hop3_fill  : out_biz[offsets[i] .. offsets[i+1]) = hop3(users[i]) in ascending order,
 *                    offsets = exclusive prefix sum of counts (n+1 entries)
 * users / counts / offsets / out_biz are DEVICE arrays; `stream` is a cudaStream_t.
 */
int blp_hop3_count(blp_graph* g, const int32_t* users, int64_t n, int64_t* counts, void* stream);
int blp_hop3_fill(blp_graph* g, const int32_t* users, int64_t n, const int64_t* offsets,
                  int32_t* out_biz, void* stream);

/*
 * Evaluation (SURVEY.md section 8f, rank 4): what eval.run_evaluation (eval.py:10-32) computes from
 * one score file, on DEVICE arrays in the file's iteration order.
 *   blp_eval_precision_at_k : offsets (n_groups+1) delimit each user's pairs; precision_out[g] =
 *       mean label of the first min(k, #pairs) entries of a stable descending sort by score
 *       (eval.py:21-24).  The caller sums precision_out and divides by the number of users.
 *   blp_eval_roc_auc : counts4_host (HOST, 4 x uint64) = { #positives, #negatives,
 *       #(pos, neg) pairs with s+ > s-, #(pos, neg) pairs with s+ == s- };
 *       roc_auc_score (eval.py:26) = (counts[2] + counts[3]/2) / (counts[0] * counts[1]).
 */
int blp_eval_precision_at_k(const int64_t* offsets, const int32_t* labels, const double* scores,
                            int64_t n_groups, int32_t k, double* precision_out, void* stream);
int blp_eval_roc_auc(const int32_t* labels, const double* scores, int64_t n,
                     uint64_t* counts4_host, void* stream);

/*
 * Leave `n_sms` streaming multiprocessors out of the persistent scoring grids of this handle
 * (0 = use all, the default).  A caller that overlaps the final result gather with scoring
 * (NCCL's send/receive kernels need somewhere to run) reserves a few.
 */
int blp_graph_reserve_sms(blp_graph* g, int n_sms);

/*
 * Peer windows -- the final gather of the multi-GPU path (SURVEY.md section 8e; the reference is a
 * single process and has no counterpart) without a collective.  The destination rank allocates one
 * device buffer and exports it; every other rank (ONE PROCESS PER GPU: a handle cannot be opened
 * by the process that exported it) maps it and passes addresses inside it as the output pointers
 * of blp_score_pairs, so the scoring kernels' epilogue stores carry every result over
 * NVLink / NVSwitch as it is produced.  The rows are complete on the owner once the writers'
 * streams have been synchronised (then signal the owner, e.g. with a barrier).
 *   blp_peer_alloc : cudaMalloc `bytes` on `device`, handle_out = BLP_IPC_HANDLE_BYTES opaque bytes
 *                    to hand to the other ranks (torch.distributed, a pipe, a file ...)
 *   blp_peer_open  : map an exported buffer for kernels running on `device`; enables peer access
 *   blp_peer_close / blp_peer_free : undo open / alloc (both wait for the device to go idle)
 */
#define BLP_IPC_HANDLE_BYTES 64
int blp_peer_alloc(int device, int64_t bytes, void** dev_ptr, unsigned char* handle_out);
int blp_peer_open(int device, const unsigned char* handle, void** dev_ptr);
int blp_peer_close(int device, void* dev_ptr);
int blp_peer_free(int device, void* dev_ptr);
/* Copy-engine transfer of `bytes` from local device memory into a (peer) window, asynchronous on
 * `stream` (a cudaStream_t of `device`): for results that are produced in one burst -- the
 * business side's un-permute pass writes its columns in a fraction of a millisecond, which seven
 * peers cannot push through one GPU's NVLink ingress at once -- so that the transfer rides on a
 * side stream under the next kernels instead of stalling the stores of this one. */
int blp_peer_push(int device, void* dst, const void* src, int64_t bytes, void* stream);

/*
 * The result columns that are exact functions of the others and of the graph, computed where they
 * are needed instead of being moved: u_jaccard / b_jaccard from (cn, union) with the scoring
 * kernels' own expression (similarity.py:108-111; 0.0 where union is 0, i.e. the pair is not in the
 * graph) and pa = deg(u) * deg(v) from the pair ids ("Link prediction.R":400-415).  The multi-GPU
 * path does not send pa through the peer window at all (it is a function of the pair ids alone)
 * and can leave jaccard out as well (32 instead of 40 of the 48 reference bytes per pair on the
 * wire); the destination rank calls this for the peers' rows.  DEVICE arrays of n elements; any
 * output may be NULL.
 */
int blp_derive_pairs(blp_graph* g, const int32_t* pair_u, const int32_t* pair_b, int64_t n,
                     const int32_t* u_cn, const int32_t* u_union, const int32_t* b_cn,
                     const int32_t* b_union, double* u_jaccard, double* b_jaccard, int64_t* pa,
                     void* stream);

/* Accounting of the most recent blp_score_pairs on this handle (per side; with
 * blp_score_pairs_host: of the last slice).  The two event times
 * are valid once that call's work has completed (the function waits for its end event). */
int blp_score_stats(const blp_graph* g, int side, blp_score_stats_t* stats);

#ifdef __cplusplus
}
#endif
#endif /* BLP_H_ */
