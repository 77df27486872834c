/*
 * libfrcfrc_cuda — C ABI of the B200 (sm_100a) UniFrac engine.
 *
 * This is the drop-in boundary for the one hot path of fluhus/frackyfrac:
 * the call `unifrac(abnd, tree, *wgt)` at frcfrc/frcfrc.go:58, i.e. everything
 * in frcfrc/unifrac.go (embedding :32-67,:97-124; pair distances :144-228).
 * Everything that touches strings (flags, Newick, TSV / sparse tables, species
 * validation, text output) stays on the host side of this boundary.
 *
 * Conventions
 *   - plain C, no CUDA / torch types; all pointers are HOST pointers unless a
 *     parameter says "device".
 *   - every entry point returns an frc_status (0 = ok) except frc_destroy,
 *     frc_ctx_destroy, frc_last_error and frc_abi_version.
 *   - inputs are borrowed and fully copied before frc_create returns (cgo
 *     forbids retaining Go pointers).
 *   - failures (bad argument, CUDA error, out of memory) are errors; there is
 *     no CPU fallback anywhere behind this ABI.
 *   - entry points of one job/context must be called from one host thread at a
 *     time.
 *   - the calling thread's current CUDA device is the same after every call as
 *     before it (a job may drive several devices).
 *
 * ABI v2 (this file) over v1: frc_opts_t gained n_devices / devices (one process,
 * several GPUs, ONE ordered stream), `normalize` gained the value 2, frc_next_f32 /
 * frc_chunk_exceptions deliver the fast paths' native fp32 distances without the
 * host widening pass, frc_ctx_create_multi.
 */
#ifndef FRCFRC_CUDA_H
#define FRCFRC_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FRC_ABI_VERSION 2

typedef enum {
  FRC_OK = 0,
  FRC_ERR_ARG = 1,         /* invalid tree / table / option                    */
  FRC_ERR_CUDA = 2,        /* a CUDA runtime or driver call failed             */
  FRC_ERR_OOM = 3,         /* device or pinned host memory exhausted           */
  FRC_ERR_STATE = 4,       /* call sequence violated                           */
  FRC_ERR_UNSUPPORTED = 5  /* device is not sm_100 / problem exceeds a limit   */
} frc_status;

/* Replaces the `weighted bool` argument of unifrac() (frcfrc/unifrac.go:97),
 * set from flag -w (frcfrc/frcfrc.go:22). */
typedef enum { FRC_UNWEIGHTED = 0, FRC_WEIGHTED = 1 } frc_mode;

/* Which pair kernel runs.
 *   AUTO : EXACT when n_pairs * n_nodes is small (bit-exact testdata .want files),
 *          otherwise FAST.
 *   FAST : unweighted -> tcgen05 GEMM (u8 block floating point with exact int32
 *          accumulation by default, bf16 hi/lo planes with FRC_FLAG_UW_BF16);
 *          weighted -> FP32 L1 tiles.  Within 1e-5 relative of the reference.
 *   EXACT: fp64, the reference's summation order (ascending node id, separate
 *          multiply and add): bit-identical to frcfrc/unifrac.go:144-205. */
typedef enum { FRC_PATH_AUTO = -1, FRC_PATH_FAST = 0, FRC_PATH_EXACT = 1 } frc_path;

/* The flattened tree: what enumerateNodes (frcfrc/unifrac.go:127-133) and the
 * treeDists loop (:117-120) produce.  Node ids are PRE-ORDER indices, root = 0,
 * so parent[v] < v for v > 0 and siblings appear in file order. */
typedef struct {
  int32_t n_nodes;
  const int32_t *parent;  /* [n_nodes], parent[0] = -1                          */
  const double *length;   /* [n_nodes], node.Distance verbatim, root included   */
} frc_tree_t;

/* One row per sample: the per-sample map[string]float64 of frcfrc.go:41-51
 * after name resolution.  col = id of a LEAF node carrying that species name
 * (a name carried by several leaves is expanded to all of them, a name that
 * only matches internal nodes is dropped: unifrac.go:38-43).  val > 0, finite.
 * A leaf may appear at most once per row (checked when values are used: weighted and
 * exact jobs; for presence a repeat is harmless); order within a row is free. */
typedef struct {
  int64_t n_samples;
  const int64_t *row_ptr; /* [n_samples + 1], row_ptr[0] = 0                    */
  const int32_t *col;     /* [row_ptr[n_samples]]                               */
  const double *val;      /* [row_ptr[n_samples]]                               */
} frc_csr_t;

#define FRC_FLAG_NO_D2H 1u /* keep distances in HBM: frc_next returns DEVICE
                              pointers (kernel-only timing, GPU consumers)     */

#define FRC_FLAG_UW_BF16 2u /* fast unweighted: run the bf16 hi/lo (kind::f16) tensor-core
                              kernel instead of the default u8 block-floating-point
                              (kind::i8, exact integer accumulation) one             */

#define FRC_FLAG_SHARD_EMBED 4u /* world > 1 (one process per GPU): build the embedding for this rank's
                                  sample shard only and exchange the compact form: the presence bit
                                  columns are stored into every rank's HBM by the kernel that produces
                                  them (CUDA IPC mappings over NVLink; NCCL all-gather when IPC is not
                                  available), weighted panels are all-gathered with NCCL.  Needs a
                                  context with a communicator (frc_ctx_comm_init).  Every rank of the
                                  communicator must create its job with the same inputs (the call is
                                  collective).  Without the flag each rank rebuilds the whole embedding.
                                  (Jobs over several devices of ONE process, opts.n_devices, shard and
                                  exchange over peer memory by themselves.)                          */

#define FRC_FLAG_UW_BITS 8u /* fast unweighted, u8 integer mode: expand the operand tiles inside
                              the pair kernel from the presence bits instead of materialising
                              them in HBM (3 bytes per (sample, node) saved; info.operand_kind 3) */

#define FRC_FLAG_L_TILES 16u /* normalize == 0 (-l as coded): allow the FP32 tile kernel instead of the
                               exact list walk.  The walk's mis-pairing has a closed form: node v is
                               matched iff both samples hold it and the largest present leaf id under v
                               is the same for both (DESIGN.md); the tiles carry that key per (node,
                               sample) next to the values.  Within 1e-5 relative of the reference
                               instead of bit-exact.  path FAST: always the tiles; AUTO: exact for small
                               inputs (the AUTO rule of every mode), tiles above.  Without the flag
                               normalize == 0 always runs the exact walk and FAST is refused.  Ignored
                               for normalize 1 and 2.  One process over several GPUs and
                               FRC_FLAG_SHARD_EMBED are supported; the capacity mode (panels sharded
                               over devices) is not: FRC_ERR_UNSUPPORTED where it would be chosen.  */

#define FRC_FLAG_PRUNE 32u /* run on the subtree the table observes: the root and every node with a listed leaf
                             below it (any row of col[], also rows another rank of a FRC_FLAG_SHARD_EMBED job
                             stages).  The other nodes hold 0 in every sample and add nothing.  The fast paths
                             also merge every unary chain that is left into its lowest node (lengths summed,
                             the default normaliser counts the chain's nodes), so the kernels run over at most
                             2 x (listed leaves) nodes instead of n_nodes.  Exact path: pruned, never merged,
                             bit-identical to the unpruned run.  Fast paths: within 1e-5 of the reference, but
                             not byte-identical to the unpruned run.  The path choice (AUTO), every error and
                             its message (original node ids) are the same as without the flag;
                             info.n_nodes_padded and info.tree_height describe the tree that ran (DESIGN.md). */

typedef struct {
  int32_t mode;       /* frc_mode                                               */
  int32_t normalize;  /* flag -l (frcfrc.go:25):
                         1 = no -l: sort + divide by the all-node total (unifrac.go:56-67)
                         0 = -l AS CODED in the reference: normalizeFlatNodes is skipped
                             (unifrac.go:108-110) and with it the id-sort (:57), so the
                             merge-join (:178-203) walks POST-ORDER lists and mis-pairs nodes;
                             reproduced bit for bit by a dedicated kernel (csrc/exact.cu), or
                             within 1e-5 by the key-matched FP32 tiles (FRC_FLAG_L_TILES)
                         2 = -l as documented: id-sorted lists, raw values
                         0 and 2 need mode == FRC_WEIGHTED (frcfrc.go:84-86)            */
  int32_t path;       /* frc_path                                               */
  int32_t device;     /* CUDA device ordinal; -1 = current device (n_devices <= 1) */
  int32_t rank;       /* tile-band sharding over `world` PROCESSES (one per GPU):  */
  int32_t world;      /*   every G consecutive bands go to G different ranks; 0/1 = all  */
  int64_t band_rows;  /* rows of the lower triangle per output chunk; 0 = auto
                         (bands of equal pair count, see frc_plan_bands)        */
  uint32_t flags;     /* FRC_FLAG_*                                             */
  int32_t n_devices;  /* 0 / 1: one GPU (`device`).  > 1: THIS process drives that many GPUs:
                         one validation + staging pass, per-device uploads / embedding / tile
                         bands / pinned rings, and frc_next hands the bands out in flat-index
                         order from their owners' rings -- one ordered stream behind the seam
                         (frcfrc.go:58-62).  -1 = every visible sm_100 device.  Needs
                         world <= 1.  Ignored when `ctx` is given (the context's devices).  */
  const int32_t *devices; /* [n_devices] ordinals; NULL = 0 .. n_devices-1      */
} frc_opts_t;

typedef struct frc_ctx frc_ctx_t; /* device + streams + reusable memory pools  */
typedef struct frc_job frc_job_t; /* one unifrac() call                         */

/* What a finished or running job did; for benchmarks and tests. */
typedef struct {
  int32_t path_taken;      /* FRC_PATH_FAST / FRC_PATH_EXACT                    */
  int32_t n_bands_total;   /* bands of the whole triangle                       */
  int32_t n_bands_mine;    /* bands this rank yields                            */
  int32_t tree_height;     /* level-synchronous passes of the embedding         */
  int64_t n_pairs_total;   /* n(n-1)/2 (frc_create_cross: n_q * n_ref)           */
  int64_t n_pairs_mine;
  int64_t n_nodes_padded;  /* contraction length the pair kernel runs over      */
  int64_t kernel_launches; /* kernels of this library launched so far           */
  double h2d_ms, embed_ms;  /* device time (CUDA events) of the upload / embedding */
  double pairs_ms;          /* sum over delivered bands of (band start -> pair kernel end) on the band's
                               stream: the kernel's own time when the job runs ONE band with
                               FRC_FLAG_NO_D2H (bench.py's roofline leg); with several bands in flight
                               the spans overlap and the sum is only an upper bound        */
  double fixup_ms;          /* same for (pair kernel end -> fix-up end)                   */
  double run_ms;            /* embedding start -> last band (and its D2H) done;
                               valid once the stream has been read to its end      */
  int64_t h2d_bytes, d2h_bytes;
  int64_t embed_bytes;     /* algorithmic HBM bytes of the embedding stage      */
  int64_t flagged_pairs;   /* fast unweighted: pairs recomputed exactly (d tiny) */
  int64_t operand_kind;    /* fast unweighted: 1 = bf16 hi/lo planes, 2 = u8 block floating
                              point, 3 = u8 expanded in-kernel from bits; 0 otherwise */
  int64_t gather_bytes;    /* bytes this rank received in the embedding exchange    */
  int32_t n_devices;       /* GPUs this job drives (1 unless opts.n_devices > 1)     */
  int32_t value_bytes;     /* bytes per distance on PCIe / in HBM: 4 (fast paths, fp32) or 8 (exact) */
  int64_t exceptions;      /* distances delivered so far that fp32 could not carry (frc_chunk_exceptions) */
  double create_ms;        /* host wall clock of frc_create                          */
} frc_info_t;

int frc_abi_version(void);

/* Optional reusable context.  A job created with ctx == NULL owns a private
 * one.  Reusing a context across jobs reuses its device / pinned allocations. */
int frc_ctx_create(int32_t device, frc_ctx_t **out);
/* A context over several GPUs of this process (opts.n_devices semantics: n_devices == -1 = all
 * visible sm_100 devices, devices == NULL = ordinals 0..n-1).  Peer access between the devices is
 * enabled when the hardware allows it (the sharded embedding then stores its bit columns straight
 * into every device's HBM over NVLink); without it every device rebuilds the whole embedding. */
int frc_ctx_create_multi(int32_t n_devices, const int32_t *devices, frc_ctx_t **out);
void frc_ctx_destroy(frc_ctx_t *ctx);

/* Multi-GPU, one process per GPU.  frc_comm_unique_id produces the 128-byte NCCL id on one
 * rank; the host distributes it (any channel) and every rank calls frc_ctx_comm_init
 * (collective) on its context.  The communicator is destroyed with the context. */
#define FRC_COMM_ID_BYTES 128
int frc_comm_unique_id(char *id /* [FRC_COMM_ID_BYTES] */);
int frc_ctx_comm_init(frc_ctx_t *ctx, const char *id, int32_t rank, int32_t world);

/* Replaces the body of unifrac() (frcfrc/unifrac.go:97-124): validates, copies
 * and uploads the inputs, builds the branch embedding on the device and queues
 * the first tile bands.  Returns without waiting for the device. */
int frc_create(frc_ctx_t *ctx, const frc_tree_t *tree, const frc_csr_t *abnd,
               const frc_opts_t *opts, frc_job_t **out);

/* Query x reference distances (an extension: the reference CLI has no such mode).  The job yields the
 * n_q x n_ref block of distances between every query sample and every reference sample, and nothing else
 * (no reference x reference or query x query pairs).
 *   distance  d(q, r) is exactly what frc_create over the concatenated table [ref rows; query rows] gives for
 *             the pair (i, j) = (n_ref + q, r): the query sample is the FIRST sample of the pair (row i,
 *             common.go:25), which matters for normalize = 0, whose merge-join is not symmetric in fp.
 *   stream    frc_next / frc_next_f32 / frc_chunk_exceptions use the flat index q * n_ref + r (query-major),
 *             contiguous runs in strictly increasing order, one band of whole 128-row query tiles per run;
 *             frc_restart and FRC_FLAG_NO_D2H work as for frc_create.  frc_job_info: n_pairs_total =
 *             n_q * n_ref.  n_ref == 0 or n_q == 0 is an empty stream; an empty sample gives NaN.
 *   options   mode, normalize 0 / 1 / 2, path (AUTO applies its rule to the block's pair count), device,
 *             n_devices / devices (one ordered stream), band_rows (counted in QUERY rows), and the flags
 *             FRC_FLAG_NO_D2H, FRC_FLAG_UW_BF16, FRC_FLAG_UW_BITS, FRC_FLAG_L_TILES and FRC_FLAG_PRUNE (the
 *             support is the union of the leaves both tables list).
 *   refused   FRC_ERR_UNSUPPORTED for world > 1, FRC_FLAG_SHARD_EMBED, and the capacity mode of the fast
 *             weighted path over several devices (FRC_CAPACITY=1, or panels beyond about half of one device's
 *             free HBM).
 * Both tables get every check of frc_create; the messages name the table and the row within it.  The
 * argument checks (also the refusals above except the capacity mode) come before any CUDA call. */
int frc_create_cross(frc_ctx_t *ctx, const frc_tree_t *tree, const frc_csr_t *ref, const frc_csr_t *query,
                     const frc_opts_t *opts, frc_job_t **out);

/* Replaces ranging over the iter.Seq[float64] that unifrac() returns
 * (frcfrc/frcfrc.go:58-62, unifrac.go:209-228).  Yields contiguous runs of the
 * flat lower-triangle vector, index(i,j) = i(i-1)/2 + j for j < i
 * (common/common.go:21-31), in strictly increasing index order (frc_create_cross:
 * the query-major block, index q * n_ref + r).  `*data` is
 * engine-owned pinned host memory (device memory with FRC_FLAG_NO_D2H), valid
 * until the next call on this job.  *count == 0 means the stream has ended.
 * A run is one tile band of the plan (frc_plan_bands) or, for the fast paths on
 * the host route, a piece of one of at most 2^21 values: those distances cross
 * PCIe as fp32 and are widened here into a cache-sized buffer (csrc/wire.cu).
 * With FRC_FLAG_NO_D2H only exact-path jobs can be read through this call (device
 * doubles); fast-path jobs keep fp32 in HBM: frc_next_f32. */
int frc_next(frc_job_t *job, const double **data, int64_t *first_index, int64_t *count);

/* The same stream in the fast paths' native precision.  The tensor-core and FP32 tile kernels
 * produce fp32 ratios and store them as fp32, a band crosses PCIe as 4 bytes per pair, and this call
 * hands out the pinned landing buffer itself: one run per band, no host pass over the data.  (frc_next
 * on a fast-path job widens the same fp32 values into doubles on the host, so both calls deliver the
 * same numbers.)  Exact-path jobs are float64 only: FRC_ERR_STATE.  The two calls may not be mixed
 * on one pass of a job.  With FRC_FLAG_NO_D2H `*data` is a device pointer. */
int frc_next_f32(frc_job_t *job, const float **data, int64_t *first_index, int64_t *count);

/* Distances of the run returned by the LAST frc_next_f32 call that fp32 cannot carry to 2^-23
 * relative (|d| < 1.2e-38, only ever produced by the exact fix-up passes on pathological trees):
 * their flat indices and float64 values.  frc_next applies them itself.  Usually *count == 0. */
int frc_chunk_exceptions(frc_job_t *job, const int64_t **index, const double **value, int64_t *count);

/* Re-runs embedding + pair stage on the inputs already resident in HBM
 * (benchmarking the device path without the host→device copy). */
int frc_restart(frc_job_t *job);

int frc_job_info(const frc_job_t *job, frc_info_t *info);

/* Pure host helper (no device needed): the band decomposition frc_create uses for these
 * options (band_rows, world and FRC_FLAG_NO_D2H in `flags` select it).  Writes, for the bands
 * that `rank` of `world` yields (all bands when world <= 1), the flat index of their first pair
 * and their pair count, in stream order; returns the number of such bands (also when it exceeds
 * `cap`), or a negative frc_status.  Lets a multi-process host merge the per-rank streams back
 * into IterPairs order. */
int64_t frc_plan_bands(int64_t n_samples, int64_t band_rows, int32_t rank, int32_t world,
                       uint32_t flags, int64_t *first_index, int64_t *count, int64_t cap);

/* Legal at any time, also mid-stream (the consumer's `break`, frcfrc.go:59-61). */
void frc_destroy(frc_job_t *job);

/* Message of the last failed call on this job; with job == NULL, of the last
 * failed frc_create / frc_ctx_create on the calling thread. */
const char *frc_last_error(const frc_job_t *job);

#ifdef __cplusplus
}
#endif
#endif /* FRCFRC_CUDA_H */
