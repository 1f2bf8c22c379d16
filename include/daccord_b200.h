/* daccord_b200.h -- C ABI of the B200 window-consensus engine.
 *
 * gt1/daccord has no plugin / FFI interface of its own (SURVEY.md section 8b): the seam this
 * library replaces is the per-window body of HandleContext::operator()
 * (reference src/HandleContext.hpp:2051-2494) together with the DebruijnGraphInterface
 * calls it drives (reference src/DebruijnGraphInterface.hpp:29-65: setup, filterFreq,
 * computeFeasibleKmerPositions, getLevelSuccessors, setupNodes, setupAddHeap,
 * addNextFromHeap, traverse, checkCandidatesU, getCandidate).  A per-window virtual call
 * cannot feed a GPU, so the boundary is batch level: the caller (the daccord main loop,
 * reference src/daccord.cpp:2107-2540) hands over thousands of windows per call, each a
 * list of (read, offset, length, strand) slices into the packed read database, and gets
 * back, per window, the consensus string, its summed edit distance and the placement
 * trace of align(A-window, consensus) (reference src/HandleContext.hpp:2434-2493).
 *
 * Plain pointers and sizes only; int return codes (0 = ok); no exceptions cross the
 * boundary.  A dcu_ctx is used from one host thread at a time and holds one resident batch; a
 * caller that wants several batches in flight on one GPU (one being piled or voted while
 * another runs the window kernel) creates one dcu_ctx per in-flight batch -- the library
 * serialises their window passes and lets everything else overlap.  All input arrays stay
 * owned by the caller and may be released when the call returns.
 */
#ifndef DACCORD_B200_H
#define DACCORD_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

/* CLI + error-profile parameters of the path (reference src/daccord.cpp:101-169, :1282-1305,
 * :1867-1913): -w, -k lo[,hi], -m, --minfilterfreq/--maxfilterfreq, -e and the (p_i, p_d,
 * est_cor) triple from the .eprof that seeds computeOffsetLikely / KmerLimit. */
typedef struct dcu_params {
  uint32_t w;          /* window size (-w), <= 59 */
  uint32_t k_lo, k_hi; /* k-mer range (-k), 3..14 (the reference compiles 3..12) */
  uint32_t min_cov;    /* -m */
  int32_t  min_ff, max_ff; /* --minfilterfreq / --maxfilterfreq */
  uint64_t max_err;    /* -e (UINT64_MAX = unlimited) */
  double   p_i, p_d, est_cor;
} dcu_params;

/* one sequence slice of a window; slice 0 of a window is the A-read window itself
 * (reference src/HandleContext.hpp:2032-2043).  gpos = index of the first forward-strand base
 * of the slice in the packed database (4 * byte offset of the read + position); for a
 * reverse-complemented B read (flags&1, reference HandleContext.hpp:1910) the slice is the
 * reverse complement of forward bases [gpos, gpos+len). */
typedef struct dcu_slice { uint32_t gpos; uint16_t len; uint16_t flags; } dcu_slice;
/* one window [astart, astart+w) of A-read aread (reference HandleContext.hpp:382-447) */
typedef struct dcu_window { uint32_t slice_begin; uint16_t slice_cnt; uint16_t reserved; uint32_t aread; uint32_t astart; } dcu_window;

enum { DCU_WIN_SKIPPED = 0,   /* slice_cnt < -m : "insufficient depth" (HandleContext.hpp:2499-2503) */
       DCU_WIN_OK = 1,        /* consensus found */
       DCU_WIN_FAILED = 2,    /* all k / filterfreq attempts failed (HandleContext.hpp:2496-2497) */
       DCU_WIN_OVERFLOW = 250 }; /* the window exceeded every workspace capacity of this build (err = capacity code): no consensus;
                                    callers treat it like DCU_WIN_FAILED and log it -- one window never fails a batch (the reference
                                    swallows a read's exception and continues, src/daccord.cpp:2466-2478) */
#define DCU_CONS_STRIDE 64    /* bytes of consensus arena per window (ASCII) */
#define DCU_OPS_STRIDE 128    /* bytes of placement-trace arena per window */
/* placement trace steps, one byte each, forward order (libmaus2 BaseConstants::STEP_*) */
enum { DCU_STEP_MATCH = 0, DCU_STEP_MISMATCH = 1, DCU_STEP_INS = 2, DCU_STEP_DEL = 3 };

typedef struct dcu_result {
  uint8_t  status;   /* DCU_WIN_* */
  uint8_t  k;        /* k of the graph that produced the consensus */
  int8_t   ff;       /* filter frequency at which it was found */
  uint8_t  clen;     /* consensus length */
  uint32_t err;      /* summed edit distance of the consensus to all slices (checkCandidatesU) */
  uint16_t nops;     /* placement trace length */
  uint16_t ncand;    /* candidates the successful traverse produced */
  int32_t  elength;  /* expected length estimate (HandleContext.hpp:2172) */
} dcu_result;

typedef struct dcu_ctx dcu_ctx;

/* builds the OffsetLikely / KmerLimit tables on the host and uploads them (replaces reference
 * src/daccord.cpp:1867-1913, :1981-1988 + per-thread HandleContext construction :1989-2023) */
int dcu_create(const dcu_params* params, int device, dcu_ctx** out);
void dcu_destroy(dcu_ctx* ctx);
/* packed 2-bit read database, Dazzler .bps layout: 4 bases per byte, first base in the top
 * two bits (replaces DecodedReadContainer, reference src/DecodedReadContainer.hpp:81-84) */
int dcu_set_reads(dcu_ctx* ctx, const uint8_t* packed, uint64_t nbytes);
/* same, but the buffer is already resident in device memory on ctx's device (e.g. after an
 * ncclBroadcast of the database); the library does not take ownership */
int dcu_set_reads_device(dcu_ctx* ctx, const void* dpacked, uint64_t nbytes);
/* same database as `owner` (a dcu_ctx on the same device that got it through dcu_set_reads[_device]); owner must outlive ctx's use of it */
int dcu_share_reads(dcu_ctx* ctx, dcu_ctx* owner);
/* run one batch: host buffers in, host buffers out (results in submission order).
 * cons must hold nwin*DCU_CONS_STRIDE bytes, ops nwin*DCU_OPS_STRIDE bytes. */
int dcu_run(dcu_ctx* ctx, const dcu_window* win, uint64_t nwin, const dcu_slice* sl, uint64_t nsl,
            dcu_result* res, uint8_t* cons, uint8_t* ops);
/* split form used by the measurement harness: upload, launch (device timed), download */
int dcu_upload(dcu_ctx* ctx, const dcu_window* win, uint64_t nwin, const dcu_slice* sl, uint64_t nsl);
int dcu_launch(dcu_ctx* ctx, float* kernel_ms);   /* runs the resident batch; kernel_ms may be NULL */
int dcu_download(dcu_ctx* ctx, dcu_result* res, uint8_t* cons, uint8_t* ops);
/* ---- caller stage on the GPU (SURVEY 8f N1): trace reconstruction + window / slice extraction --------------------
 * Replaces, for tspace <= 128 (any -w / -a), the host work of reference src/HandleContext.hpp:1740-2049
 * (OverlapDataInterface::computeTrace per activated overlap, advanceA / getStringLengthUsed per window, the active set
 * ordered by (escore<<32)|z).  Input: the overlaps the caller selected for its A-reads (reference
 * src/daccord.cpp:2112-2288: top -D by score, ordered by abpos), grouped by A-read in ascending order, with their
 * trace points.  The descriptors are built in device memory and become the resident batch (as after dcu_upload). */
typedef struct dcu_overlap {
  int32_t abpos, aepos, bbpos, bepos; uint32_t flags; int32_t aread, bread, diffs;
  int32_t tlen, reserved;       /* number of trace values (2 per tile) */
  uint64_t trace_off;           /* index of this overlap's first value in `trace` */
} dcu_overlap;
int dcu_pile(dcu_ctx* ctx, const dcu_overlap* ovl, uint64_t novl, const uint16_t* trace, uint64_t ntrace, int32_t tspace,
             const uint64_t* read_boff /* byte offset of every read in the packed DB */, const uint32_t* read_len, uint64_t nreads,
             uint32_t advance, uint64_t maxalign, uint64_t* nwin, uint64_t* nsl);
/* window descriptors of the resident batch (aread / astart are what the pile vote needs), nwin entries */
int dcu_get_windows(dcu_ctx* ctx, dcu_window* win, dcu_slice* sl /* may be NULL */);
/* ---- caller stage behind the kernel on the GPU (SURVEY 8f N2): pile vote ------------------------------------------
 * Replaces, for the resident batch after dcu_launch, the host work of reference src/HandleContext.hpp:2446-2493
 * (placement walk into PileElements) and :2541-2710 (sort, optional -f fill, runs of consecutive positions spanning
 * >= 100 bases, column vote), so that corrected bases instead of per-window traces cross PCIe.  The windows of the
 * batch must be grouped by ascending A-read and ordered by astart inside a read (what dcu_pile and the reference's
 * window loop produce).  read_boff / read_len are needed for producefull (-f) only and may be NULL otherwise.
 * A segment is one output sequence of the reference (:2710-2724): its FastA header is
 * ">{aread+1}/{counter}/{first}_{first+len} A=[{first},{last}]", its bases chars[off .. off+len). */
typedef struct dcu_segment { uint32_t aread, first, last, reserved; uint64_t len, off; } dcu_segment;
int dcu_vote(dcu_ctx* ctx, int producefull, uint64_t minlen, const uint64_t* read_boff, const uint32_t* read_len, uint64_t nreads,
             uint64_t* nseg, uint64_t* nchars);
/* segments (in A-read, position order) and the character buffer (nchars bytes) of the last dcu_vote */
int dcu_get_corrected(dcu_ctx* ctx, dcu_segment* seg, char* chars);
/* statistics of the last launch: kernels launched, windows that needed the large-workspace pass */
int dcu_last_stats(dcu_ctx* ctx, uint64_t* launches, uint64_t* hard_windows);
/* more statistics of the last launch: windows the first pass handed to the plain HBM passes, windows beyond every capacity
 * (status DCU_WIN_OVERFLOW), warps per SM and shared-memory bytes per warp of a first pass that keeps data in shared memory (the hybrid
 * pass: k-mer table only, 32 warps; DCU_SMEM=1: the graph, 12-16 warps; 0 warps = plain HBM first pass) */
int dcu_last_stats2(dcu_ctx* ctx, uint64_t* second_pass_windows, uint64_t* lost_windows, uint32_t* smem_warps, uint32_t* smem_bytes_per_warp);
/* dump the tables as they sit in device memory (for tests): returns number of doubles written / needed, -1 on a CUDA error */
int64_t dcu_get_tables(dcu_ctx* ctx, int which, double* out, int64_t cap);
const char* dcu_strerror(int code);
const char* dcu_last_error(dcu_ctx* ctx);

enum { DCU_OK = 0, DCU_ERR_PARAM = 1, DCU_ERR_CUDA = 2, DCU_ERR_UNSUPPORTED = 3, DCU_ERR_OVERFLOW = 4, DCU_ERR_STATE = 5 };

#ifdef __cplusplus
}
#endif
#endif
