/*
 * onesweep_b200.h -- C-ABI of the B200-native OneSweep radix sort (libonesweep_b200.so).
 *
 * This is the drop-in boundary for the ONE hot path of b0nes164/GPUSorting that this repository
 * rebuilds: the CUDA OneSweep 8-bit LSD radix sort.  Plain C types only (no torch / C++ types).
 * Each entry point cites the reference interface it replaces; paths are relative to
 * /root/reference/GPUSortingCUDA/ unless stated otherwise.
 *
 * Conventions
 *   - All `d_*` pointers are device pointers on the handle's device; keys must be 16-byte aligned
 *     (the reference assumes this too: Sort/OneSweep.cu:77 reinterpret_cast<uint4*>), and so must the values
 *     of the osb200_sort_* calls (the result is moved home in 16-byte words after an odd number of executed
 *     passes).  A misaligned key or value pointer is OSB200_ERR_INVALID_ARG in every call that would sort,
 *     whatever its n (n <= 1, begin_bit == end_bit and n > max_n are decided before the pointers are looked at).
 *   - The sorted result is returned IN the caller's key/value buffers (even number of passes, like
 *     Sort/OneSweepDispatcher.cuh:325-335 which ends in m_sort).
 *   - Calls are asynchronous on `stream` (a cudaStream_t passed as void*; NULL = default stream) and
 *     never synchronise the host, unlike the reference (cudaDeviceSynchronize inside the dispatch,
 *     OneSweepDispatcher.cuh:318).  One sort in flight per handle; distinct handles are independent.
 *   - Return value: 0 on success, a negative osb200_status otherwise.  Nothing aborts or prints (the
 *     reference ignores every CUDA error and printf()s on misuse, OneSweepDispatcher.cuh:195-199).
 *   - n == 0 or 1 is a successful no-op; n > max_n (from create) is OSB200_ERR_SIZE.
 *   - There is NO CPU fallback: if no sm_100 device / driver is usable, create fails.
 */
#ifndef ONESWEEP_B200_H_
#define ONESWEEP_B200_H_

#include <stddef.h>
#include <stdint.h>

#if defined(OSB200_BUILDING) && defined(__GNUC__)
#define OSB200_API __attribute__((visibility("default")))
#else
#define OSB200_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef struct osb200_sorter* osb200_handle;          /* opaque single-GPU sorter  */
typedef struct osb200_sharded_sorter* osb200_sharded_handle; /* opaque multi-GPU sorter */

typedef enum osb200_status {
    OSB200_OK = 0,
    OSB200_ERR_INVALID_ARG = -1, /* null handle/pointer, bad key/value width, misaligned keys/values */
    OSB200_ERR_SIZE = -2,        /* n > max_n of the handle                                        */
    OSB200_ERR_UNSUPPORTED = -3, /* combination not built (e.g. u64 keys with values)              */
    OSB200_ERR_NO_DEVICE = -4,   /* no CUDA device of compute capability 10.x                      */
    OSB200_ERR_ALLOC = -5,       /* device allocation failed                                       */
    OSB200_ERR_NCCL = -6,        /* NCCL failure in the sharded path                               */
    OSB200_ERR_CUDA = -1000      /* -(1000 + cudaError_t) for any other CUDA runtime error         */
} osb200_status;

/* ABI version of this header (major*1000 + minor). */
OSB200_API int osb200_version(void);
/* Static string for a status code returned by any function below. */
OSB200_API const char* osb200_status_string(int status);

/* ------------------------------------------------------------------------------------------------
 * Sorter object.  Replaces  OneSweepDispatcher::OneSweepDispatcher(bool keysOnly, uint32_t maxSize)
 * / ~OneSweepDispatcher()  (Sort/OneSweepDispatcher.cuh:42-83): owns the alternate (ping-pong)
 * buffers, the global histogram, the tile tickets and the chained-scan tile descriptors.  Unlike the
 * reference the caller owns the keys/values being sorted (as in the Unity API,
 * /root/reference/GPUSortingUnity/Runtime/OneSweep.cs:297-306).
 *   key_bytes   4 (uint32 keys, the reference's only CUDA type) or 8 (uint64 keys, 8 digit passes)
 *   value_bytes 0 (keys only == keysOnly=true) or 4 (uint32 payload == keysOnly=false)
 *   max_n       largest n a sort call may pass (reference: maxSize), up to 2^34
 * The device is the calling thread's current CUDA device.
 * ---------------------------------------------------------------------------------------------- */
OSB200_API int osb200_create(osb200_handle* out, uint64_t max_n, int key_bytes, int value_bytes);
OSB200_API int osb200_destroy(osb200_handle h);
/* Device bytes a handle with these parameters allocates (alt buffers + control state). */
OSB200_API uint64_t osb200_workspace_bytes(uint64_t max_n, int key_bytes, int value_bytes);

/* ------------------------------------------------------------------------------------------------
 * Sort entry points.
 *   osb200_sort_keys_u32      replaces OneSweepDispatcher::DispatchKernelsKeysOnly(uint32_t size)
 *                             (Sort/OneSweepDispatcher.cuh:311-336)
 *   osb200_sort_pairs_u32     replaces OneSweepDispatcher::DispatchKernelsPairs(uint32_t size)
 *                             (Sort/OneSweepDispatcher.cuh:338-363); stable: equal keys keep their
 *                             input order (in-order ranking, Sort/OneSweep.cu:207-253)
 *   osb200_sort_keys_u64      no CUDA reference (SURVEY D3); same plan with 8 digit places, shape of
 *                             GPUSortingUnity/Runtime/OneSweep.cs:297-306 Sort(...)
 * ---------------------------------------------------------------------------------------------- */
OSB200_API int osb200_sort_keys_u32(osb200_handle h, uint32_t* d_keys, uint64_t n, void* stream);
OSB200_API int osb200_sort_pairs_u32(osb200_handle h, uint32_t* d_keys, uint32_t* d_values, uint64_t n, void* stream);
OSB200_API int osb200_sort_keys_u64(osb200_handle h, uint64_t* d_keys, uint64_t n, void* stream);

/* Typed keys and descending order (the reference has them only in its HLSL path: IntToUint / FloatToUint and inverses,
 * GPUSortingD3D12/Shaders/SortCommon.hlsl:134-154; descending :594-656).  The order-preserving bit transform is fused
 * into the first pass (and the histogram) and undone in the last pass's stores: no extra traffic.  Floats follow the
 * IEEE total order of their bit patterns (-0.0 < +0.0, NaNs at the ends), as the reference's transform does.
 * Descending is the complement of the transformed key, so equal keys KEEP their input order (stable) -- unlike the
 * reference's index reversal, which reverses ties.  key_type must match the handle's key width. */
typedef enum osb200_key_type {
    OSB200_KEY_U32 = 0, OSB200_KEY_I32 = 1, OSB200_KEY_F32 = 2, OSB200_KEY_U64 = 3, OSB200_KEY_I64 = 4, OSB200_KEY_F64 = 5
} osb200_key_type;
OSB200_API int osb200_sort_keys_typed(osb200_handle h, void* d_keys, uint64_t n, int key_type, int descending, void* stream);
OSB200_API int osb200_sort_pairs_typed(osb200_handle h, void* d_keys, uint32_t* d_values, uint64_t n, int key_type,
                                       int descending, void* stream);

/* Sort on a bit range [begin_bit, end_bit) of the (unsigned) key only, CUB-style: keys that agree on those bits keep their
 * input order (stable).  ceil((end_bit-begin_bit)/8) digit passes instead of key_bytes; the last digit may be narrower
 * than 8 bits; an odd pass count is handled inside (the result is always returned in the caller's buffers).  d_values may
 * be NULL (keys only).  begin_bit == end_bit is a no-op.  Reference: none in CUDA (its passes are fixed at radixShift
 * 0/8/16/24, Sort/OneSweepDispatcher.cuh:325-335); SURVEY 8f rank 2. */
OSB200_API int osb200_sort_bits(osb200_handle h, void* d_keys, uint32_t* d_values, uint64_t n, int begin_bit, int end_bit,
                                void* stream);

/* Segmented sort: every segment [offsets[i], offsets[i+1]) of d_keys (and d_values, may be NULL) is sorted ascending and
 * stable, in place, by ONE thread block in shared memory (all four digit passes in one launch; no histogram, descriptor or
 * lookback traffic).  d_segment_offsets: num_segments + 1 non-decreasing element offsets in device memory.
 * max_segment_len: an upper bound of the segment lengths known to the caller; it picks the block geometry (<= 256 or 2,048 keys:
 * 256 threads, up to 8 blocks per SM; <= 16,384: 512 threads) -- segments longer than 16,384 keys return OSB200_ERR_SIZE
 * (sort those with osb200_sort_*), segments longer than max_segment_len are left untouched.  Empty segments are fine.
 * Reference: SplitSort, the reference's segmented sort (GPUSortingCUDA/SegSort/SplitSort/SplitSort.cuh:702-938 bins
 * segments by length and dispatches one kernel per bin); SURVEY 8f rank 4.  The same kernel is the small-n path of every
 * osb200_sort_* call: n <= 16,384 (8,192 for 64-bit keys) is one segment, one launch (option "small_path", default 1). */
OSB200_API int osb200_segmented_sort_u32(osb200_handle h, uint32_t* d_keys, uint32_t* d_values, const uint64_t* d_segment_offsets,
                                         uint64_t num_segments, uint32_t max_segment_len, void* stream);

/* Host-buffer entry points: copy in, sort, copy back, synchronise.  `h_*` may be pageable or pinned
 * host memory.  This is the end-to-end call a host-side caller of the reference would make (the
 * reference itself has no host-data API; its buffers are generated on the device,
 * OneSweepDispatcher.cuh:215-219). */
OSB200_API int osb200_sort_host_keys_u32(osb200_handle h, uint32_t* h_keys, uint64_t n);
OSB200_API int osb200_sort_host_pairs_u32(osb200_handle h, uint32_t* h_keys, uint32_t* h_values, uint64_t n);
OSB200_API int osb200_sort_host_keys_u64(osb200_handle h, uint64_t* h_keys, uint64_t n);

/* ------------------------------------------------------------------------------------------------
 * Kernel-level entry points (for parity tests against the reference's individual kernels).
 *   osb200_global_histogram   replaces OneSweep::GlobalHistogram<<<...>>> (Sort/OneSweep.cu:44-123):
 *                             d_hist[place*256 + digit], uint64 counts, key_bytes places, overwritten.
 *   osb200_digit_binning_pass replaces OneSweep::Scan + one OneSweep::DigitBinningPassKeysOnly/Pairs
 *                             launch (Sort/OneSweep.cu:125-162,164-344,346-600): a stable counting
 *                             sort of d_in (and d_in_values, may be NULL) on the 8-bit digit at
 *                             `radix_shift` into d_out (d_out_values).  Out-of-place.  radix_shift is 0/8/16/24
 *                             in the reference; any shift below the key width is accepted (a shift within 8
 *                             bits of the top yields fewer than 256 bins -- the sharded exchange uses that).
 *   osb200_validate           replaces Validate<<<...>>> (UtilityKernels.cuh:403-429,432-479):
 *                             *h_err_count = number of adjacent inversions in d_keys (synchronises).
 * ---------------------------------------------------------------------------------------------- */
OSB200_API int osb200_global_histogram(osb200_handle h, const void* d_keys, uint64_t n, uint64_t* d_hist, void* stream);
OSB200_API int osb200_digit_binning_pass(osb200_handle h, const void* d_in, void* d_out, const uint32_t* d_in_values,
                              uint32_t* d_out_values, uint64_t n, uint32_t radix_shift, void* stream);
OSB200_API int osb200_validate(osb200_handle h, const void* d_keys, uint64_t n, uint64_t* h_err_count, void* stream);

/* Test-input generator.  Replaces InitRandom<<<256,256>>> (UtilityKernels.cuh:53-83 keys, :85-117 pairs):
 * the reference's deterministic hybrid Tausworthe/LCG generator with Thearling-Smith entropy reduction
 * (and_count = ENTROPY_PRESET value 0..4).  d_payload may be NULL; if not, it receives a copy of the key
 * (reference behaviour, UtilityKernels.cuh:115) or the element index when payload_is_index != 0 (stricter
 * stability test, SURVEY 8c).  The whole 64-bit n is honoured (the reference takes uint32 size). */
OSB200_API int osb200_init_random_u32(uint32_t* d_keys, uint32_t* d_payload, uint64_t n, uint32_t and_count, uint32_t seed,
                           int payload_is_index, void* stream);

/* Tuning / introspection (no reference equivalent; the reference's constants are #defines,
 * Sort/OneSweep.cu:17-42).  Returns OSB200_ERR_INVALID_ARG for unknown keys/values.  Options:
 *   "rank_mode"      0 = atomic-ranked (default), 1 = ballot-ranked.  The default ranks keys with ONE shared-memory
 *                    atomicAdd per key and relies on sm_100 handing the return values of one warp-wide ATOMS.ADD to
 *                    same-address lanes in ascending lane order -- an UNDOCUMENTED hardware property on which the
 *                    stability of every pass rests.  osb200_create verifies it on the device (a self-test kernel in the
 *                    production geometry) and falls back to 1 if it ever fails; 1 is the supported escape hatch: it uses
 *                    the reference's documented 8-ballot warp multisplit (Sort/OneSweep.cu:208-253) at ~2x the pass time.
 *                    Round 2 saw the assumption fail in ONE development build of the pairs kernel (rank phase of some
 *                    warps concurrent with the chained-scan loads of others, n >= 2^28; DESIGN.md 4.1,
 *                    profiles/r02_pairs_order_violation.md); the shipped kernels never overlap the two and the GPU suite
 *                    compares full-size sorts element by element.
 *   "variant"        kernel variant id (2 = default wide-tile kernel; 0/1 development baselines)
 *   "short_circuit"  1 (default) = digit passes on which ALL keys agree are skipped, decided on the device from the
 *                    global histogram without any host synchronisation; 0 = always run every pass like the reference
 *   "spin_cap"       lookback polls of one predecessor tile before a digit thread stops waiting and re-reduces that
 *                    tile itself (forward-progress fallback, reference: Sort/EmulatedDeadlocking.cu:159-267)
 *   "debug_stall_every"  test hook for that fallback: N > 0 makes every N-th tile withhold its reduction
 *   "profile"        1 = record CUDA events between the kernels of a sort (osb200_get_profile)
 *   "small_path"     1 (default) = a sort of at most one tile (info "small_path_max_n": 16,384 keys, 8,192 for 64-bit keys)
 *                    is ONE launch of the single-block shared-memory sort (see osb200_segmented_sort_u32); 0 = always the
 *                    multi-kernel path
 *   "hot_passes"     1 (default) = a digit place in which one bin holds >= n/8 keys (low-entropy inputs; reference presets
 *                    UtilityKernels.cuh:42-52) is executed by the HOT instantiation of the DigitBinningPass, which ranks
 *                    a tile's most frequent digit with one ballot per round instead of serialised same-address atomics;
 *                    decided on the device, both instantiations are enqueued for every pass; 0 = plain kernel only
 * Info keys: "tile_keys","launches_per_sort","memsets_per_sort","sm_count","rank_mode","variant","atomic_order_ok",
 * "max_n","epoch","short_circuit","spin_cap","small_path","small_path_max_n","hot_passes","last_skip_mask",
 * "last_hot_mask","last_executed_passes" (the last three read the device plan of the previous sort and synchronise). */
OSB200_API int osb200_set_option(osb200_handle h, const char* key, int64_t value);
OSB200_API int64_t osb200_get_info(osb200_handle h, const char* key);
/* With option "profile"=1 every sort records CUDA events on its stream between its kernels.  Returns the number of
 * intervals written (waits for the last sort): out_ms[0]=GlobalHistogram, [1]=Scan, [2+p]=DigitBinningPass p.
 * (The reference times only the whole dispatch, OneSweepDispatcher.cuh:221-224.) */
OSB200_API int osb200_get_profile(osb200_handle h, float* out_ms, int capacity); /* "tile_keys","launches_per_sort","sm_count",... ; <0 if unknown */

/* ------------------------------------------------------------------------------------------------
 * Multi-GPU sharded sort (one process per GPU).  No reference equivalent (the reference is single
 * device, SURVEY 2.1); this is BASELINE.json's "MSD bucket-exchange then local OneSweep".
 *
 *   osb200_sharded_unique_id  rank 0 fills a 128-byte NCCL unique id; the host application broadcasts
 *                             it to all ranks (torch.distributed / MPI / files).
 *   osb200_sharded_create     every rank: joins the communicator (world ranks on ONE node), allocates
 *                             receive + local-sort workspace for up to max_n_local keys per rank plus
 *                             `slack_percent` head-room for bucket imbalance.  max_n_local and slack_percent MUST
 *                             be the same on every rank: if any rank's share exceeds that capacity, every rank
 *                             returns OSB200_ERR_SIZE from the sort call together (no rank is left in a collective).
 *   osb200_sharded_sort_keys_u32
 *                             every rank passes its n_local unsorted keys.  After the call rank r owns
 *                             the r-th contiguous slice of the global ascending order: *d_out points
 *                             into handle-owned memory valid until the next call, *n_out is its length.
 *                             Steps: local top-digit histogram -> all-gather of the 256-bin histograms
 *                             -> bucket->rank assignment -> exchange pass (keys move over NVLink) ->
 *                             local OneSweep.
 * ---------------------------------------------------------------------------------------------- */
OSB200_API int osb200_sharded_unique_id(void* out_128_bytes);
OSB200_API int osb200_sharded_create(osb200_sharded_handle* out, const void* unique_id_128_bytes, int rank, int world,
                          uint64_t max_n_local, int slack_percent);
OSB200_API int osb200_sharded_destroy(osb200_sharded_handle h);
OSB200_API int osb200_sharded_sort_keys_u32(osb200_sharded_handle h, const uint32_t* d_keys_local, uint64_t n_local,
                                 uint32_t** d_out, uint64_t* n_out, void* stream);
/* The host-side exchange plan, a pure function of the all-gathered histograms (exported so the N>1 logic can be
 * tested on CPU): dest[256] = owner rank of every most-significant-digit bucket (contiguous, non-decreasing,
 * balanced on the global counts); recv_count[world] = keys every rank ends up with; recv_off[256] = for source
 * `rank`, the element offset inside dest[d]'s receive buffer where its bucket-d keys go (bucket-major,
 * source-rank-minor: the globally stable order of the MSD partition). */
OSB200_API int osb200_sharded_plan(const uint64_t* hist_all /*[world][256]*/, int world, int rank, int32_t* dest,
                                   uint64_t* recv_count, uint64_t* recv_off);
/* 1 (default when CUDA IPC peer mapping works) = the exchange is the DigitBinningPass kernel scattering straight into
 * the peers' receive buffers over NVLink; 0 = staged: local pass + ncclSend/ncclRecv.  Same value on every rank. */
OSB200_API int osb200_sharded_set_fused(osb200_sharded_handle h, int fused);
/* Exchange granularity: by default, when world is a power of two and the equal-width split of the key space fits the
 * receive buffers, the exchange bins on the top log2(world) bits only (long runs, full NVLink sectors); otherwise on
 * the top 8 bits with the greedy plan.  on=1 forces the 256-bucket plan (tests / skewed data).  Same on every rank. */
OSB200_API int osb200_sharded_force_fine(osb200_sharded_handle h, int on);
/* The two single-GPU sorters inside a sharded sorter (exchange pass / local sort), e.g. to set options. */
OSB200_API int osb200_sharded_local_handle(osb200_sharded_handle h, osb200_handle* exch, osb200_handle* local);
/* Milliseconds of the phases of the last sharded sort on this rank: [0]=histogram+allgather,
 * [1]=exchange, [2]=local sort, [3]=total (device time, CUDA events). */
OSB200_API int osb200_sharded_last_timing(osb200_sharded_handle h, float* out_ms4);

#ifdef __cplusplus
} /* extern "C" */
#endif
#endif /* ONESWEEP_B200_H_ */
