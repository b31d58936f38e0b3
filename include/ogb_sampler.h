/*
 * ogb_sampler.h -- C-ABI of libogbsampler.so, the B200 (sm_100a) replay sampler.
 *
 * The reference (hliuson/ogbench) has no FFI: its hot path is a Python class API in
 * impls/utils/datasets.py.  This header is the boundary a ctypes stub binds (see INTEGRATION.md); each entry
 * point cites the reference interface it stands in for.  Plain pointers and sizes only, no torch types.
 * All functions return 0 on success and a negative ogb_status on failure; ogb_last_error() gives the message
 * (thread-local).  No C++ exception crosses this boundary: an internal one (e.g. host memory exhausted) comes back
 * as a status code.  Entry points switch to the dataset's CUDA device for their own work and restore the calling
 * thread's current device before returning.  There is no CPU fallback: without a CUDA device every compute entry point fails with
 * OGB_ERR_CUDA.
 */
#ifndef OGB_SAMPLER_H_
#define OGB_SAMPLER_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OGB_ABI_VERSION 1
#define OGB_MAX_NDIM 6
#define OGB_MAX_SLOTS 10

typedef enum {
  OGB_OK = 0,
  OGB_ERR_INVALID = -1,   /* bad argument; maps to ValueError */
  OGB_ERR_ASSERT = -2,    /* a reference `assert` failed (datasets.py:54,188,191-196,208); maps to AssertionError */
  OGB_ERR_INDEX = -3,     /* row index out of range; maps to IndexError (numpy fancy indexing in the reference) */
  OGB_ERR_CUDA = -4,      /* CUDA runtime / driver error, or no device */
  OGB_ERR_UNSUPPORTED = -5
} ogb_status;

typedef enum {
  OGB_U8 = 0, OGB_I8 = 1, OGB_I16 = 2, OGB_I32 = 3, OGB_I64 = 4, OGB_F16 = 5, OGB_F32 = 6, OGB_F64 = 7, OGB_BOOL = 8,
  OGB_U16 = 9, OGB_U32 = 10, OGB_U64 = 11
} ogb_dtype;

typedef enum {
  OGB_KIND_GC = 0,    /* GCDataset.sample,  datasets.py:213-294 (non-TRL) */
  OGB_KIND_HGC = 1,   /* HGCDataset.sample, datasets.py:496-643 */
  OGB_KIND_PLAIN = 2, /* Dataset.sample / get_subset, datasets.py:72-83 (also ReplayBuffer.sample, :86-146) */
  OGB_KIND_ATC = 3    /* ATCDataset.sample, datasets.py:369-464 */
} ogb_kind;

/* One dataset field as handed to Dataset.create(**fields) (datasets.py:45-57): C-contiguous, rows on axis 0. */
typedef struct {
  const char* name;
  const void* data;              /* host pointer (on_device 0), device pointer on the target device (1), or NULL (2) */
  int32_t dtype;                 /* ogb_dtype */
  int32_t ndim;                  /* including the leading row axis */
  int64_t shape[OGB_MAX_NDIM];
  int32_t on_device;             /* 2: allocate a zero-filled buffer (ReplayBuffer.create, datasets.py:101-103) */
} ogb_field;

/* The sampler hyper-parameters GCDataset/HGCDataset read from `config` (datasets.py:157-169,473-475,515-517,543,
 * 563,592-594).  The host wrapper resolves the optional *_subgoal_steps overrides exactly as the reference does
 * and builds the float64 reward tables with numpy so that `discount ** steps` is numpy's, not libm's. */
typedef struct {
  double discount;
  double value_p_curgoal, value_p_trajgoal, value_p_randomgoal;
  double actor_p_curgoal, actor_p_trajgoal, actor_p_randomgoal;
  int32_t value_geom_sample, actor_geom_sample;
  int32_t gc_negative;
  int32_t has_p_aug;             /* 0 <=> config['p_aug'] is None */
  double p_aug;
  int32_t frame_stack;           /* 0 <=> config['frame_stack'] is None */
  int32_t crop_padding;          /* 3 in GCDataset.augment (datasets.py:331); 0..127 (shifts are kept as int8) */
  int32_t value_subgoal_steps, actor_subgoal_steps, low_subgoal_steps; /* HGC only, already resolved */
  int32_t has_low_discount;
  double low_discount;
  int32_t lut_len;               /* max subgoal steps + 1 */
  const double* neg_reward_lut;  /* [lut_len] -(1 - discount**s)/(1 - discount), numpy-built (datasets.py:537-539) */
  const double* pow_lut;         /* [lut_len] discount**s, numpy-built (datasets.py:541) */
  int32_t dedup_keys;            /* 1: keys that the reference fills with equal values share one buffer */
  int32_t trl;                   /* config['agent_name'] in (trl, latent_trl, discrete_latent_trl), datasets.py:254-276:
                                    1 = with the valid_idxs override of :198-204, 2 = without it (lost at :211), 0 = off */
  int32_t jax_compat;            /* 1: the scalar keys are written as float32 (masks, rewards) / int32 (offsets, steps) --
                                    what `jit` makes of the reference's float64 / int64 numpy arrays with x64 off
                                    (impls/main.py:204-207) -- so that jax.dlpack.from_dlpack needs no cast */
  int32_t pad_;
} ogb_config;

/* Validation mode: the reference's own random draws, in its call order (SURVEY.md Appendix C).  Host pointers,
 * each [batch] unless noted; NULL where the reference did not make that call. */
typedef struct {
  const int64_t* rand_pos;   /* randint(n_valid)       datasets.py:303 -> :68/:70 */
  const int64_t* offset;     /* geometric(1-discount)  datasets.py:309 */
  const double* dist;        /* rand()                 datasets.py:313 */
  const double* u_traj;      /* rand()                 datasets.py:321 */
  const double* u_cur;       /* rand()                 datasets.py:325 */
} ogb_goal_draws;

typedef struct {
  const int64_t* idx_pos;    /* randint(n_valid), datasets.py:226 -> :68/:70; NULL when idxs are given */
  ogb_goal_draws goals[3];   /* [0] value goals, [1] low-value goals (HGC + low_discount), [2] actor goals */
  int32_t has_aug_coin;
  double aug_coin;           /* rand(), datasets.py:279 / :622 */
  const int64_t* crop;       /* [batch,2] randint(0, 2*padding+1), datasets.py:333; NULL unless the coin passed */
  const int64_t* trl_midpoints; /* randint(idxs, value_goal_idxs), datasets.py:259 (TRL samplers only) */
} ogb_draws;

typedef struct {
  const char* name;
  int32_t dtype;
  int32_t ndim;
  int64_t shape[OGB_MAX_NDIM + 1];
  void* device_ptr;
  size_t nbytes;
  size_t offset;             /* byte offset inside the batch's single device block */
  int32_t alias_of;          /* index of the key whose storage this one shares, or -1 */
} ogb_key_info;

typedef struct ogb_dataset ogb_dataset;
typedef struct ogb_sampler ogb_sampler;
typedef struct ogb_batch ogb_batch;

const char* ogb_last_error(void);
int ogb_abi_version(void);
int ogb_device_count(int* out);

/* Dataset.create + Dataset.__init__ (datasets.py:45-63): uploads every field into HBM -- fields with rows of at most
 * 2 KB as sub-fields of one packed record per dataset row (observations first; 16-byte offsets for sub-fields longer
 * than 16 B; record padded to 32 B, 64 B or a multiple of 128 B), longer rows as arrays of their own -- and builds the
 * valid-row tables from `valids`. */
int ogb_dataset_create(const ogb_field* fields, int32_t n_fields, int32_t device, ogb_dataset** out);
int ogb_dataset_size(const ogb_dataset* ds, int64_t* out);
int ogb_dataset_num_valid(const ogb_dataset* ds, int64_t* out);   /* -1 when the dataset has no 'valids' */
int ogb_dataset_set_active_rows(ogb_dataset* ds, int64_t n);      /* ReplayBuffer.size (datasets.py:131,142): rows to draw from */
int ogb_dataset_resident_bytes(const ogb_dataset* ds, size_t* out);
int ogb_dataset_destroy(ogb_dataset* ds);

/* Resident build of a dataset too large to hand over in one call (a directory of shards): the record layout
 * ogb_dataset_create would give these fields (shape[0] = capacity, data NULL), zero-filled, with no tables yet. */
int ogb_dataset_create_empty(const ogb_field* fields, int32_t n_fields, int32_t device, ogb_dataset** out);
/* Write dense host rows of every field (field order, NULL = leave untouched) into rows [row0, row0 + n_rows), through a
 * pinned double buffer; synchronous at return.  Refused on views, past the capacity, and while a sampler or a view holds
 * the dataset.  The dataset is unsealed until ogb_dataset_seal. */
int ogb_dataset_write_rows(ogb_dataset* ds, int64_t row0, int64_t n_rows, const void* const* field_rows, int32_t n_fields);
/* size = n_rows (<= capacity); builds the shadow next observation and the terminal and valid tables from the device
 * contents, exactly as ogb_dataset_create does. */
int ogb_dataset_seal(ogb_dataset* ds, int64_t n_rows);
/* The dataset of rows [row0, row0 + n_rows) of a sealed parent, sharing its memory (and holding a reference on it), with
 * its own size, terminal flags and valid tables: every entry point sees a dataset of n_rows rows.  Refused where a field's
 * base pointer would lose an alignment the kernels assume (OGB_ERR_UNSUPPORTED). */
int ogb_dataset_view(ogb_dataset* parent, int64_t row0, int64_t n_rows, ogb_dataset** out);

/* GCDataset.__post_init__ (datasets.py:182-211): trajectory boundaries from `terminals`, the asserts, search
 * acceleration tables.  `seed`/`stream_id` key the Philox streams (stream_id = rank or replica number). */
int ogb_sampler_create(ogb_dataset* ds, const ogb_config* cfg, int32_t kind, uint64_t seed, uint32_t stream_id,
                       ogb_sampler** out);
int ogb_sampler_set_stream(ogb_sampler* s, void* cuda_stream);    /* launch on the caller's stream instead */
int ogb_sampler_set_debug(ogb_sampler* s, int32_t flags);         /* bit 0: keep the index vectors readable; bit 1: canary fill;
                                                                     bit 3: row gathers walk their tiles with a fixed stride instead
                                                                     of taking them from the ticket counter; any other bit:
                                                                     OGB_ERR_INVALID */
int ogb_sampler_set_host_chunks(ogb_sampler* s, int32_t n_chunks); /* batches headed for host memory (ogb_batch_copy_to_host): issue
                                                                     big launches in up to n_chunks row chunks and copy each
                                                                     chunk out while the next is computed */
int ogb_sampler_set_deferred_index_check(ogb_sampler* s, int32_t on); /* given `idxs` are range-checked by the kernel instead of a
                                                                     host scan; OGB_ERR_INDEX then comes from ogb_batch_copy_to_host
                                                                     or ogb_batch_sync (batches that are read on the host anyway) */
int ogb_sampler_set_profile(ogb_sampler* s, int32_t on);          /* record CUDA events around the dominant kernel of each call */
int ogb_sampler_num_choices(const ogb_sampler* s, int64_t* out);   /* len(dataset.valid_idxs) as this sampler sees it (TRL overrides it) */
int ogb_sampler_num_terminals(const ogb_sampler* s, int64_t* out);
/* ReplayBuffer.add_transition (datasets.py:134-142): write one row of every field (host pointers in field order,
 * NULL = leave untouched), stream-ordered between the sampler's sample() calls. */
int ogb_sampler_write_row(ogb_sampler* s, int64_t row, const void* const* field_rows, int32_t n_fields);
/* ReplayBuffer.add_transition called for n transitions (datasets.py:134-142) in one stream-ordered launch: source row i of
 * every field goes to row (row0 + i) mod size, for i in [skip, n).  field_rows[f] is a C-contiguous [n, row] array (NULL =
 * leave the field untouched): host memory where on_device[f] == 0 (on_device NULL: every field), else device memory on the
 * dataset's device.  n - skip must not exceed the size, so that every row is written once (pass skip = n - size when n is
 * larger: only the last `size` transitions survive).  Host rows go through a pinned stage; the call returns once the
 * caller's host memory may be reused.  Device rows are read after the work already issued on producer_stream (NULL: no
 * wait; 1 / 2: the legacy / per-thread default stream) and after the call returns: *out_ticket numbers this call, and
 * every call numbered <= *out_retired has finished reading its sources (their memory may be reused).  Refused on views. */
int ogb_sampler_write_ring(ogb_sampler* s, int64_t row0, int64_t n, int64_t skip, const void* const* field_rows, int32_t n_fields,
                           const int32_t* on_device, void* producer_stream, uint64_t* out_ticket, uint64_t* out_retired);
/* The CUDA stream the sampler launches on (a DLPack producer orders its writes before it: __dlpack__(stream=...)). */
int ogb_sampler_get_stream(const ogb_sampler* s, void** out);
int ogb_sampler_copy_bounds(const ogb_sampler* s, int64_t* terminal_locs, int64_t* initial_locs); /* host out */
/* Debug: the start-row and trajectory tables sample() reads (read-only; changes nothing). */
typedef struct {
  int32_t valid_mode;        /* 0 no 'valids', 1 explicit row table (also TRL rows), 2 gap ranks, 3 one-probe segment table */
  int32_t seg_shift;         /* bucket width log2 of the segment table, -1 when it was refused */
  int32_t n_seg_table;       /* its entries (16 bytes each) */
  int32_t gap_shift;         /* bucket width log2 of the gap-rank search */
  int32_t term_shift;        /* bucket width log2 of the terminal search */
  int32_t pad_;
  int64_t n_choices;         /* len(valid_idxs) as this sampler sees it */
} ogb_table_info;
int ogb_sampler_table_info(const ogb_sampler* s, ogb_table_info* info);
int ogb_sampler_get_counter(const ogb_sampler* s, uint64_t* out); /* checkpointable RNG position */
int ogb_sampler_set_counter(ogb_sampler* s, uint64_t counter);
int ogb_sampler_destroy(ogb_sampler* s);

/* GCDataset.sample / HGCDataset.sample (datasets.py:213, :496).  n_batches >= 1 successive sample() calls are
 * produced by one launch and stacked on a leading axis (omitted when n_batches == 1).  `idxs` (host, may be
 * NULL) as in the reference: when given (batch_size * n_batches entries) no index draw is consumed.  `draws` NULL
 * selects the on-device Philox mode; otherwise validation mode (n_batches must be 1).  batch_size == 0 is legal, as
 * in the reference (every key with zero rows, nothing launched).  Asynchronous: returns after enqueueing on the
 * sampler's stream. */
int ogb_sampler_sample(ogb_sampler* s, int64_t batch_size, int32_t n_batches, const int64_t* idxs,
                       int32_t evaluation, const ogb_draws* draws, ogb_batch** out);

/* get_observations / get_goal_observations (datasets.py:341-357): one-key batch with rows `idxs` (host) of the
 * observations (frame-stacked as configured; which = 0) or of the goal representation (which = 1). */
int ogb_sampler_gather(ogb_sampler* s, int32_t which, const int64_t* idxs, int64_t n, ogb_batch** out);

/* The reference's helper methods, for explicit rows (host arrays in and out).
 * GCDataset.sample_goals (datasets.py:296-327): `draws` NULL = on-device Philox (advances the sampler's counter by one),
 * else the reference's own draws for this call (rand_pos, offset or dist, u_traj, u_cur). */
int ogb_sampler_sample_goals(ogb_sampler* s, const int64_t* idxs, int64_t n, double p_curgoal, double p_trajgoal, int32_t geom_sample,
                             double discount, const ogb_goal_draws* draws, int64_t* out_goal_idxs);
/* HGCDataset.compute_high_next_idxs (datasets.py:478-491) */
int ogb_sampler_compute_high_next_idxs(ogb_sampler* s, const int64_t* idxs, const int64_t* final_state_idxs, const int64_t* goal_idxs,
                                       int64_t n, int64_t subgoal_steps, int64_t* out_next, int64_t* out_steps);
/* GCDataset.augment / batched_random_crop (datasets.py:329-339, :17-33) for one image array: rows `idxs` of the
 * observations, row r cropped at crop[r] = (cy, cx) after edge padding by `padding` (0..127). */
int ogb_sampler_gather_cropped(ogb_sampler* s, const int64_t* idxs, int64_t n, const int64_t* crop, int32_t padding, ogb_batch** out);

/* ATCDataset (datasets.py:369-464), for samplers created with OGB_KIND_ATC.  The anchor set of a temporal offset k
 * (get_valid_atc_idxs, :417-436) is built once per k and cached, like the reference's _atc_valid_cache. */
int ogb_sampler_num_atc_anchors(ogb_sampler* s, int64_t k, int64_t* out);
int ogb_sampler_copy_atc_anchors(ogb_sampler* s, int64_t k, int64_t* out_host);
int ogb_sampler_sample_atc(ogb_sampler* s, int64_t batch_size, int32_t n_batches, int64_t k, int32_t evaluation,
                           const ogb_draws* draws, ogb_batch** out);

int ogb_batch_num_keys(const ogb_batch* b, int32_t* out);
int ogb_batch_key_info(const ogb_batch* b, int32_t i, ogb_key_info* out);
int ogb_batch_keep_leading_axis(ogb_batch* b, int32_t on);        /* shapes keep the [n_batches] axis even when n_batches == 1 */
int ogb_batch_nbytes(const ogb_batch* b, size_t* out);            /* size of the single device block */
int ogb_batch_device_block(const ogb_batch* b, void** out);       /* its base: key i lives at base + ogb_key_info.offset */
int ogb_batch_launches(const ogb_batch* b, int32_t* out);         /* kernels launched to produce it */
int ogb_batch_kernel_names(const ogb_batch* b, const char** buf, int32_t cap, int32_t* n_out);
                                                                  /* debug: the kernel of every launch, in issue order, named as
                                                                     ogb_batch_dominant_kernel names them (static strings); the
                                                                     first min(cap, n) go to buf, *n_out = n */
int ogb_batch_dominant_kernel(ogb_batch* b, const char** name, float* ms); /* the kernel that moved the batch's bytes, named with its
                                                                     template arguments as ncu prints them (the string lives
                                                                     as long as the batch), and, in profile mode, its device
                                                                     time (host-waits for it); else -1 */
int ogb_batch_sync(ogb_batch* b);                                 /* host-wait for the batch to be ready */
int ogb_batch_wait_on_stream(ogb_batch* b, void* consumer_stream);/* make a consumer stream wait (DLPack protocol) */
int ogb_batch_copy_to_host(ogb_batch* b, void* dst, size_t nbytes);  /* whole block, D2H, synchronous at return (= begin + end) */
int ogb_batch_copy_to_host_begin(ogb_batch* b, void* dst, size_t nbytes); /* enqueue that copy on the sampler's copy stream (behind the
                                                                     batch's kernels) and return: copies begun one after the other
                                                                     run back to back; `dst` (pinned) must stay valid until _end */
int ogb_batch_copy_to_host_end(ogb_batch* b);                     /* host-wait for the begun copy; raises the deferred index error */
int ogb_batch_copy_key_to_host(ogb_batch* b, int32_t i, void* dst, size_t nbytes); /* one key, D2H, synchronous */
int ogb_batch_copy_slice_to_host(ogb_batch* b, int32_t i, int64_t batch_index, void* dst, size_t nbytes); /* one batch of one key */
int ogb_batch_index_vector(ogb_batch* b, int32_t slot, int64_t* dst_host); /* debug: needs set_debug(1) */
int ogb_batch_check_gaps(ogb_batch* b, int64_t* n_bad);           /* debug: needs set_debug(2); bytes written outside every key */
int ogb_batch_crop_shifts(ogb_batch* b, int64_t* dst_host);       /* debug: [rows,2] applied (cy,cx), -1 if none */
/* DLPack export of key i (DLManagedTensor*, legacy v0 ABI); the deleter drops one reference on the batch. */
int ogb_batch_dlpack(ogb_batch* b, int32_t i, void** out_dl_managed_tensor);
/* ... of ONE batch of a multi-batch launch, as [batch, ...]: the i-th `sample(batch_size)` of impls/main.py:202 when the
 * K calls were drawn ahead in one launch (GCDataset(..., lookahead=K)). */
int ogb_batch_dlpack_slice(ogb_batch* b, int32_t i, int64_t batch_index, void** out_dl_managed_tensor);
int ogb_batch_mark_escaped(ogb_batch* b);                         /* a raw device pointer was handed out (e.g. __cuda_array_interface__):
                                                                     the block is recycled only after a device-wide sync */
int ogb_batch_retain(ogb_batch* b);
int ogb_batch_release(ogb_batch* b);

/* Pinned host staging for the numpy-returning mode of the Python wrapper. */
int ogb_host_alloc(size_t nbytes, void** out);
int ogb_host_free(void* p);

/* One-shot helpers used by tests and the build check. */
int ogb_searchsorted_warp(const int64_t* sorted_host, int64_t n, const int64_t* keys_host, int64_t m, int32_t side_right,
                          int32_t device, int64_t* out_host);      /* warp-cooperative searchsorted, np.searchsorted parity */
int ogb_philox_fill(uint64_t seed, uint32_t stream_id, uint64_t batch, uint32_t purpose, int64_t n, int32_t device,
                    uint32_t* out_host);                           /* [n,4] raw Philox4x32-10 words, for RNG tests */

int ogb_debug_timeline(double* out_ms, int32_t capacity, int32_t* n_out);
                                                                   /* debug (env OGB_TIMELINE=1): device times, in ms since the
                                                                      first, of index begin/end and gather begin/end per call */
int ogb_geometric_check(double discount, uint64_t seed, int64_t n, int32_t device, int64_t* mismatches);
                                                                   /* 2n geometric draws: float32 fast path vs the float64
                                                                      expression ceil(log(1-U)/log(discount)); counts differences */

#ifdef __cplusplus
}
#endif
#endif /* OGB_SAMPLER_H_ */
