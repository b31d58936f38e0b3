// The index algebra and the row-gather kernels of the replay sampler.
//
// relabel_row (one thread per batch row) restates the reference's per-row index algebra
// (impls/utils/datasets.py:296-327 sample_goals, :478-491 compute_high_next_idxs, :250-252 and :533-582
// rewards/masks; SURVEY.md Appendix E) from either injected draws (validation mode) or Philox draws.  It writes the
// scalar keys (masks, rewards, offsets, steps), copies the fields whose rows are <= 16 bytes, and leaves the dataset
// row of every index-vector slot in registers.  It runs inside
//   relabel_index_kernel      stand-alone (rows go to int32 index vectors in memory for the gather kernels),
//   relabel_gather_kernel     fused with the row gather: sample() is one launch.
//
// gather_rows_async_body gathers the dataset rows those slots name (datasets.py:78-83 get_subset, :341-357
// get_observations / get_goal_observations) into the dense output arrays: per-warp cp.async rings, span jobs over the
// packed record table, coalesced 16-byte stores.  gather_rows_kernel<V> is the register-staged form for rows > 4 KB.
#pragma once
#include "device_common.cuh"

namespace ogb {

constexpr int kMaxSlots = 10;
constexpr int kMaxRowJobs = 24;
constexpr int kRelabelThreads = 256;
constexpr int kGatherMinBlocks = 4;   // resident CTAs per SM the gather kernel is compiled for (register cap 64)

// index-vector slots
enum : int {
  SLOT_IDX = 0, SLOT_NEXT = 1,
  GC_VALUE_GOAL = 2, GC_ACTOR_GOAL = 3, GC_NUM_SLOTS = 4,
  GC_TRL_MID = 4, GC_TRL_PLUS1 = 5, GC_TRL_NUM_SLOTS = 6,
  HGC_HV_GOAL = 2, HGC_HV_NEXT = 3, HGC_LV_NEXT = 4, HGC_HA_GOAL = 5, HGC_HA_NEXT = 6, HGC_LA_GOAL = 7,
  HGC_LA_NEXT = 8, HGC_LV_GOAL = 9, HGC_NUM_SLOTS = 10
};

struct GoalSpec {
  // Philox mode: the goal-mix coins are 32-bit words w, and (w * 2^-32 < p) <=> (w < ceil(p * 2^32)) exactly, so the
  // kernel compares integers; *_always covers thresholds >= 2^32 (p >= 1)
  uint32_t thr_traj32, thr_cur32;
  uint8_t traj_always, cur_always;
  uint8_t geom;      // geometric (1) or uniform-in-remainder (0) future goals
  uint8_t cur_only;  // p_curgoal == 1.0 short-circuit (datasets.py:317-318)
  float geo_abs_margin;  // absolute slack of the float32 geometric estimate, 2^-26 / |log(1-p)|
  double thr_traj;   // p_trajgoal / (1.0 - p_curgoal), float64 as the reference evaluates it (datasets.py:321)
  double p_cur;
  double log_1mp;    // log(1 - (1 - discount)) for the geometric inversion
};

struct GoalInject {
  const int64_t* rand_pos;
  const int64_t* offset;
  const double* dist;
  const double* u_traj;
  const double* u_cur;
};

struct RowJob {
  const uint8_t* src;   // field base in HBM
  uint8_t* dst;         // dense output [total_rows, row_bytes]
  uint32_t src_stride;  // padded row stride of the resident copy
  uint32_t row_bytes;   // dense output row size
  uint16_t epr;         // elements (of 1 << vec_log2 bytes) per row
  uint16_t n_coliter;   // ceil(epr / lanes-per-row)
  uint8_t vec_log2;     // element = 1,2,4,8,16 bytes
  uint8_t lpr_log2;     // lanes per row = 1 << lpr_log2 (<= 32)
  uint8_t slot;         // which index vector names the source rows
  uint8_t pad_;
};

// A field whose whole row is at most 16 bytes (terminals, valids, 2-D observations ...) is gathered by the index
// kernel itself: the thread that computed row g's index vectors copies those few bytes straight away.
constexpr int kMaxTinyJobs = 16;
struct TinyJob {
  const uint8_t* src;
  uint8_t* dst;
  uint8_t slot;
  uint8_t size_log2;   // element size
  uint8_t n_elem;      // row = n_elem elements (<= 16 bytes in total)
  uint8_t row_bytes;
  uint16_t stride;     // resident row stride (row_bytes, or the stride of the packed record table)
  uint16_t pad2_;
};

// Tiny fields that sit next to each other in the packed record table and are gathered through the same index vector
// (observations, actions, terminals, valids of a point-maze transition: 24 bytes of one 32-byte record) are loaded
// ONCE: one or two 16-byte loads per group, the fields are then cut out of registers.  The index kernel is bound by
// scattered-load wavefronts (L1TEX), not by ALU work, so trading three loads for a few selects pays.
constexpr int kMaxTinyGroups = 2;
constexpr int kMaxTinyFields = 16;
struct TinyGroup {
  const uint8_t* src;   // record table base + 16-byte aligned span offset
  uint16_t stride;
  uint8_t slot;
  uint8_t n_vec;        // 16-byte loads: 1 or 2
  uint8_t first_field;  // into RelabelParams::tiny_fields
  uint8_t n_fields;
  uint16_t pad_;
};
struct TinyField {
  uint8_t* dst;
  uint8_t word;         // first 4-byte word of the field inside the group's span (0..7)
  uint8_t n_words;      // 1..4
  uint8_t group;
  uint8_t pad_[5];
};

struct RelabelParams {
  // ---- dataset-side tables (all int32, resident) ----
  const int32_t* term;         // terminal_locs (datasets.py:186)
  const int32_t* term_bucket;  // lower_bound(term, b << term_shift)
  const int32_t* valid_table;  // valid_idxs (datasets.py:63) -- valid_mode 1
  const int32_t* gap_c;        // valid_mode 2: c[m] = (m-th invalid row) - m; valid_idxs[j] = j + #{m: c[m] <= j}
  const int32_t* gap_bucket;
  int64_t n_choices;           // len(valid_idxs), or size when the dataset has no 'valids'
  int32_t n_rows_ds;
  int32_t term_shift;
  int32_t gap_shift;
  int32_t valid_mode;          // 0: no 'valids'; 1: table; 2: gap ranks; 3: segment table (one probe, see valid_row_fast)
  const int4* seg_table;       // valid_mode 3, one entry per bucket b of 2^seg_shift positions, lo = lower_bound(c, b << seg_shift):
                               //   {c[lo] (INT_MAX past the end), final_state(segment lo), final_state(segment lo+1), lo}
  const int32_t* seg_bucket;   // (unused: the bucket table is folded into seg_table)
  int32_t seg_shift;
  int32_t n_seg_table;         // entries of seg_table / seg_bucket (for the shared-memory copy of the index kernel)
  int32_t n_seg_bucket;
  int32_t pad_seg_;
  // ---- sampler config ----
  GoalSpec goal[3];            // value, low-value, actor
  const double* neg_lut;       // -(1 - discount**s)/(1 - discount)
  const double* pow_lut;       // discount**s
  int32_t kind;                // 0 GC, 1 HGC, 2 PLAIN, 3 ATC
  int32_t next_offset;         // SLOT_NEXT = idx + next_offset (1; the temporal offset k for ATC)
  int32_t trl;                 // TRL branch of GCDataset.sample (datasets.py:254-276)
  const int64_t* in_trl_mid;   // injected randint(idxs, value_goal_idxs)
  int64_t* trl_offsets;
  int64_t* trl_mid_offsets;
  int32_t has_low_goal;
  int32_t k_val, k_act, k_lo;
  int32_t gc_negative;
  int32_t stacked_next;        // frame_stack set: next_observations uses un-clamped idx+1 (datasets.py:231)
  int32_t actor_mix;           // the actor goal mix is a real random choice: draw its two coins (PURPOSE_MIX)
  int32_t aug_mode;            // draw the per-batch coin (p_aug is not None and not evaluation)
  int32_t crop_pad;
  double p_aug;
  // ---- randomness ----
  RngKey key;
  uint64_t batch0;
  const int64_t* in_idx_pos;
  GoalInject in_goal[3];
  const int64_t* in_crop;
  double in_coin;
  const int64_t* given_idxs;
  int32_t* idx_error;          // deferred index check (host-output mode): set to 1 when a given index is out of range
  int64_t idx_last;            //   largest admissible index
  // ---- launch shape ----
  int64_t batch;               // rows per sample() call
  uint64_t batch_magic;        // ceil(2^64 / batch), 0 when batch == 1: g / batch == umul64hi(g, magic) for g < 2^32
  int64_t total_rows;          // batch * n_batches (also the stride of the [slot][row] index vectors)
  int64_t row_begin, row_end;  // rows this launch handles
  int32_t n_slots;
  int32_t narrow;              // jax_compat: the scalar outputs below are float32 / int32 arrays
  int32_t pad1_[2];
  // ---- scalar outputs (float64 / int64 like the reference; float32 / int32 when `narrow`) ----
  double* masks;
  double* rewards;
  int64_t* hv_offsets;
  int64_t* hv_steps;
  int64_t* lv_steps;
  double* hv_masks;
  double* hv_rewards;
  double* lv_masks;
  double* lv_rewards;
  // ---- index outputs: [slot][total_rows] ----
  int32_t* vec_rows;           // row index vectors, consumed by the gather kernels
  int32_t* vec_init;           // first row of each row's trajectory segment (frame stacking only; may be null)
  int8_t* crop_out;            // [total_rows][2] (dy, dx) or -128 when the batch is not augmented (may be null)
  // ---- rows of <= 16 bytes, copied by the index kernel ----
  int32_t n_tiny;              // the first n_tiny_fast of them have rows of 4, 8 or 16 bytes
  int32_t n_tiny_fast;
  int32_t write_vecs;          // 0: no later kernel needs the index vectors (everything was tiny) and debug is off
  TinyJob tiny[kMaxTinyJobs];
  int32_t n_tiny_groups;
  int32_t n_tiny_fields;
  TinyGroup tiny_groups[kMaxTinyGroups];
  TinyField tiny_fields[kMaxTinyFields];
};

// scalar keys: float64 / int64 as the reference returns them, or -- jax_compat -- the float32 / int32 that `jit` narrows
// them to with x64 off ((float)double rounds to nearest even like numpy's astype; the integers are far below 2^31)
__device__ __forceinline__ void put_f64(const RelabelParams& p, double* base, const int64_t g, const double v) {
  if (p.narrow) reinterpret_cast<float*>(base)[g] = (float)v; else base[g] = v;
}
__device__ __forceinline__ void put_i64(const RelabelParams& p, int64_t* base, const int64_t g, const int64_t v) {
  if (p.narrow) reinterpret_cast<int32_t*>(base)[g] = (int32_t)v; else base[g] = v;
}

// word `i` (0..7) of the eight words held in two uint4
__device__ __forceinline__ uint32_t select_word(const uint4& a, const uint4& b, const uint32_t i) {
  const uint4 t = (i & 4u) ? b : a;
  const uint2 h = (i & 2u) ? make_uint2(t.z, t.w) : make_uint2(t.x, t.y);
  return (i & 1u) ? h.y : h.x;
}

// valid_mode 3 -- datasets whose invalid rows are far apart (every compact OGBench dataset: one per trajectory) and
// whose trajectories end where their valid rows end.  Position pos among the valid rows falls into segment
// m = #{invalid rows before it} = upper_bound(c, pos); buckets are narrower than the smallest gap between two c[m],
// so a bucket holds at most one boundary, and the table has one entry PER BUCKET that carries everything the bucket
// can answer: {the boundary c[lo] inside or after it, final_state(segment lo), final_state(segment lo + 1), lo}.
// One 16-byte load gives the row AND the trajectory's final state (datasets.py:306 needs a second search in the
// reference).
// Where the segment table is read from: global memory (read-only path), or the copy a persistent index kernel made in
// shared memory (scattered 4/16-byte table reads then cost bank cycles instead of L1TEX tag lookups).
struct SegView {
  const int32_t* bucket;
  const int4* table;
};

template <bool kSmemTables>
__device__ __forceinline__ int32_t valid_row_fast(const RelabelParams& p, const SegView& seg, const uint32_t pos, int32_t& fin) {
  const int4 e = kSmemTables ? seg.table[pos >> p.seg_shift] : __ldg(seg.table + (pos >> p.seg_shift));   // ONE 16-byte load
  const bool past = e.x <= (int32_t)pos;
  fin = past ? e.z : e.y;
  return (int32_t)pos + e.w + (past ? 1 : 0);
}

// the general forms (no 'valids', explicit table, gap ranks with a binary search): out of line, the segment table
// serves every compact OGBench dataset
__device__ __noinline__ int32_t valid_row_general(const RelabelParams& p, int64_t pos) {
  if (p.valid_mode == 0) return (int32_t)pos;
  if (p.valid_mode == 1) return __ldg(p.valid_table + pos);
  const int j = (int)pos;
  return j + lower_bound_bucketed(p.gap_c, p.gap_bucket, p.gap_shift, j + 1);  // upper_bound(c, j)
}

template <bool kSmemTables, bool kSegOnly = false>
__device__ __forceinline__ int32_t valid_row(const RelabelParams& p, const SegView& seg, int64_t pos) {
  if (kSegOnly || p.valid_mode == 3) { int32_t unused; return valid_row_fast<kSmemTables>(p, seg, (uint32_t)pos, unused); }
  return valid_row_general(p, pos);
}

// datasets.py:313-316 -- float64, separate multiply/add (no FMA contraction), round half to even
__device__ __forceinline__ int32_t uniform_future_goal(int32_t i, int32_t fin, double d) {
  const int32_t lo = (i + 1 < fin) ? i + 1 : fin;
  return (int32_t)rint(__dadd_rn(__dmul_rn((double)lo, d), __dmul_rn((double)fin, __dsub_rn(1.0, d))));
}

// Validation mode: the reference's own draws (float64 uniforms, int64 offsets) decide.
template <bool kSmemTables, bool kSegOnly = false>
__device__ __forceinline__ int32_t pick_goal_injected(const RelabelParams& p, const SegView& seg, const int gs, const int32_t i,
                                                      const int32_t fin, const int64_t g) {
  const GoalSpec& s = p.goal[gs];
  if (s.cur_only) return i;                                  // p_curgoal == 1.0  (datasets.py:317-318)
  const GoalInject& in = p.in_goal[gs];
  if (in.u_cur[g] < s.p_cur) return i;                       // np.where(rand < p_cur, idxs, ...)  :325
  if (!(in.u_traj[g] < s.thr_traj)) return valid_row<kSmemTables, kSegOnly>(p, seg, in.rand_pos[g]);   // random goal  :303,:320-322
  if (s.geom) {                                              // :309-310
    const int64_t t = (int64_t)i + in.offset[g];
    return (int32_t)(t < (int64_t)fin ? t : (int64_t)fin);
  }
  return uniform_future_goal(i, fin, in.dist[g]);
}

// Philox mode: `mix` = (u_traj, u_cur) as 32-bit words, `bits` = the 64 random bits of this goal set, spent either
// on the random-goal position or on the geometric / distance uniform -- never both, since the mix decides first.
template <bool kSmemTables, bool kSegOnly = false>
__device__ __forceinline__ int32_t pick_goal_philox(const RelabelParams& p, const SegView& seg, const int gs, const int32_t i,
                                                    const int32_t fin, const uint2 mix, const uint2 bits) {
  const GoalSpec& s = p.goal[gs];
  if (s.cur_only) return i;
  if (s.cur_always || mix.y < s.thr_cur32) return i;
  if (!(s.traj_always || mix.x < s.thr_traj32)) return valid_row<kSmemTables, kSegOnly>(p, seg, bounded_u32n(bits.x, bits.y, (uint32_t)p.n_choices));
  if (s.geom) {
    const int64_t t = (int64_t)i + geometric_from_words(bits.x, bits.y, s.log_1mp, s.geo_abs_margin);
    return (int32_t)(t < (int64_t)fin ? t : (int64_t)fin);
  }
  return uniform_future_goal(i, fin, unit_double(bits.x, bits.y));
}

// datasets.py:478-491
__device__ __forceinline__ void subgoal_step(int32_t i, int32_t fin, int32_t goal, int32_t k, int32_t& next, int32_t& s) {
  s = fin - i < k ? fin - i : k;
  const int32_t d = goal - i;
  if (0 <= d && d < s) s = d;
  next = i + s;
}

// (frame stacking only; out of line so that the put_slot sites do not each carry a search)
__device__ __noinline__ int32_t trajectory_first_row(const RelabelParams& p, int32_t x) {
  // initial_locs[searchsorted(initial_locs, x, 'right') - 1] (datasets.py:361) expressed on terminal_locs:
  // with t = lower_bound(term, x) the start is 0 when t == 0, else term[t-1] + 1.
  x = x < p.n_rows_ds ? x : p.n_rows_ds - 1;
  const int t = lower_bound_bucketed(p.term, p.term_bucket, p.term_shift, x);
  return t == 0 ? 0 : __ldg(p.term + t - 1) + 1;
}

// kLean (the point-maze kernel): the host has checked that no later kernel reads the index vectors and that there is no
// frame stacking, so the two stores and their parameter loads are compiled out.
template <bool kLean = false>
__device__ __forceinline__ void put_slot(const RelabelParams& p, int32_t* sr, const int slot, const int64_t g, const int32_t x) {
  sr[slot] = x;  // `slot` is a compile-time constant at every call site, so sr[] stays in registers
  if (kLean) return;
  if (p.write_vecs) p.vec_rows[(int64_t)slot * p.total_rows + g] = x;
  if (p.vec_init != nullptr) p.vec_init[(int64_t)slot * p.total_rows + g] = trajectory_first_row(p, x);
}

template <int kSlots>
__device__ __forceinline__ int32_t pick_slot(const int32_t* sr, const int slot) {
  int32_t x = sr[0];
#pragma unroll
  for (int v = 1; v < kSlots; ++v) x = (slot == v) ? sr[v] : x;
  return x;
}

// kernel flavours: which index algebra is compiled in
enum : int { FLAVOUR_GC = 0, FLAVOUR_HGC = 1, FLAVOUR_PLAIN = 2 };  // PLAIN also serves ATC (index + offset, crop)
template <int kFlavour> struct FlavourSlots { static constexpr int value = kFlavour == FLAVOUR_GC ? GC_TRL_NUM_SLOTS : (kFlavour == FLAVOUR_HGC ? HGC_NUM_SLOTS : 2); };

__device__ __forceinline__ void split_row(const RelabelParams& p, const int64_t g, uint64_t& batch_id, uint32_t& r) {
  // g / batch with the host's magic number; g < 2^32 (a launch holds at most 2^31 rows)
  const uint32_t g32 = (uint32_t)g;
  uint32_t kb = g32;
  if (p.batch_magic != 0) {
    const uint64_t lo = (uint64_t)g32 * (uint32_t)p.batch_magic;
    const uint64_t hi = (uint64_t)g32 * (uint32_t)(p.batch_magic >> 32) + (lo >> 32);
    kb = (uint32_t)(hi >> 32);
  } else if (p.batch != 1) {
    kb = (uint32_t)(g / p.batch);   // batch >= 2^32: never on the fast path
  }
  r = g32 - kb * (uint32_t)p.batch;
  batch_id = p.batch0 + (uint64_t)kb;
}

// All per-row work of sample(): index draws, goal relabelling, rewards/masks, the rows of <= 16 bytes, crop shifts.
// On return sr[] holds the dataset row of every slot for batch row g.
// kPoint: the copies of the point-maze record are compiled in (see the host's point_record check): ONE tiny group of the
// transition's own 32-byte record laid out as observations f32[2] | actions f32[2] | terminals | valids | shadow next
// observation f32[2], plus the two 8-byte goal rows.  The generic descriptor walk below costs ~420 of the index kernel's
// ~820 instructions per 32 rows on that shape (profiles/r2_c1_lines_before.txt); with the layout fixed at compile time it
// is 4 loads and 7 stores.  Every OGBench pointmaze dataset has this shape; anything else takes the generic path.
template <bool kInject, int kFlavour, bool kSmemTables = false, bool kPoint = false>
__device__ __forceinline__ void relabel_row(const RelabelParams& p, const SegView& seg, const int64_t g, int32_t* sr) {
  constexpr int kSlots = FlavourSlots<kFlavour>::value;
  uint64_t batch_id;
  uint32_t r;
  split_row(p, g, batch_id, r);

  uint4 w0 = make_uint4(0, 0, 0, 0);
  if (!kInject) w0 = draw4(p.key, batch_id, r, PURPOSE_IDX);
  int32_t i, fin = -1;
  if (p.given_idxs != nullptr) {
    const int64_t given = p.given_idxs[g];
    i = (int32_t)given;
    if (p.idx_error != nullptr && (uint64_t)given > (uint64_t)p.idx_last) {   // negative or too large: report, stay in bounds
      *p.idx_error = 1;
      i = 0;
    }
  } else {
    const int64_t pos = kInject ? p.in_idx_pos[g] : (int64_t)bounded_u32n(w0.x, w0.y, (uint32_t)p.n_choices);
    if (kPoint || p.valid_mode == 3) i = valid_row_fast<kSmemTables>(p, seg, (uint32_t)pos, fin);  // datasets.py:65-70 and :306 in one probe
    else i = valid_row<kSmemTables>(p, seg, pos);
  }
  put_slot<kPoint>(p, sr, SLOT_IDX, g, i);
  // Grouped tiny fields of the transition's own record (observations, actions, terminals, valids of a point-maze row,
  // plus the shadow copy of the next row's observation): fetched NOW, so the load flies under the goal algebra below
  // (its first use was the hottest stall of C1's launch, 14 % of the samples, when it was issued after the goals).
  uint4 grp_a[kMaxTinyGroups], grp_b[kMaxTinyGroups];
#pragma unroll
  for (int u = 0; u < kMaxTinyGroups; ++u) {
    grp_a[u] = make_uint4(0, 0, 0, 0);
    grp_b[u] = make_uint4(0, 0, 0, 0);
    if (kPoint ? u == 0 : (u < p.n_tiny_groups && p.tiny_groups[u].slot == SLOT_IDX)) {
      const TinyGroup& grp = p.tiny_groups[u];
      const uint4* sp = reinterpret_cast<const uint4*>(grp.src + (size_t)(uint32_t)i * grp.stride);
      if (kPoint) {   // the 32-byte record in one 256-bit load: +1.2 % on C1 over two 128-bit loads (0.740 vs 0.731, batch r2l)
        asm volatile("ld.global.nc.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=r"(grp_a[u].x), "=r"(grp_a[u].y), "=r"(grp_a[u].z), "=r"(grp_a[u].w), "=r"(grp_b[u].x), "=r"(grp_b[u].y),
                       "=r"(grp_b[u].z), "=r"(grp_b[u].w)
                     : "l"(sp));
      } else {
        grp_a[u] = __ldg(sp);
        if (grp.n_vec > 1) grp_b[u] = __ldg(sp + 1);
      }
    }
  }
  // :82 clamps idx + 1 to size - 1; with frame stacking (:231) and for ATC (:408) the reference does not clamp, and a
  // row past the table is an IndexError there: here the gather stays inside the table and the error is reported through
  // the deferred index flag when the caller enabled it
  if (!kPoint) {   // (the point-maze record carries the next row's observation itself: nothing gathers through SLOT_NEXT)
    int32_t nxt = i + p.next_offset;
    if (nxt >= p.n_rows_ds) {
      nxt = p.n_rows_ds - 1;
      if (p.stacked_next && p.idx_error != nullptr) *p.idx_error = 1;
    }
    put_slot(p, sr, SLOT_NEXT, g, nxt);
  }

  if (kFlavour != FLAVOUR_PLAIN) {
    uint4 gb = make_uint4(0, 0, 0, 0), amix = make_uint4(0, 0, 0, 0);
    if (!kInject) {
      gb = draw4(p.key, batch_id, r, PURPOSE_GOAL);
      if (p.actor_mix) amix = draw4_cold(p.key, batch_id, r, PURPOSE_MIX);
    }
    if (fin < 0) {                                                      // final_state_idxs  :306,:505
      const int tl = lower_bound_bucketed(p.term, p.term_bucket, p.term_shift, i);
      fin = __ldg(p.term + tl);
    }
    const double neg = p.gc_negative ? 1.0 : 0.0;
    const int32_t vg = kInject ? pick_goal_injected<kSmemTables, kPoint>(p, seg, 0, i, fin, g)           // :233-239 / :508-514
                               : pick_goal_philox<kSmemTables, kPoint>(p, seg, 0, i, fin, make_uint2(w0.z, w0.w), make_uint2(gb.x, gb.y));
    const int32_t ag = kInject ? pick_goal_injected<kSmemTables, kPoint>(p, seg, 2, i, fin, g)           // :240-246 / :585-591
                               : pick_goal_philox<kSmemTables, kPoint>(p, seg, 2, i, fin, make_uint2(amix.x, amix.y), make_uint2(gb.z, gb.w));
    const double succ = (i == vg) ? 1.0 : 0.0;                         // :250-252 / :579-582
    put_f64(p, p.masks, g, 1.0 - succ);
    put_f64(p, p.rewards, g, succ - neg);
    if (kFlavour == FLAVOUR_GC) {
      put_slot<kPoint>(p, sr, GC_VALUE_GOAL, g, vg);
      put_slot<kPoint>(p, sr, GC_ACTOR_GOAL, g, ag);
      if (!kPoint && p.trl) {                                                     // :259-267
        const int64_t span = vg > i ? (int64_t)vg - i : 1;             // the reference asserts idxs != value_goal_idxs
        int32_t mid;
        if (kInject) {
          mid = (int32_t)p.in_trl_mid[g];
        } else {
          const uint4 t = draw4_cold(p.key, batch_id, r, PURPOSE_TRL_MID);
          mid = i + (int32_t)bounded_u32n(t.x, t.y, (uint32_t)span);   // randint(idxs, value_goal_idxs): [i, vg)
        }
        put_slot(p, sr, GC_TRL_MID, g, mid);
        put_slot(p, sr, GC_TRL_PLUS1, g, i + 1);
        put_i64(p, p.trl_offsets, g, (int64_t)vg - i);
        put_i64(p, p.trl_mid_offsets, g, (int64_t)mid - i);
      }
    } else {
      const int32_t hv = vg;
      int32_t hv_next, hv_s, lv_next, lv_s;
      subgoal_step(i, fin, hv, p.k_val, hv_next, hv_s);                             // :519-524
      subgoal_step(i, fin, hv, p.k_lo, lv_next, lv_s);                              // :544-549
      put_slot(p, sr, HGC_HV_GOAL, g, hv);
      put_slot(p, sr, HGC_HV_NEXT, g, hv_next);
      put_slot(p, sr, HGC_LV_NEXT, g, lv_next);
      put_i64(p, p.hv_offsets, g, (int64_t)hv - (int64_t)i);                                   // :531
      put_i64(p, p.hv_steps, g, hv_s);
      put_i64(p, p.lv_steps, g, lv_s);
      const double hv_succ = hv_s < p.k_val ? 1.0 : 0.0;                            // :533
      const double lv_succ = lv_s < p.k_lo ? 1.0 : 0.0;                             // :552
      put_f64(p, p.hv_masks, g, 1.0 - hv_succ);
      put_f64(p, p.hv_rewards, g, p.gc_negative ? __ldg(p.neg_lut + hv_s) : __dmul_rn(__ldg(p.pow_lut + hv_s), hv_succ));
      double lv_mask = 1.0 - lv_succ;
      double lv_rew = p.gc_negative ? __ldg(p.neg_lut + lv_s) : __dmul_rn(__ldg(p.pow_lut + lv_s), lv_succ);
      if (p.has_low_goal) {                                                         // :563-576
        int32_t lvg;
        if (kInject) {
          lvg = pick_goal_injected<kSmemTables>(p, seg, 1, i, fin, g);
        } else {
          const uint4 lb = draw4_cold(p.key, batch_id, r, PURPOSE_GOAL_LOW);
          lvg = pick_goal_philox<kSmemTables>(p, seg, 1, i, fin, make_uint2(lb.z, lb.w), make_uint2(lb.x, lb.y));
        }
        put_slot(p, sr, HGC_LV_GOAL, g, lvg);
        const double s = (i == lvg) ? 1.0 : 0.0;
        lv_mask = 1.0 - s;
        lv_rew = s - neg;
      }
      put_f64(p, p.lv_masks, g, lv_mask);
      put_f64(p, p.lv_rewards, g, lv_rew);
      const int32_t ha = ag;
      int32_t ha_next, la_next, unused;
      subgoal_step(i, fin, ha, p.k_act, ha_next, unused);                           // :595-600
      subgoal_step(i, fin, ha, p.k_lo, la_next, unused);                            // :613-618
      const int64_t la = (int64_t)i + p.k_act;                                      // :610
      put_slot(p, sr, HGC_HA_GOAL, g, ha);
      put_slot(p, sr, HGC_HA_NEXT, g, ha_next);
      put_slot(p, sr, HGC_LA_GOAL, g, (int32_t)(la < (int64_t)fin ? la : (int64_t)fin));
      put_slot(p, sr, HGC_LA_NEXT, g, la_next);
    }
  }

  if (kPoint) {
    const uint2 vgo = __ldg(reinterpret_cast<const uint2*>(p.tiny[0].src + (size_t)(uint32_t)sr[GC_VALUE_GOAL] * p.tiny[0].stride));
    const uint2 ago = __ldg(reinterpret_cast<const uint2*>(p.tiny[1].src + (size_t)(uint32_t)sr[GC_ACTOR_GOAL] * p.tiny[1].stride));
    reinterpret_cast<uint2*>(p.tiny_fields[0].dst)[g] = make_uint2(grp_a[0].x, grp_a[0].y);     // observations
    reinterpret_cast<uint2*>(p.tiny_fields[1].dst)[g] = make_uint2(grp_a[0].z, grp_a[0].w);     // actions
    reinterpret_cast<uint32_t*>(p.tiny_fields[2].dst)[g] = grp_b[0].x;                          // terminals
    reinterpret_cast<uint32_t*>(p.tiny_fields[3].dst)[g] = grp_b[0].y;                          // valids
    reinterpret_cast<uint2*>(p.tiny_fields[4].dst)[g] = make_uint2(grp_b[0].z, grp_b[0].w);     // next_observations (shadow)
    reinterpret_cast<uint2*>(p.tiny[0].dst)[g] = vgo;                                           // value_goals
    reinterpret_cast<uint2*>(p.tiny[1].dst)[g] = ago;                                           // actor_goals
  } else {
  // grouped tiny fields: one record load per group (the groups of the transition's own row were fetched above), all
  // loads issued before any store.  (Unrolling the field and job loops completely, so that the descriptors sit at fixed
  // constant-bank offsets, was measured: the code growth costs more than the saved LDCs, 0.052 vs 0.047 ms on C1 and
  // 0.223 vs 0.203 ms on C2's fused kernel.)
  {
#pragma unroll
    for (int u = 0; u < kMaxTinyGroups; ++u) {
      if (u < p.n_tiny_groups && p.tiny_groups[u].slot != SLOT_IDX) {
        const TinyGroup& grp = p.tiny_groups[u];
        const uint4* sp = reinterpret_cast<const uint4*>(grp.src + (size_t)(uint32_t)pick_slot<kSlots>(sr, grp.slot) * grp.stride);
        grp_a[u] = __ldg(sp);
        if (grp.n_vec > 1) grp_b[u] = __ldg(sp + 1);
      }
    }
#pragma unroll 1
    for (int f = 0; f < p.n_tiny_fields; ++f) {
      const TinyField& fld = p.tiny_fields[f];
      uint4 a = grp_a[0], b = grp_b[0];
#pragma unroll
      for (int u = 1; u < kMaxTinyGroups; ++u)
        if (fld.group == u) { a = grp_a[u]; b = grp_b[u]; }
      uint32_t* dp = reinterpret_cast<uint32_t*>(fld.dst) + (size_t)g * fld.n_words;
      const uint32_t w0 = select_word(a, b, fld.word);
      if (fld.n_words == 1) {
        dp[0] = w0;
      } else if (fld.n_words == 2) {
        *reinterpret_cast<uint2*>(dp) = make_uint2(w0, select_word(a, b, fld.word + 1u));
      } else if (fld.n_words == 4) {
        *reinterpret_cast<uint4*>(dp) = (fld.word & 4u) ? b : a;
      } else {
        dp[0] = w0; dp[1] = select_word(a, b, fld.word + 1u); dp[2] = select_word(a, b, fld.word + 2u);
      }
    }
  }

  // rows of <= 16 bytes: this thread copies them now (datasets.py:78-83 for the per-transition fields).  Rows of 4, 8
  // or 16 bytes (the host lists them first) are loaded four jobs at a time before any is stored, so their L2 latencies
  // overlap; any other size is copied element by element.
#pragma unroll 1
  for (int j0 = 0; j0 < p.n_tiny_fast; j0 += 4) {
    uint4 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (j0 + u < p.n_tiny_fast) {
        const TinyJob& job = p.tiny[j0 + u];
        const uint8_t* sp = job.src + (size_t)(uint32_t)pick_slot<kSlots>(sr, job.slot) * job.stride;
        if (job.row_bytes == 4) v[u].x = __ldg(reinterpret_cast<const uint32_t*>(sp));
        else if (job.row_bytes == 8) { const uint2 t = __ldg(reinterpret_cast<const uint2*>(sp)); v[u].x = t.x; v[u].y = t.y; }
        else v[u] = __ldg(reinterpret_cast<const uint4*>(sp));
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (j0 + u < p.n_tiny_fast) {
        const TinyJob& job = p.tiny[j0 + u];
        uint8_t* dp = job.dst + (size_t)g * job.row_bytes;
        if (job.row_bytes == 4) *reinterpret_cast<uint32_t*>(dp) = v[u].x;
        else if (job.row_bytes == 8) *reinterpret_cast<uint2*>(dp) = make_uint2(v[u].x, v[u].y);
        else *reinterpret_cast<uint4*>(dp) = v[u];
      }
    }
  }
#pragma unroll 1
  for (int j = p.n_tiny_fast; j < p.n_tiny; ++j) {
    const TinyJob& job = p.tiny[j];
    const uint8_t* sp = job.src + (size_t)(uint32_t)pick_slot<kSlots>(sr, job.slot) * job.stride;
    uint8_t* dp = job.dst + (size_t)g * job.row_bytes;
    if (job.size_log2 == 2) for (int e = 0; e < job.n_elem; ++e) reinterpret_cast<uint32_t*>(dp)[e] = __ldg(reinterpret_cast<const uint32_t*>(sp) + e);
    else if (job.size_log2 == 1) for (int e = 0; e < job.n_elem; ++e) reinterpret_cast<uint16_t*>(dp)[e] = __ldg(reinterpret_cast<const uint16_t*>(sp) + e);
    else for (uint32_t e = 0; e < job.row_bytes; ++e) dp[e] = __ldg(sp + e);
  }

  }

  if (p.crop_out != nullptr) {
    int dy = -128, dx = -128;
    if (p.aug_mode) {                                                               // :278-279, :621-622
      double coin;
      if (kInject) {
        coin = p.in_coin;
      } else {
        const uint4 c = draw4_cold(p.key, batch_id, 0xFFFFFFFFu, PURPOSE_COIN);
        coin = unit_double(c.x, c.y);
      }
      if (coin < p.p_aug) {                                                         // :333
        int cy, cx;
        if (kInject) {
          cy = (int)p.in_crop[2 * g];
          cx = (int)p.in_crop[2 * g + 1];
        } else {
          const uint32_t span = 2u * (uint32_t)p.crop_pad + 1u;
          const uint4 cw = draw4_cold(p.key, batch_id, r, PURPOSE_CROP);
          const uint32_t joint = __umulhi(cw.x, span * span);          // (cy, cx) jointly uniform on span x span
          cy = (int)(joint / span);
          cx = (int)(joint % span);
        }
        dy = cy - p.crop_pad;
        dx = cx - p.crop_pad;
      }
    }
    p.crop_out[2 * g] = (int8_t)dy;
    p.crop_out[2 * g + 1] = (int8_t)dx;
  }
}

// kSmemTables: a persistent grid (a few CTAs per SM) whose CTAs first copy the segment table into shared memory
// (dynamic: 16 B * n_seg_table + 4 B * n_seg_bucket) and then walk the rows with a grid stride.
template <bool kInject, int kFlavour, bool kSmemTables, bool kPoint = false, int kMinBlocks = 4>
__global__ void __launch_bounds__(kRelabelThreads, kMinBlocks) relabel_index_kernel(const __grid_constant__ RelabelParams p) {
  extern __shared__ __align__(16) uint8_t smem_tables[];
  SegView seg{p.seg_bucket, p.seg_table};
  if (kSmemTables) {
    int4* s_table = reinterpret_cast<int4*>(smem_tables);
    int32_t* s_bucket = reinterpret_cast<int32_t*>(s_table + p.n_seg_table);
    for (int t = threadIdx.x; t < p.n_seg_table; t += blockDim.x) s_table[t] = __ldg(p.seg_table + t);
    for (int t = threadIdx.x; t < p.n_seg_bucket; t += blockDim.x) s_bucket[t] = __ldg(p.seg_bucket + t);
    __syncthreads();
    seg.bucket = s_bucket;
    seg.table = s_table;
  }
  for (int64_t g = p.row_begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < p.row_end; g += (int64_t)gridDim.x * blockDim.x) {
    int32_t sr[kMaxSlots];
#pragma unroll
    for (int v = 0; v < kMaxSlots; ++v) sr[v] = 0;
    relabel_row<kInject, kFlavour, kSmemTables, kPoint>(p, seg, g, sr);
  }
}

// ---------------------------------------------------------------------------------------------------------
// Row gather.  Each warp owns 32 consecutive batch rows and walks the job list; lane l holds the source row of
// batch row l for the current job and broadcasts it with a shuffle.  A warp-wide access covers 32 >> lpr_log2
// rows of (1 << lpr_log2) elements (short rows) or one 32-element slice of one row (long rows).  Every warp
// issues kU independent loads before the matching stores so that enough bytes are in flight to cover HBM
// latency; there is no block-level synchronisation at all.
// ---------------------------------------------------------------------------------------------------------
struct GatherParams {
  const int32_t* vec_rows;     // [slot][total_rows]
  int64_t total_rows;
  int64_t row_begin, row_end;  // row_begin is a multiple of 32
  int32_t n_jobs;
  RowJob jobs[kMaxRowJobs];
};

// read-once data: do not allocate in L1 (keeps the small index / table lines resident)
__device__ __forceinline__ uint32_t load_stream(const uint32_t* p) {
  uint32_t v; asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(v) : "l"(p)); return v;
}
__device__ __forceinline__ uint2 load_stream(const uint2* p) {
  uint2 v; asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p)); return v;
}
__device__ __forceinline__ uint4 load_stream(const uint4* p) {
  uint4 v; asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p)); return v;
}
__device__ __forceinline__ uint16_t load_stream(const uint16_t* p) { return __ldg(p); }
__device__ __forceinline__ uint8_t load_stream(const uint8_t* p) { return __ldg(p); }

template <typename V>
struct GatherTuning {
  static constexpr int kU = sizeof(V) >= 16 ? 4 : 8;  // independent loads in flight per warp
};

template <typename V>
__global__ void __launch_bounds__(kRelabelThreads, kGatherMinBlocks) gather_rows_kernel(const __grid_constant__ GatherParams p) {
  constexpr int kU = GatherTuning<V>::kU;
  const int lane = threadIdx.x & 31;
  const int64_t warp_global = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps_global = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int64_t n_warp_tiles = (p.row_end + 31) >> 5;

#pragma unroll 1
  for (int64_t wt = (p.row_begin >> 5) + warp_global; wt < n_warp_tiles; wt += n_warps_global) {
    const int64_t g0 = wt << 5;
    const int n = (int)(p.row_end - g0 < 32 ? p.row_end - g0 : 32);
    // lane l holds the source row of batch row g0 + l; the vector of the next job is fetched one job ahead
    int32_t next_row = lane < n ? __ldg(p.vec_rows + (int64_t)p.jobs[0].slot * p.total_rows + g0 + lane) : 0;
#pragma unroll 1
    for (int j = 0; j < p.n_jobs; ++j) {
      const RowJob& job = p.jobs[j];
      const int32_t my_row = next_row;
      if (j + 1 < p.n_jobs) next_row = lane < n ? __ldg(p.vec_rows + (int64_t)p.jobs[j + 1].slot * p.total_rows + g0 + lane) : 0;
      const uint8_t* __restrict__ src = job.src;
      uint8_t* __restrict__ dst = job.dst + (size_t)g0 * job.row_bytes;
      const uint32_t stride = job.src_stride, row_bytes = job.row_bytes;
      const int epr = job.epr;
      if (job.n_coliter == 1) {
        const int lpr_log2 = job.lpr_log2;
        const int sub = lane >> lpr_log2;                       // row within the pass
        const int col = lane & ((1 << lpr_log2) - 1);
        const int rpp_log2 = 5 - lpr_log2;
        const int n_pass = (n + (1 << rpp_log2) - 1) >> rpp_log2;
        const bool col_ok = col < epr;
        // lanes beyond the row (col >= epr) and rows beyond the tile re-read a valid element instead of being
        // predicated off: no extra sectors are touched and every val[] register is unconditionally defined
        const uint32_t src_off = (uint32_t)(col_ok ? col : epr - 1) * (uint32_t)sizeof(V);
        const uint32_t dst_off = (uint32_t)sub * row_bytes + (uint32_t)col * (uint32_t)sizeof(V);
        const uint32_t pass_bytes = row_bytes << rpp_log2;
#pragma unroll 1
        for (int pass0 = 0; pass0 < n_pass; pass0 += kU) {
          V val[kU];
#pragma unroll
          for (int u = 0; u < kU; ++u) {
            const int row = min(((pass0 + u) << rpp_log2) + sub, n - 1);
            const uint32_t src_row = (uint32_t)__shfl_sync(0xffffffffu, my_row, row);
            val[u] = load_stream(reinterpret_cast<const V*>(src + (size_t)src_row * stride + src_off));
          }
#pragma unroll
          for (int u = 0; u < kU; ++u) {
            const int row = ((pass0 + u) << rpp_log2) + sub;
            if (col_ok && row < n) *reinterpret_cast<V*>(dst + (uint32_t)(pass0 + u) * pass_bytes + dst_off) = val[u];
          }
        }
      } else {
        // long rows: 2 rows x up to 4 column slices per sweep
        constexpr int kRowsPerSweep = 2, kSlices = (kU > 8 ? 8 : kU) / kRowsPerSweep;
        const int n_coliter = job.n_coliter;
#pragma unroll 1
        for (int row0 = 0; row0 < n; row0 += kRowsPerSweep) {
          const uint8_t* sp[kRowsPerSweep];
#pragma unroll
          for (int rr = 0; rr < kRowsPerSweep; ++rr)
            sp[rr] = src + (size_t)(uint32_t)__shfl_sync(0xffffffffu, my_row, min(row0 + rr, n - 1)) * stride;
#pragma unroll 1
          for (int c0 = 0; c0 < n_coliter; c0 += kSlices) {
            V val[kRowsPerSweep][kSlices];
#pragma unroll
            for (int rr = 0; rr < kRowsPerSweep; ++rr)
#pragma unroll
              for (int c = 0; c < kSlices; ++c) {
                const int col = min(((c0 + c) << 5) + lane, epr - 1);
                val[rr][c] = load_stream(reinterpret_cast<const V*>(sp[rr]) + col);
              }
#pragma unroll
            for (int rr = 0; rr < kRowsPerSweep; ++rr)
#pragma unroll
              for (int c = 0; c < kSlices; ++c) {
                const int col = ((c0 + c) << 5) + lane;
                if (row0 + rr < n && col < epr) reinterpret_cast<V*>(dst + (size_t)(row0 + rr) * row_bytes)[col] = val[rr][c];
              }
          }
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// Row gather, asynchronous variant (the default for rows of 17 .. kAsyncMaxStride bytes).
//
// The register-staged kernel above keeps one register per in-flight load, which caps the bytes a warp can have
// in flight.  Here the source rows go HBM -> shared memory with cp.async (LDGSTS, 16 bytes per lane, L1
// bypassed) into a per-warp ring of kAsyncStages stages, so several KB per warp are in flight without holding
// registers, and the drain is shared-memory loads + *flat* coalesced stores: the dense output tile of a job is
// one contiguous span, so lanes store consecutive 16-byte pieces no matter how long a row is.
// Work item = (warp tile of 32 batch rows, job, sub-range of rows that fits one stage).
//
// Both inner loops are written for instruction count (the first version spent 17 integer instructions per memory
// instruction): the (row, chunk) position of a lane advances incrementally in the issue loop, and the drain turns
// a dense word index into a stage offset with one multiply-high per word (row = word / words_per_row).
// ---------------------------------------------------------------------------------------------------------
constexpr int kAsyncStages = 3;
constexpr int kAsyncWarps = 8;
constexpr int kAsyncMaxStride = 4096;

// The work of one 32-row warp tile is a fixed list of pipeline ITEMS -- (load job, sub-range of rows that fits one
// stage) -- and every item feeds one or more dense OUTPUTS (datasets.py:78-83: every field of the dataset is gathered
// at the same rows, so one staged record feeds several keys).  The list is the same for every tile of a launch, so the
// host lays it out once, with everything that can be derived ahead of time already derived, and every CTA keeps a copy
// in shared memory: an item costs the warp three 16-byte shared loads to set up, an output two (the first version
// walked job/output descriptors in the constant bank and re-derived cursors, ring addresses and alignment per item:
// 47 % of the executed instructions of C2's fused launch were that bookkeeping, profiles/r2_c2_sass_before.txt).
struct __align__(16) ItemDesc {
  // ---- words 0-3 ----
  const uint4* src16;     // span base: field base, or record table base + span offset; 16-byte aligned
  uint32_t stride16;      // source row stride in 16-byte units
  uint32_t cpr;           // 16-byte chunks copied per row (the row pitch inside a stage is exactly cpr chunks)
  // ---- words 4-7 ----
  uint32_t cpr_magic;     // ceil(2^32 / cpr), or 0 when cpr == 1: e / cpr == umulhi(e, magic) for e * cpr < 2^32
  uint32_t dr;            // 32 / cpr   } advance of a lane's (row, chunk) position per issue iteration
  uint32_t dch;           // 32 % cpr   }
  uint32_t slot;          // which index vector names the source rows
  // ---- words 8-11 (all the drain needs) ----
  uint32_t sub;           // first row of the item inside the tile
  uint32_t rows;          // rows of the item in a full tile
  uint32_t flags;         // bit 0: first item of its (tile, job) pair; bits 8-15: slot of the NEXT pair; bit 16: that pair
                          // belongs to the next tile (index-vector prefetch of the un-fused kernel)
  uint32_t out_begin_n;   // first output | number of outputs << 16
};
static_assert(sizeof(ItemDesc) == 48, "ItemDesc is read as three 16-byte words");

enum : int { DRAIN_WORDS = 0, DRAIN_DENSE16 = 1, DRAIN_ELEMS = 2, DRAIN_WORDS_UNALIGNED = 3 };

struct __align__(16) OutDesc {
  // ---- words 0-3 ----
  uint8_t* dst;           // key base + sub * row_bytes: output of the item's first row in tile 0
  uint32_t tile_bytes;    // 32 * row_bytes: advance per tile
  uint32_t soff;          // byte offset of the sub-field inside a staged row
  // ---- words 4-7 ----
  uint32_t epr;           // output elements per row: 4-byte words (DRAIN_WORDS*), 1 << vec_log2 bytes (DRAIN_ELEMS), bytes (DENSE16)
  uint32_t epr_magic;     // ceil(2^32 / epr), or 0 when epr == 1
  uint32_t gap;           // stage pitch - row_bytes: bytes between the end of this sub-field in one staged row and its start in the next
  uint32_t kind;          // DRAIN_* | vec_log2 << 8 | stage pitch << 16 (DRAIN_ELEMS only)
};
static_assert(sizeof(OutDesc) == 32, "OutDesc is read as two 16-byte words");

constexpr int kMaxItems = 64;      // per launch; the host splits the job list over several launches beyond that
constexpr int kMaxItemOuts = 192;

struct AsyncGatherParams {
  const int32_t* vec_rows;
  int64_t total_rows;
  int64_t row_begin, row_end;  // row_begin is a multiple of 32
  int32_t n_items;             // items of one tile
  int32_t n_outs;              // outputs of all items
  int32_t stage_bytes;
  int32_t ring_bytes;          // kAsyncStages * stage_bytes
  int32_t ring_offset;         // the per-warp rings start this far into dynamic shared memory (after the tables and the tile FIFOs)
  int32_t claim_item;          // dynamic tile scheduling: the item at whose issue a warp claims its next tile
  uint32_t* sched;             // [0] tile tickets, [1] CTAs finished; nullptr: static round-robin tiles (see below)
  ItemDesc items[kMaxItems];
  OutDesc outs[kMaxItemOuts];
};

__device__ __forceinline__ void cp_async16(uint32_t smem_addr, const void* gptr) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_addr), "l"(gptr) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ uint32_t fast_div(uint32_t e, uint32_t magic) { return magic ? __umulhi(e, magic) : e; }

__device__ __forceinline__ uint32_t lds32(uint32_t addr) {
  uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr)); return v;
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v; asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr)); return v;
}

// Output rows are written once and read by another kernel much later: store them with the streaming (evict-first)
// policy so that they do not push dataset rows out of L2 (+2 % on C3 over plain stores).
// (The converse hint -- loading the rows with an L2 evict-last policy -- was measured as well: no effect on C2/C3/C5.)
__device__ __forceinline__ void store_out(uint4* p, const uint4 v) { __stcs(p, v); }

// generic element drain (rows whose size is not a multiple of 4 bytes): flat element index, coalesced stores
template <typename V>
__device__ __forceinline__ void drain_flat(const uint8_t* __restrict__ sbase, uint8_t* __restrict__ dbase, const uint32_t n_elem,
                                           const uint32_t stride, const uint32_t epr, const uint32_t epr_magic, const int lane) {
  for (uint32_t e = lane; e < n_elem; e += 32) {
    const uint32_t r = fast_div(e, epr_magic), col = e - r * epr;
    reinterpret_cast<V*>(dbase)[e] = *reinterpret_cast<const V*>(sbase + r * stride + col * (uint32_t)sizeof(V));
  }
}

// Word rows (float32 observations, actions ...): output word w of the item lives at stage offset 4*w + gap*(w / epr).
// Each lane assembles 16 consecutive output bytes from four shared words and issues one 16-byte store, so a
// warp-wide store covers 512 contiguous bytes of the dense output.  `dbase` must be 16-byte aligned.
__device__ __forceinline__ void drain_words(const uint32_t sbase, uint8_t* __restrict__ dbase, const uint32_t n_words,
                                            const uint32_t epr_magic, const uint32_t gap, const int lane) {
  const uint32_t n_quads = n_words >> 2;
#pragma unroll 2
  for (uint32_t q = lane; q < n_quads; q += 32) {
    const uint32_t w = q << 2;
    const uint32_t a0 = sbase + 4u * w + gap * fast_div(w, epr_magic);
    const uint32_t a1 = sbase + 4u * w + 4u + gap * fast_div(w + 1u, epr_magic);
    const uint32_t a2 = sbase + 4u * w + 8u + gap * fast_div(w + 2u, epr_magic);
    const uint32_t a3 = sbase + 4u * w + 12u + gap * fast_div(w + 3u, epr_magic);
    const uint32_t v0 = lds32(a0), v1 = lds32(a1), v2 = lds32(a2), v3 = lds32(a3);
    store_out(reinterpret_cast<uint4*>(dbase) + q, make_uint4(v0, v1, v2, v3));
  }
  for (uint32_t w = (n_quads << 2) + lane; w < n_words; w += 32)    // ragged last tile only
    reinterpret_cast<uint32_t*>(dbase)[w] = lds32(sbase + 4u * w + gap * fast_div(w, epr_magic));
}

// same layout, 4-byte stores: used when the item's output span does not start on a 16-byte boundary
__device__ __forceinline__ void drain_words_unaligned(const uint32_t sbase, uint8_t* __restrict__ dbase, const uint32_t n_words,
                                                      const uint32_t epr_magic, const uint32_t gap, const int lane) {
  for (uint32_t w = lane; w < n_words; w += 32)
    reinterpret_cast<uint32_t*>(dbase)[w] = lds32(sbase + 4u * w + gap * fast_div(w, epr_magic));
}

// rows without padding whose size is a multiple of 16: the stage already holds the dense output span
__device__ __forceinline__ void drain_dense16(const uint32_t sbase, uint8_t* __restrict__ dbase, const uint32_t n_bytes, const int lane) {
  const uint32_t n16 = n_bytes >> 4;
#pragma unroll 2
  for (uint32_t i = lane; i < n16; i += 32) store_out(reinterpret_cast<uint4*>(dbase) + i, lds128(sbase + (i << 4)));
}

struct TileCursor {
  int32_t tile; // warp tile (32 batch rows); a launch holds < 2^31 rows, so tiles fit 32 bits comfortably
  int32_t k;    // item of the tile (index into the item table)
  int32_t n;    // rows of this tile (32 except for the ragged last tile)
};

// One body, two kernels.  kFused == false: the source rows come from the index vectors an earlier
// relabel_index_kernel wrote.  kFused == true: the warp computes the index algebra of its 32 batch rows itself
// (relabel_row, one lane per row) when it enters a tile and keeps the rows of every slot in registers -- sample() is
// then a single launch.
// (A TMA variant -- one cp.async.bulk per source row instead of 16-byte LDGSTS chunks -- was measured and dropped:
// equal on 224/288-byte rows, 17 % slower on 128-byte rows.)
__device__ __forceinline__ void sts32(uint32_t addr, int32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); }

// every CTA copies the launch's item / output tables from the constant bank into shared memory once
__device__ __forceinline__ void stage_tables(const AsyncGatherParams& p, uint8_t* smem_dyn) {
  uint4* items_s = reinterpret_cast<uint4*>(smem_dyn);
  const int n_item_vecs = p.n_items * (int)(sizeof(ItemDesc) / 16);
  for (int i = threadIdx.x; i < n_item_vecs; i += blockDim.x) items_s[i] = reinterpret_cast<const uint4*>(p.items)[i];
  uint4* outs_s = items_s + n_item_vecs;
  const int n_out_vecs = p.n_outs * (int)(sizeof(OutDesc) / 16);
  for (int i = threadIdx.x; i < n_out_vecs; i += blockDim.x) outs_s[i] = reinterpret_cast<const uint4*>(p.outs)[i];
}

template <bool kFused, bool kInject, int kFlavour, int kStages = kAsyncStages, int kWarps = kAsyncWarps>
__device__ __forceinline__ void gather_rows_async_body(const AsyncGatherParams& p, const RelabelParams& rp, uint8_t* smem_dyn) {
  constexpr int kSlots = FlavourSlots<kFlavour>::value;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int32_t n_warps_global = (int32_t)gridDim.x * kWarps;
  const int32_t n_tiles = (int32_t)((p.row_end + 31) >> 5);
  const int32_t last_n = (int32_t)(p.row_end - ((int64_t)(n_tiles - 1) << 5));      // rows of the last tile
  const int32_t first_tile = (int32_t)(p.row_begin >> 5) + (int32_t)blockIdx.x * kWarps + warp;
  const int32_t n_items = p.n_items;
  const uint4* items_s = reinterpret_cast<const uint4*>(smem_dyn);
  const uint4* outs_s = items_s + n_items * (int)(sizeof(ItemDesc) / 16);
  const uint32_t ring_u32 = (uint32_t)__cvta_generic_to_shared(smem_dyn) + (uint32_t)p.ring_offset + (uint32_t)warp * (uint32_t)p.ring_bytes;

  // Tile scheduling.  Every warp starts on the tile of its global index; after that it either strides by the number of
  // warps (static) or -- p.sched != nullptr -- takes the next unclaimed tile from a global ticket counter.  The SMs do not
  // run at one speed (a DRAM-bound launch shares HBM unevenly), so with static tiles the slowest SM sets the launch time;
  // with tickets every warp is busy until the tiles run out (profiles/r2_ab_shapes.txt, batches r2i-r2k: C5 0.85 -> 0.91
  // of the HBM peak at equal launch size).  The ticket is asked for at item `claim_item`, which the host places one to
  // three (tile, job) pairs before the item where the head needs the tile, so that the atomic's round trip hides behind
  // those pairs' issue loops.  The tail cursor drains the same tile sequence a few items
  // later: the warp keeps its claimed tiles in a four-entry FIFO in shared memory (the head is at most kStages - 1 tile
  // boundaries ahead of the tail, plus the tile it has resolved but not entered).
  const bool dyn = p.sched != nullptr;
  const int32_t dyn_base = (int32_t)(p.row_begin >> 5) + n_warps_global;            // ticket t names tile dyn_base + t
  const uint32_t fifo_u32 = (uint32_t)__cvta_generic_to_shared(smem_dyn) + (uint32_t)p.ring_offset - 16u * (uint32_t)(kWarps - warp);
  uint32_t ticket = 0;                   // lane 0: the ticket in flight
  int32_t head_next = 0;                 // the tile after the head's, once resolved
  bool head_resolved = false;
  uint32_t head_ord = 0, tail_ord = 0;   // ordinals of the head's and the tail's tile in this warp's sequence
  auto resolve = [&]() {                 // wait for the ticket and publish the tile to the tail
    head_next = dyn_base + (int32_t)__shfl_sync(0xffffffffu, ticket, 0);
    head_resolved = true;
    if (lane == 0) sts32(fifo_u32 + (((head_ord + 1u) & 3u) << 2), head_next);
  };
  auto advance_head = [&](TileCursor& c) {
    if (++c.k == n_items) {
      c.k = 0;
      if (dyn) {
        if (!head_resolved) resolve();
        c.tile = head_next;
        head_resolved = false;
        ++head_ord;
      } else {
        c.tile += n_warps_global;
      }
      c.n = c.tile == n_tiles - 1 ? last_n : 32;
    }
  };
  auto advance_tail = [&](TileCursor& c) {
    if (++c.k == n_items) {
      c.k = 0;
      if (dyn) c.tile = (int32_t)lds32(fifo_u32 + (((++tail_ord) & 3u) << 2));   // written before an earlier __syncwarp of the loop
      else c.tile += n_warps_global;
      c.n = c.tile == n_tiles - 1 ? last_n : 32;
    }
  };
  // lane l keeps the source row of batch row (tile*32 + l) for the (tile, job) pair being issued
  int32_t sr[kMaxSlots];                 // fused: rows of every slot for the tile being issued
#pragma unroll
  for (int v = 0; v < kMaxSlots; ++v) sr[v] = 0;
  int32_t issue_rows = 0;
  // un-fused: the vector of the pair after the current one is fetched one pair ahead, so its latency hides behind a job
  auto load_rows = [&](int32_t tile, uint32_t slot) -> int32_t {
    if (tile >= n_tiles) return 0;
    const int n = tile == n_tiles - 1 ? last_n : 32;
    return __ldg(p.vec_rows + (int64_t)slot * p.total_rows + ((int64_t)tile << 5) + min(lane, n - 1));
  };
  int32_t pref_rows = 0;
  if (!kFused) pref_rows = load_rows(first_tile, items_s[1].w);
  auto issue = [&](const TileCursor& c, const uint32_t stage_u32) {
    if (c.tile < n_tiles) {
      const uint4* it = items_s + c.k * (int)(sizeof(ItemDesc) / 16);
      const uint4 d0 = it[0], d1 = it[1], d2 = it[2];
      if (dyn && c.k == p.claim_item && lane == 0) ticket = atomicAdd(p.sched, 1u);
      if (d2.z & 1u) {                                           // entering the next (tile, job) pair
        if (kFused) {
          if (c.k == 0 && lane < c.n) relabel_row<kInject, kFlavour>(rp, SegView{rp.seg_bucket, rp.seg_table}, ((int64_t)c.tile << 5) + lane, sr);
          issue_rows = pick_slot<kSlots>(sr, (int)d1.w);
        } else {
          issue_rows = pref_rows;
          int32_t pref_tile = c.tile;
          if (d2.z & 0x10000u) {                                 // the pair after this one opens the warp's next tile
            if (dyn) { resolve(); pref_tile = head_next; }
            else pref_tile = c.tile + n_warps_global;
          }
          pref_rows = load_rows(pref_tile, (d2.z >> 8) & 0xffu);
        }
      }
      const uint32_t cpr = d0.w, stride16 = d0.z, dr = d1.y, dch = d1.z;
      const int rows = min((int)d2.y, c.n - (int)d2.x);          // <= 0: the ragged last tile ends before this item
      const int n_chunks = rows * (int)cpr;
      // lane -> (row r, chunk ch) of the item; both advance incrementally, no division inside the loop.  Chunk e of an
      // item lands at stage offset 16 * e (the stage pitch is exactly cpr chunks).  Source addresses are formed in
      // 16-byte units (32-bit), so a field must stay below 64 GB (host-checked).
      uint32_t r = fast_div((uint32_t)lane, d1.x);
      uint32_t ch = (uint32_t)lane - r * cpr;
      r += d2.x;
      uint32_t soff = stage_u32 + ((uint32_t)lane << 4);
      const uint4* __restrict__ src16 = reinterpret_cast<const uint4*>(((uint64_t)d0.y << 32) | (uint64_t)d0.x);
      if (dch == 0) {                                            // chunks per row divide 32: a lane stays on its chunk column
#pragma unroll 2
        for (int e = lane; e - lane < n_chunks; e += 32) {
          const uint32_t src_row = (uint32_t)__shfl_sync(0xffffffffu, issue_rows, (int)r);
          if (e < n_chunks) cp_async16(soff, src16 + (src_row * stride16 + ch));
          r += dr; soff += 512u;
        }
      } else {
#pragma unroll 2
        for (int e = lane; e - lane < n_chunks; e += 32) {
          const uint32_t src_row = (uint32_t)__shfl_sync(0xffffffffu, issue_rows, (int)r);
          if (e < n_chunks) cp_async16(soff, src16 + (src_row * stride16 + ch));
          r += dr; ch += dch; soff += 512u;
          if (ch >= cpr) { ch -= cpr; ++r; }
        }
      }
    }
    cp_async_commit();
  };

  auto drain = [&](const TileCursor& c, const uint32_t sbase) {
    const uint4 d2 = items_s[c.k * (int)(sizeof(ItemDesc) / 16) + 2];
    const int rows = min((int)d2.y, c.n - (int)d2.x);
    if (rows <= 0) return;
    const uint4* od = outs_s + (d2.w & 0xffffu) * (uint32_t)(sizeof(OutDesc) / 16);
#pragma unroll 1
    for (uint32_t o = d2.w >> 16; o != 0; --o, od += sizeof(OutDesc) / 16) {
      const uint4 o0 = od[0], o1 = od[1];
      uint8_t* dbase = reinterpret_cast<uint8_t*>(((uint64_t)o0.y << 32) | (uint64_t)o0.x) + (uint64_t)(uint32_t)c.tile * o0.z;
      const uint32_t s0 = sbase + o0.w;
      const uint32_t kind = o1.w & 0xffu;
      if (kind == DRAIN_WORDS) {
        drain_words(s0, dbase, (uint32_t)rows * o1.x, o1.y, o1.z, lane);
      } else if (kind == DRAIN_DENSE16) {
        drain_dense16(s0, dbase, (uint32_t)rows * o1.x, lane);
      } else if (kind == DRAIN_WORDS_UNALIGNED) {
        drain_words_unaligned(s0, dbase, (uint32_t)rows * o1.x, o1.y, o1.z, lane);
      } else {
        const uint8_t* sgen = smem_dyn + (size_t)(s0 - (uint32_t)__cvta_generic_to_shared(smem_dyn));
        const uint32_t n_elem = (uint32_t)rows * o1.x, pitch = o1.w >> 16;
        if (((o1.w >> 8) & 0xffu) == 1u) drain_flat<uint16_t>(sgen, dbase, n_elem, pitch, o1.x, o1.y, lane);
        else drain_flat<uint8_t>(sgen, dbase, n_elem, pitch, o1.x, o1.y, lane);
      }
    }
  };

  TileCursor head{first_tile, 0, first_tile == n_tiles - 1 ? last_n : 32};  // next item to issue
  TileCursor tail = head;                                                    // next item to drain
  const uint32_t stage_bytes = (uint32_t)p.stage_bytes, ring_bytes = (uint32_t)p.ring_bytes;
  uint32_t head_off = 0, tail_off = 0;                                       // stage offsets inside this warp's ring
#pragma unroll 1
  for (int t = 0; tail.tile < n_tiles; ++t) {
    issue(head, ring_u32 + head_off);    // one cp.async group per iteration (empty once the head has run off the end)
    if (head.tile < n_tiles) advance_head(head);
    head_off += stage_bytes;
    if (head_off == ring_bytes) head_off = 0;
    if (t >= kStages - 1) {
      cp_async_wait<kStages - 1>();        // everything but the newest kStages-1 groups has landed
      __syncwarp();                        // ... for every lane of this warp
      drain(tail, ring_u32 + tail_off);
      __syncwarp();                        // the stage may be overwritten by the next issue
      advance_tail(tail);
      tail_off += stage_bytes;
      if (tail_off == ring_bytes) tail_off = 0;
    }
  }
}

// Dynamic tile scheduling leaves its two counters at zero for the next launch that is handed the same pair: the last
// CTA to finish clears them (every ticket has been consumed by then -- a warp uses the value of its last ticket before
// it leaves the loop).
__device__ __forceinline__ void sched_release(uint32_t* sched) {
  if (sched == nullptr) return;
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(sched + 1, 1u) == gridDim.x - 1) {
      sched[0] = 0;
      sched[1] = 0;
    }
  }
}

// resident CTAs per SM a (stages, warps) shape is compiled for: the register cap follows from it
constexpr int gather_min_blocks(int warps) { return warps <= 8 ? 2 : 1; }

template <int kStages = kAsyncStages, int kWarps = kAsyncWarps>
__global__ void __launch_bounds__(kWarps * 32, gather_min_blocks(kWarps)) gather_rows_async_kernel(const __grid_constant__ AsyncGatherParams p) {
  extern __shared__ __align__(128) uint8_t smem_dyn[];
  stage_tables(p, smem_dyn);
  __syncthreads();
  gather_rows_async_body<false, false, FLAVOUR_PLAIN, kStages, kWarps>(p, *reinterpret_cast<const RelabelParams*>(&p), smem_dyn);
  sched_release(p.sched);
}

struct FusedParams {
  RelabelParams relabel;
  AsyncGatherParams gather;
};

// sample() in one launch: index algebra + row gathers (datasets.py:213-294 / :496-643 for vector observations)
template <bool kInject, int kFlavour, int kStages = kAsyncStages, int kWarps = kAsyncWarps>
__global__ void __launch_bounds__(kWarps * 32, gather_min_blocks(kWarps)) relabel_gather_kernel(const __grid_constant__ FusedParams p) {
  extern __shared__ __align__(128) uint8_t smem_dyn[];
  stage_tables(p.gather, smem_dyn);
  __syncthreads();
  gather_rows_async_body<true, kInject, kFlavour, kStages, kWarps>(p.gather, p.relabel, smem_dyn);
  sched_release(p.gather.sched);
}

}  // namespace ogb
