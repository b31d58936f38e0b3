"""The index algebra (`relabel_row`: draws -> rows, goals, masks) at every valid-row table form, bucket width and index-kernel
instance, position by position.

`Tables` restates the table selection of ogb_sampler.cu (`build_valid_tables`, `shift_for`, `build_buckets`,
`build_segment_table`) and `route` the choice of the index instance (`fuse`, `use_aux`, the shared-memory condition of
`index_launch`, `is_point_record`, `choose_index_kernel`).  `test_catalogue_reaches_every_form_and_instance` (no GPU) shows
that the catalogue below reaches each form, the bucket widths, both sides of every threshold and every instance the
routing can produce; `UNREACHABLE` lists the others with the reason.

On the device, every catalogue dataset reports its form through `ogb_sampler_table_info`, and validation draws with
`idx_pos = arange(n_choices)` read every table entry in one batch, for each goal kind, against the oracle and against
closed forms computed here (valid_idxs[pos], the first terminal at or after a row, the trajectory's first row).  Each
index instance then runs in both draw modes with its kernel list asserted (`ogb_batch_kernel_names`), and two large
datasets take the gap-rank search past the 2^17-bucket cap and past the 2^22-bucket limit of the segment table.

Observations hold the row number (int32 bit patterns in float32 rows), so every gathered row names its source row.
"""

import ctypes as C
import itertools
import os
import tempfile

import numpy as np
import pytest

from oracle.replay_oracle import Draws, DrawsSource, GoalDraws, OracleATCSampler, OracleSampler, pick_goals, shifted_edge_crop, stacked_frames, subgoal_step
from tests.golden.make_golden import cfg
from tests.test_gpu_rows import RowPlan

# ------------------------------------------------ the table selection, restated ------------------------------------------------
BUCKET_CAP = 1 << 17          # shift_for: at most 2^17 buckets
SEG_MIN_GAP = 16              # build_segment_table (a): boundaries at least 16 positions apart
SEG_MAX_BUCKETS = 1 << 22     # ... and (n_valid >> shift) <= 2^22
SMEM_TABLE_BYTES = 48 * 1024  # index_launch: segment table in shared memory up to 48 KB ...
SMEM_MIN_ROWS = 65536         # ... for launches of at least 65,536 rows on the auxiliary stream
OVERLAP_MIN_ROWS = 32768      # kOverlapMinRows
GC, HGC, PLAIN = 0, 1, 2      # FLAVOUR_*


def shift_for(key_range, table_len):
    shift = 4
    mean_gap = max(1, key_range // table_len) if table_len > 0 else key_range
    while (1 << (shift + 1)) < mean_gap // 2:
        shift += 1
    while (key_range >> shift) > BUCKET_CAP:
        shift += 1
    return shift


def build_buckets(table, max_key, shift):
    return np.searchsorted(table, np.arange((max_key >> shift) + 2, dtype=np.int64) << shift, side='left')


class Tables:
    """What ogb_dataset_create and ogb_sampler_create build for these flags.  `mode` is valid_mode as sample() uses it
    (3: the segment table); `why` records the threshold that decided it."""

    def __init__(self, terminals, valids=None, trl=False):
        size = len(terminals)
        self.term = np.nonzero(terminals > 0)[0]
        self.term_shift = shift_for(size, len(self.term))
        self.seg_shift, self.n_seg_table, self.gap_shift, self.why = -1, 0, 0, set()
        if valids is None:
            self.mode, self.n_valid = 0, -1
        else:
            ok = valids > 0
            self.valid_idxs = np.nonzero(ok)[0]
            self.n_valid = len(self.valid_idxs)
            gap_rows = np.nonzero(~ok)[0]
            self.gaps = gap_rows - np.arange(len(gap_rows))
            if len(self.gaps) * 8 <= size:
                self.why.add('gaps*8<=size')
                self.mode = 2
                self.gap_shift = shift_for(self.n_valid + 1, len(self.gaps))
                self.why.add('gap_shift capped' if shift_for(self.n_valid + 1, len(self.gaps)) !=
                             _mean_gap_shift(self.n_valid + 1, len(self.gaps)) else 'gap_shift from mean gap')
                self._segment_table(size)
            else:
                self.why.add('gaps*8>size')
                self.mode = 1
        self.n_choices = (size - len(self.term)) if trl else (size if self.mode == 0 else self.n_valid)
        if trl:
            self.mode = 1

    def _segment_table(self, size):
        c = self.gaps
        if len(c) == 0:
            self.why.add('no gaps')
            return
        min_gap = int(np.min(np.diff(c))) if len(c) > 1 else self.n_valid
        if min_gap < SEG_MIN_GAP:
            self.why.add('min_gap<16')
            return
        self.why.add('min_gap>=16')
        shift = 4
        while (1 << (shift + 1)) <= min_gap:
            shift += 1
        if (self.n_valid >> shift) > SEG_MAX_BUCKETS:
            self.why.add('n_valid>>shift>2^22')
            return
        self.why.add('n_valid>>shift<=2^22')
        m = np.arange(len(c) + 1)
        first = np.where(m == 0, 0, np.concatenate([[0], c + np.arange(len(c)) + 1]))
        last = np.concatenate([c + np.arange(len(c)) - 1, [size - 1]])
        used = first <= last
        fin = self.term[np.minimum(np.searchsorted(self.term, first[used]), len(self.term) - 1)]
        if np.any(fin < last[used]) or np.any(self.term[-1] < last[used]):
            self.why.add('terminal inside a segment')
            return
        self.why.add('no terminal inside a segment')
        self.mode, self.seg_shift = 3, shift
        self.n_seg_table = len(build_buckets(c, self.n_valid + 1, shift))
        self.why.add('table<=48KB' if self.n_seg_table * 16 <= SMEM_TABLE_BYTES else 'table>48KB')


def _mean_gap_shift(key_range, table_len):
    shift = 4
    mean_gap = max(1, key_range // table_len) if table_len > 0 else key_range
    while (1 << (shift + 1)) < mean_gap // 2:
        shift += 1
    return shift


def index_name(inject, flavour, smem, point):
    """choose_index_kernel"""
    if point and not inject:
        return f'relabel_index_kernel<0, 0, {int(smem)}, 1, 5>'
    if point and not smem:
        return 'relabel_index_kernel<1, 0, 0, 1, 4>'
    return f'relabel_index_kernel<{int(inject)}, {flavour}, {int(smem)}, 0, 4>'


ALL_INDEX = {index_name(i, f, s, False) for i, f, s in itertools.product((0, 1), (GC, HGC, PLAIN), (0, 1))} | {
    index_name(0, GC, 0, True), index_name(0, GC, 1, True), index_name(1, GC, 0, True)}
UNREACHABLE = {
    # shared memory needs the auxiliary stream, which needs a gather after the index kernel (use_aux: any_frames or a row
    # over 16 bytes); the point-maze record needs no gather after it (is_point_record: !any_gather)
    'relabel_index_kernel<0, 0, 1, 1, 5>': 'the point-maze kernel runs with no gather after it, the auxiliary stream only with one',
}
# (GCDataset.augment() and ATCDataset.augment() crop through a PLAIN sampler over a temporary dataset of the batch's images,
# which has no 'valids' and so no segment table: at any size they take <1, 2, 0, 0, 4>.  The PLAIN shared-memory instances
# are reached by get_observations and ogb_sampler_gather_cropped on a sampler whose dataset has one.)
FUSED_UNREACHABLE = {
    'relabel_gather_kernel<0, 0, 3, 8>': 'split_span_jobs gives the fused GCDataset launch with Philox draws the 2 x 20 or 2 x 16 shape',
}


def route(kind, total, inject, any_frames, spans, lsu, mode, n_seg_table, point_layout, trl=False, debug=False):
    """run_sample + index_launch: the index instance, or None when a fused launch does the index algebra."""
    flavour = {'gc': GC, 'hgc': HGC, 'plain': PLAIN}[kind]
    any_long = spans or lsu
    fuse = spans and not any_frames and (total < OVERLAP_MIN_ROWS or kind != 'hgc')
    use_aux = not fuse and (any_frames or any_long) and (total >= OVERLAP_MIN_ROWS or any_frames)
    if fuse:
        return None
    any_gather = spans or lsu or any_frames
    point = point_layout and kind == 'gc' and not trl and not any_gather and not debug and mode == 3
    smem = use_aux and mode == 3 and 0 < n_seg_table * 16 <= SMEM_TABLE_BYTES and total >= SMEM_MIN_ROWS
    return index_name(inject, flavour, smem, point)


# ------------------------------------------------ the catalogue ------------------------------------------------
def from_invalid(size, invalid, extra_terminals=()):
    """Compact layout (ogbench's compact datasets): valids 0 at `invalid`, terminals at every invalid row, the valid row
    before it, and the last row (so that terminal_locs[-1] == size - 1)."""
    valids = np.ones(size, np.float32)
    terminals = np.zeros(size, np.float32)
    invalid = np.asarray(invalid, np.int64)
    valids[invalid] = 0
    terminals[invalid] = 1
    terminals[invalid[invalid > 0] - 1] = 1
    terminals[size - 1] = 1
    terminals[list(extra_terminals)] = 1
    return dict(terminals=terminals, valids=valids)


def from_lengths(lengths):
    """Trajectories of `lengths` rows, each ending in an invalid row (the compact layout of tests/golden/make_golden.py)."""
    ends = np.cumsum(lengths) - 1
    return from_invalid(int(ends[-1]) + 1, ends)


def regular(lengths):
    ends = np.cumsum(lengths) - 1
    terminals = np.zeros(int(ends[-1]) + 1, np.float32)
    terminals[ends] = 1
    return dict(terminals=terminals)


def with_rows(layout, obs_dim=1, act_dim=0, image=None):
    """Observations whose first int32 word is the row number (the rest: row * 8 + column), optional actions likewise."""
    n = len(layout['terminals'])
    r = np.arange(n, dtype=np.int32)[:, None]
    fields = dict(layout)
    if image is not None:
        fields['observations'] = (np.arange(n * int(np.prod(image)), dtype=np.int64).reshape(n, *image) * 7 % 251).astype(np.uint8)
    else:
        fields['observations'] = np.concatenate([r, r * 8 + np.arange(1, obs_dim, dtype=np.int32)], 1).view(np.float32)
    if act_dim:
        fields['actions'] = (r * 8 + np.arange(act_dim, dtype=np.int32) + 100).view(np.float32)
    if 'valids' not in layout:
        fields['next_observations'] = fields['observations'][np.minimum(np.arange(n) + 1, n - 1)].copy()
    return fields


def spaced(n_traj, valid_rows):
    """`n_traj` trajectories of `valid_rows` valid rows each (one invalid row closes each)."""
    return from_lengths(np.full(n_traj, valid_rows + 1))


def smem_layout(n_valid):
    """min gap 16 (shift 4) and ((n_valid + 1) >> 4) + 2 segment-table entries: trajectories of 16 valid rows and a last one
    of 16..31."""
    last = 16 + (n_valid - 16) % 16
    if last < 16:
        last += 16
    n16 = (n_valid - last) // 16
    assert n16 * 16 + last == n_valid
    return from_lengths(np.concatenate([np.full(n16, 17), [last + 1]]))


def _two_close(apart):
    """Invalid rows every 20 rows, except two whose gap ranks c = 32 and 32 + apart (one 16-position bucket when apart = 15)."""
    inv = [32, 33 + apart] + list(range(33 + apart + 20, 1000, 20))
    return from_invalid(1000, inv)


def _single_row_trajectories():
    lengths = np.random.default_rng(4).integers(20, 40, 40)
    lengths[::5] = 1                                  # a 1-row trajectory is its own invalid row: consecutive gaps
    return from_lengths(lengths)


def _view_fields():
    return with_rows(from_lengths(np.random.default_rng(5).integers(17, 40, 60)), 1)


CATALOGUE = {
    # name: (layout, expected valid_mode, expected seg_shift)
    'regular': (regular(np.random.default_rng(0).integers(1, 30, 80)), 0, -1),
    'regular_single_rows': (regular(np.concatenate([np.ones(20, int), np.random.default_rng(1).integers(2, 9, 40)])), 0, -1),
    'compact_short': (from_lengths(np.random.default_rng(2).integers(3, 8, 100)), 1, -1),
    'gaps_x8_eq_size': (from_lengths(np.full(60, 8)), 2, -1),
    'gaps_x8_eq_size_plus_one': (from_invalid(480, list(np.arange(60) * 8 + 7) + [100]), 1, -1),
    'all_valid': (dict(terminals=regular([30, 50, 20])['terminals'], valids=np.ones(100, np.float32)), 2, -1),
    'two_invalid_15_apart': (_two_close(15), 2, -1),
    'two_invalid_16_apart': (_two_close(16), 3, 4),
    'terminal_inside_segment': (from_invalid(600, np.arange(0, 600, 40)[1:], extra_terminals=[100]), 2, -1),
    'first_row_invalid': (from_invalid(500, [0] + list(range(40, 500, 40))), 3, 5),
    'last_row_valid': (from_invalid(500, list(range(40, 480, 40))), 3, 5),
    'last_row_invalid': (from_invalid(500, list(range(40, 500, 40)) + [499]), 3, 4),
    'single_invalid': (from_invalid(700, [300]), 3, 9),
    'single_row_trajectories': (_single_row_trajectories(), 2, -1),
}
for _k in (4, 5, 6, 7, 9):   # 2^k - 1, 2^k and 2^k + 1 valid rows per trajectory: each side of a bucket width
    for _d in (-1, 0, 1):
        _v = (1 << _k) + _d
        CATALOGUE[f'traj_2^{_k}{_d:+d}'] = (spaced(max(8, 3000 // _v), _v), 2 if _v < 16 else 3, -1 if _v < 16 else _k - (_d < 0))
CATALOGUE['smem_3072'] = (smem_layout(49119), 3, 4)     # ((n_valid + 1) >> 4) + 2 == 3072 entries: 48 KB
CATALOGUE['smem_3073'] = (smem_layout(49135), 3, 4)     # 3073 entries: 48 KB + 16 B
EXHAUSTIVE = [k for k in CATALOGUE if not k.startswith('smem')]


def catalogue_tables(name, trl=False):
    layout = CATALOGUE[name][0]
    return Tables(layout['terminals'], layout.get('valids'), trl)


# ------------------------------------------------ the instance cases ------------------------------------------------
# name: (catalogue layout, kind, obs_dim, act_dim, config overrides, call, rows); call 'sample' (GC/HGC sample()), 'plain'
# (Dataset.sample), 'gather' (get_observations), 'cropped' (ogb_sampler_gather_cropped).  Every case runs with Philox draws
# (inject 0) and with validation draws (inject 1), except 'gather' (no draws) and 'cropped' (always injected shifts).
INSTANCES = {
    'point_maze': ('traj_2^5+0', 'gc', 2, 2, {}, 'sample', 4096),
    'gc_tiny_rows': ('single_row_trajectories', 'gc', 1, 0, {}, 'sample', 2048),
    'hgc_tiny_rows': ('traj_2^6+0', 'hgc', 1, 0, dict(subgoal_steps=5), 'sample', 2048),
    'gc_frames_big': ('smem_3072', 'gc', 1, 0, dict(frame_stack=3), 'sample', SMEM_MIN_ROWS),
    'gc_frames_small': ('smem_3072', 'gc', 1, 0, dict(frame_stack=3), 'sample', 4096),
    'hgc_long_big': ('smem_3072', 'hgc', 6, 0, dict(subgoal_steps=5), 'sample', SMEM_MIN_ROWS),
    'hgc_long_big_48k+16': ('smem_3073', 'hgc', 6, 0, dict(subgoal_steps=5), 'sample', SMEM_MIN_ROWS),
    'hgc_long_small': ('traj_2^5+0', 'hgc', 6, 0, dict(subgoal_steps=5), 'sample', 4096),
    'gc_long': ('traj_2^5+0', 'gc', 6, 0, {}, 'sample', 4096),
    'gc_very_long': ('traj_2^4+0', 'gc', 350, 0, {}, 'sample', 512),
    'plain_tiny': ('regular', 'plain', 1, 0, {}, 'plain', 2048),
    'plain_long': ('regular', 'plain', 6, 0, {}, 'plain', 2048),
    'gather_frames_big': ('smem_3072', 'gc', 1, 0, dict(frame_stack=3), 'gather', SMEM_MIN_ROWS),
    'cropped_images_big': ('smem_3072', 'gc', (8, 8, 3), 0, {}, 'cropped', SMEM_MIN_ROWS),
    'cropped_images_small': ('smem_3072', 'gc', (8, 8, 3), 0, {}, 'cropped', 1000),
    'cropped_vectors': ('smem_3072', 'gc', 6, 0, {}, 'cropped', 1000),
}


def instance_fields(case):
    layout, kind, obs, act = INSTANCES[case][:4]
    lay = CATALOGUE[layout][0]
    if isinstance(obs, tuple):
        return with_rows(lay, image=obs)
    return with_rows(lay, obs, act)


def instance_config(case):
    kind, over = INSTANCES[case][1], INSTANCES[case][4]
    return cfg(**over) if kind != 'plain' else None


def expected_kernels(case, inject):
    """The kernel list of one call: the index instance (unless a fused launch does its work), then the gathers."""
    layout, kind, obs, act, over, call, rows = INSTANCES[case]
    fields = instance_fields(case)
    tables = catalogue_tables(layout)
    point_layout = obs == 2 and act == 2 and 'valids' in fields
    if call == 'gather':                 # get_observations of a frame-stacked sampler: one frame key
        return [route('plain', rows, False, True, False, False, tables.mode, tables.n_seg_table, False), 'gather_frames_generic_kernel']
    if call == 'cropped':
        if isinstance(obs, tuple):       # 8x8 images: not a TMA shape (W % 16), the generic frame kernel
            return [route('plain', rows, True, True, False, False, tables.mode, tables.n_seg_table, False), 'gather_frames_generic_kernel']
        return [f'relabel_gather_kernel<1, {PLAIN}, 3, 8>']      # one row span, fused (the crop applies to images only)
    fs = over.get('frame_stack')
    if fs:                               # observations, next_observations, value_goals, actor_goals: one generic launch each
        assert kind == 'gc' and obs == 1
        return [route(kind, rows, inject, True, False, False, tables.mode, tables.n_seg_table, False)] + ['gather_frames_generic_kernel'] * 4
    plan = RowPlan(fields, 'plain' if kind == 'plain' else kind, instance_config(case) or {}, rows, philox=not inject)
    flavour = {'gc': GC, 'hgc': HGC, 'plain': PLAIN}[kind]
    index = route(kind, rows, inject, False, bool(plan.spans), bool(plan.lsu), tables.mode, tables.n_seg_table, point_layout)
    assert (index is None) == plan.fused
    out = [] if plan.fused else [index]
    for i, la in enumerate(plan.launches):
        stages, warps = la['shape'] // 100, la['shape'] % 100
        if i == 0 and plan.fused:
            out.append(f'relabel_gather_kernel<{int(inject)}, {flavour}, {stages}, {warps}>')
        else:
            out.append(f'gather_rows_async_kernel<{stages}, {warps}>')
    return out + ['gather_rows_kernel'] * len(plan.lsu)


def instance_modes(case):
    call = INSTANCES[case][5]
    return {'gather': [False], 'cropped': [True], 'plain': [False]}.get(call, [False, True])


# ------------------------------------------------ no GPU: the catalogue reaches everything ------------------------------------------------
def test_restated_tables_match_closed_forms():
    """The restatement itself: the gap ranks and buckets give valid_idxs at every position of random layouts."""
    rng = np.random.default_rng(0)
    for _ in range(200):
        size = int(rng.integers(1, 400))
        valids = (rng.random(size) > rng.random() * 0.3).astype(np.float32)
        if not valids.any():
            continue
        t = Tables(np.ones(size, np.float32), valids)
        if t.mode != 2 or len(t.gaps) == 0:
            continue
        pos = np.arange(t.n_valid)
        bucket = build_buckets(t.gaps, t.n_valid + 1, t.gap_shift)
        lo = bucket[pos >> t.gap_shift]
        m = lo + np.array([np.searchsorted(t.gaps[l:], p, side='right') for l, p in zip(lo, pos)])
        assert np.array_equal(pos + m, t.valid_idxs)


def test_catalogue_reaches_every_form_and_instance():
    modes, shifts, why = set(), set(), set()
    for name, (layout, mode, seg_shift) in CATALOGUE.items():
        t = Tables(layout['terminals'], layout.get('valids'))
        assert (t.mode, t.seg_shift) == (mode, seg_shift), name
        modes.add(t.mode)
        shifts.add(t.seg_shift)
        why |= t.why
        if name.startswith('smem'):
            assert t.n_seg_table == {'smem_3072': 3072, 'smem_3073': 3073}[name], name
    # the two large cases of test_large_gap_rank_tables
    for n, spec in LARGE.items():
        t = large_tables(spec)
        assert t.mode == 2 and t.seg_shift == -1, n
        why |= t.why
    assert modes == {0, 1, 2, 3}
    assert {4, 5, 6}.issubset(shifts) and max(shifts) > 8
    assert why >= {'gaps*8<=size', 'gaps*8>size', 'min_gap<16', 'min_gap>=16', 'n_valid>>shift>2^22', 'n_valid>>shift<=2^22',
                   'terminal inside a segment', 'no terminal inside a segment', 'table<=48KB', 'table>48KB', 'gap_shift capped',
                   'gap_shift from mean gap', 'no gaps'}, why
    reached = set()
    for case in INSTANCES:
        for inject in instance_modes(case):
            reached |= {k for k in expected_kernels(case, inject) if k.startswith('relabel_')}
    index_reached = {k for k in reached if k.startswith('relabel_index')}
    assert index_reached == ALL_INDEX - set(UNREACHABLE), sorted(ALL_INDEX - set(UNREACHABLE) - index_reached)
    fused = {f'relabel_gather_kernel<{i}, {f}, 3, 8>' for i in (0, 1) for f in (GC, HGC, PLAIN)} | {
        'relabel_gather_kernel<0, 0, 2, 20>', 'relabel_gather_kernel<0, 0, 2, 16>'}
    assert {k for k in reached if k.startswith('relabel_gather')} == fused - set(FUSED_UNREACHABLE)


def test_unreachable_instances_follow_from_the_routing():
    """Every combination of the routing's inputs: the instances it never produces are exactly UNREACHABLE."""
    produced = set()
    for kind, total, inject, frames, spans, lsu, mode, n_seg, point, trl, debug in itertools.product(
            ('gc', 'hgc', 'plain'), (100, OVERLAP_MIN_ROWS, SMEM_MIN_ROWS), (False, True), (False, True), (False, True),
            (False, True), (0, 1, 2, 3), (100, 5000), (False, True), (False, True), (False, True)):
        if mode != 3 and n_seg != 100:
            continue
        name = route(kind, total, inject, frames, spans, lsu, mode, n_seg if mode == 3 else 0, point, trl, debug)
        if name:
            produced.add(name)
    assert ALL_INDEX - produced == set(UNREACHABLE)
    assert produced <= ALL_INDEX


# ------------------------------------------------ device helpers ------------------------------------------------
def table_info(sampler):
    from ogbench_b200 import _native

    info = _native.TableInfo()
    _native.check(_native.lib().ogb_sampler_table_info(sampler._sampler.ptr, C.byref(info)))
    return info


def kernel_names(handle):
    from ogbench_b200 import _native

    n = C.c_int32()
    _native.check(_native.lib().ogb_batch_kernel_names(handle.ptr, None, 0, C.byref(n)))
    buf = (C.c_char_p * max(n.value, 1))()
    _native.check(_native.lib().ogb_batch_kernel_names(handle.ptr, buf, n.value, C.byref(n)))
    return [buf[i].decode() for i in range(n.value)]


def make_sampler(fields, config, kind, **kw):
    from ogbench_b200 import ATCDataset, Dataset, GCDataset, HGCDataset

    cls = {'gc': GCDataset, 'hgc': HGCDataset, 'atc': ATCDataset}[kind]
    return cls(Dataset.create(**fields), config, output='numpy', **kw)


def row_of(arr):
    """The source row a gathered observation row names (its first int32 word)."""
    a = np.ascontiguousarray(arr)
    return a.reshape(len(a), -1).view(np.int32)[:, 0]


def assert_same(got, want, what):
    assert set(got) == set(want), (what, set(got) ^ set(want))
    for k in want:
        g, w = np.ascontiguousarray(got[k]), np.ascontiguousarray(want[k])
        assert g.dtype == w.dtype and g.shape == w.shape, (what, k, g.dtype, w.dtype, g.shape, w.shape)
        bad = np.nonzero((g.reshape(len(g), -1).view(np.uint8) != w.reshape(len(w), -1).view(np.uint8)).any(1))[0] if len(g) else []
        assert len(bad) == 0, (what, k, len(bad), bad[:5])


def closed_final(term, idxs):
    return term[np.searchsorted(term, idxs)]


def closed_first(term, idxs):
    init = np.concatenate([[0], term[:-1] + 1])
    return init[np.searchsorted(init, idxs, side='right') - 1]


# Goal kinds: (geom, offset or dist, u_traj).  u_traj 0.25 picks the trajectory goal, 0.75 the random one (p_traj = p_random
# = 0.5, p_cur = 0 below); the random goals read rand_pos, a permutation of every position.
GOAL_KINDS = [('random', True, 1, 0.75)] + [(f'offset={o}', True, o, 0.25) for o in (1, 2, 1 << 40)] + \
             [(f'dist={d!r}', False, d, 0.25) for d in (0.0, 0.5, np.nextafter(1.0, 0.0))]
MIX = dict(value_p_curgoal=0.0, value_p_trajgoal=0.5, value_p_randomgoal=0.5, actor_p_curgoal=0.0, actor_p_trajgoal=0.5,
           actor_p_randomgoal=0.5)


def goal_draws(n, n_choices, geom, value, u_traj, rng):
    g = GoalDraws(rand_pos=rng.permutation(np.arange(n) % n_choices).astype(np.int64))
    if geom:
        g.offset = np.full(n, value, np.int64)
    else:
        g.dist = np.full(n, value, np.float64)
    g.u_traj, g.u_cur = np.full(n, u_traj), np.full(n, 0.5)
    return g


def traj_goal(idxs, final, geom, value):
    if geom:
        return np.minimum(idxs + value, final)
    lo = np.minimum(idxs + 1, final)
    return np.round(lo * value + final * (1 - value)).astype(np.int64)


# ------------------------------------------------ every position, every goal kind ------------------------------------------------
SAMPLERS = ['gc', 'hgc', 'gc_fs3', 'trl', 'atc']


@pytest.mark.gpu
@pytest.mark.parametrize('name', EXHAUSTIVE)
def test_every_position_every_goal_kind(name):
    layout, mode, seg_shift = CATALOGUE[name]
    fields = with_rows(layout, 1, 1)
    n = len(fields['terminals'])
    rng = np.random.default_rng(abs(hash(name)) % 1000)
    for which in SAMPLERS:
        trl = which == 'trl'
        if which in ('gc_fs3', 'atc') and 'valids' not in fields:
            continue                                         # frame stacking needs the compact layout
        t = Tables(fields['terminals'], fields.get('valids'), trl)
        if trl and t.n_choices == 0:
            continue
        over = dict(MIX)
        if which == 'gc_fs3':
            over['frame_stack'] = 3
        if which == 'hgc':
            over['subgoal_steps'] = 5
        if trl:
            over.update(agent_name='trl', value_p_trajgoal=1.0, value_p_randomgoal=0.0)
        if which == 'atc':
            check_atc(make_sampler(fields, cfg(), 'atc'), fields, cfg(), (name, which))
            continue
        kind = 'hgc' if which == 'hgc' else 'gc'
        samplers = {}
        kinds = GOAL_KINDS if not trl else [g for g in GOAL_KINDS if g[0] != 'random']
        for gname, geom, value, u_traj in kinds:
            config = cfg(value_geom_sample=geom, actor_geom_sample=geom, **over)
            if geom not in samplers:
                samplers[geom] = make_sampler(fields, config, kind)
            sampler = samplers[geom]
            what = (name, which, gname)
            info = table_info(sampler)
            assert (info.valid_mode, info.seg_shift, info.n_choices) == (t.mode, t.seg_shift, t.n_choices), what
            assert (info.gap_shift, info.term_shift, info.n_seg_table) == (t.gap_shift, t.term_shift, t.n_seg_table), what
            rows = (np.nonzero(fields['terminals'] <= 0)[0] if trl else
                    np.arange(n) if t.mode == 0 else t.valid_idxs)
            if which == 'gc_fs3' and rows[-1] == n - 1:
                rows = rows[:-1]            # its stacked next_observations reads row n, an IndexError in the reference
            B = len(rows)
            d = Draws(idx_pos=np.arange(B, dtype=np.int64))
            d.goals = [goal_draws(B, t.n_choices, geom, value, u_traj, rng) for _ in range(2)]
            final = closed_final(t.term, rows)
            if trl:
                goal = traj_goal(rows, final, geom, value)
                d.trl_midpoints = rows + (goal - rows) // 2
            want = OracleSampler(fields, config, kind).sample(B, evaluation=True, source=DrawsSource(d))
            got = sampler.sample(B, evaluation=True, draws=d)
            assert_same(got, want, what)
            # closed forms, independent of the oracle
            obs = got['observations']
            if which == 'gc_fs3':            # frames idx - 2, idx - 1, idx, clamped at the trajectory's first row
                assert np.array_equal(row_of(obs[:, 2:3]), rows), what
                assert np.array_equal(row_of(obs[:, 0:1]), np.maximum(rows - 2, closed_first(t.term, rows))), what
            else:
                assert np.array_equal(row_of(obs), rows), what
            vg = row_of(got['value_goals'][:, -1:] if which == 'gc_fs3' else got['value_goals'])
            if u_traj < 0.5 or trl:
                assert np.array_equal(vg, traj_goal(rows, final, geom, value)), what
            else:
                assert np.array_equal(vg, (np.arange(n) if t.mode == 0 else t.valid_idxs)[d.goals[0].rand_pos]), what
            if gname == f'offset={1 << 40}':
                assert np.array_equal(vg, final), what
    check_helpers(fields, name)


def check_atc(sampler, fields, config, what):
    for k in (1, 3):
        oracle = OracleATCSampler(fields, config)
        try:
            anchors = oracle.valid_anchors(k)
        except ValueError:
            continue
        assert np.array_equal(sampler.get_valid_atc_idxs(k), anchors), what
        d = Draws(idx_pos=np.arange(len(anchors), dtype=np.int64))
        want = oracle.sample(len(anchors), k, evaluation=True, source=DrawsSource(d))
        got = sampler.sample(len(anchors), k, evaluation=True, draws=d)
        assert_same(got, want, what + (k,))
        assert np.array_equal(row_of(got['observations']), anchors), what
        assert np.array_equal(row_of(got['positive_observations']), anchors + k), what


def check_helpers(fields, name):
    """sample_goals with every row as idxs, and compute_high_next_idxs, against pick_goals / subgoal_step."""
    n = len(fields['terminals'])
    rng = np.random.default_rng(7)
    idxs = np.arange(n, dtype=np.int64)
    sampler = make_sampler(fields, cfg(**MIX), 'gc')        # (sample_goals takes the goal parameters as arguments)
    t = Tables(fields['terminals'], fields.get('valids'))
    for geom, value, u_traj in ((True, 3, 0.25), (True, 1 << 40, 0.25), (False, 0.5, 0.25), (True, 1, 0.75)):
        g = goal_draws(n, t.n_choices, geom, value, u_traj, rng)
        got = sampler._goals_native(idxs, 0.0, 0.5, geom, 0.99, g)
        final = closed_final(t.term, idxs)
        want, _ = pick_goals(idxs, final, None if t.mode == 0 else t.valid_idxs, 0.0, 0.5, geom, 0.99,
                             DrawsSource(Draws(goals=[g])), n)
        assert np.array_equal(got, want), (name, geom, value, u_traj)
    hgc = make_sampler(fields, cfg(subgoal_steps=5), 'hgc')
    final = closed_final(Tables(fields['terminals']).term, idxs)
    goal = np.where(rng.random(n) < 0.5, np.minimum(idxs + rng.integers(0, 9, n), final), rng.integers(0, n, n))
    for k in (1, 5, 40):
        nxt, steps = hgc.compute_high_next_idxs(idxs, final, goal, k)
        want_next, want_steps = subgoal_step(idxs, final, goal, k)
        assert np.array_equal(nxt, want_next) and np.array_equal(steps, want_steps), (name, k)


@pytest.mark.gpu
def test_view_of_resident_shards_builds_its_own_tables(tmp_path):
    """A shard of ResidentShards is a view: its valid and terminal tables come from the parent's flags at its rows."""
    from ogbench_b200 import GCDataset
    from ogbench_b200.loader import ResidentShards

    parts = [with_rows(from_lengths(np.random.default_rng(s).integers(17, 40, 50)), 1, 1) for s in (1, 2)]
    parts[1] = with_rows(from_invalid(1200, list(range(30, 1200, 30)) + [45]), 1, 1)     # min gap 14: the gap-rank search
    paths = []
    for i, p in enumerate(parts):
        paths.append(str(tmp_path / f'shard{i}.npz'))
        np.savez(paths[-1], **p)
    shards = ResidentShards(paths, load=lambda path: dict(np.load(path)))
    config = cfg(actor_geom_sample=True, **MIX)
    for i, part in enumerate(parts):
        t = Tables(part['terminals'], part['valids'])
        assert (t.mode, t.seg_shift) == ((3, 4), (2, -1))[i]
        sampler = GCDataset(shards[i], config, output='numpy')
        info = table_info(sampler)
        assert (info.valid_mode, info.seg_shift, info.gap_shift, info.n_choices) == (t.mode, t.seg_shift, t.gap_shift, t.n_choices), i
        B = t.n_choices
        d = Draws(idx_pos=np.arange(B, dtype=np.int64), goals=[goal_draws(B, B, True, 1 << 40, 0.25, np.random.default_rng(i))] * 2)
        got = sampler.sample(B, evaluation=True, draws=d)
        assert np.array_equal(row_of(got['observations']), t.valid_idxs), i         # the shard's own row numbers
        assert np.array_equal(row_of(got['value_goals']), closed_final(t.term, t.valid_idxs)), i
        want = OracleSampler(part, config, 'gc').sample(B, evaluation=True, source=DrawsSource(d))
        assert_same(got, want, ('view', i))


# ------------------------------------------------ every kernel instance, both draw modes ------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('case', list(INSTANCES))
def test_every_index_instance_in_both_draw_modes(case):
    from oracle import philox_np
    from tests.test_gpu_philox import goal_sets_for

    layout, kind, obs, act, over, call, rows = INSTANCES[case]
    fields = instance_fields(case)
    config = instance_config(case)
    t = catalogue_tables(layout)
    rng = np.random.default_rng(3)
    for inject in instance_modes(case):
        what = (case, 'validation' if inject else 'philox')
        expected = expected_kernels(case, inject)
        if call == 'plain':
            from ogbench_b200 import Dataset

            ds = Dataset.create(**fields)
            ps = ds._plain_sampler()
            handle = ps.sample_native(rows)
            got = ps.wrap(handle)
            r = row_of(got['observations'])
            assert r.min() >= 0 and r.max() < len(fields['terminals']), what
            for k in fields:
                assert np.array_equal(np.asarray(got[k]).view(np.uint8), fields[k][r].view(np.uint8)), (what, k)
        elif call in ('gather', 'cropped'):
            from ogbench_b200 import _native
            from ogbench_b200.datasets import BatchHandle

            sampler = make_sampler(fields, config, kind)
            idxs = rng.integers(0, len(fields['terminals']) - 1, rows).astype(np.int64)
            idxs[:min(rows, len(fields['terminals']))] = np.arange(min(rows, len(fields['terminals'])))
            out = C.c_void_p()
            if call == 'gather':
                _native.check(_native.lib().ogb_sampler_gather(sampler._sampler.ptr, 0, idxs.ctypes.data_as(C.c_void_p), rows, C.byref(out)))
                want = stacked_frames(fields['observations'], np.concatenate([[0], t.term[:-1] + 1]), idxs, 3)
            else:
                crop = rng.integers(0, 7, (rows, 2)).astype(np.int64)
                _native.check(_native.lib().ogb_sampler_gather_cropped(sampler._sampler.ptr, idxs.ctypes.data_as(C.c_void_p), rows,
                                                                       crop.ctypes.data_as(C.c_void_p), 3, C.byref(out)))
                src = fields['observations'][idxs]
                want = shifted_edge_crop(src, crop, 3) if src.ndim == 4 else src
            handle = BatchHandle(out, 0, None)
            got = next(iter(sampler._sampler.wrap(handle).values()))
            assert np.array_equal(np.asarray(got).view(np.uint8), want.view(np.uint8)), what
        else:
            sampler = make_sampler(fields, config, kind, seed=11, stream_id=2)
            n_choices = t.n_choices
            if inject:
                d = Draws(idx_pos=(np.arange(rows) % n_choices).astype(np.int64))
                d.goals = [goal_draws(rows, n_choices, bool(config[f'{s}_geom_sample']), 3 if config[f'{s}_geom_sample'] else 0.5,
                                      0.25 + 0.5 * (i % 2), rng) for i, s in enumerate(['value'] + ['actor'])]
                handle = sampler._sampler.sample_native(rows, evaluation=True, draws=d)
                knife = np.zeros(rows, bool)
            else:
                handle = sampler._sampler.sample_native(rows, evaluation=True)
                d, knife = philox_np.philox_draws(11, 2, 0, rows, n_choices, goal_sets_for(config, kind), False, 0.0)
            got = sampler._sampler.wrap(handle)
            want = OracleSampler(fields, config, kind).sample(rows, evaluation=True, source=DrawsSource(d))
            assert knife.mean() < 1e-3
            assert_same({k: np.asarray(v)[~knife] for k, v in got.items()}, {k: v[~knife] for k, v in want.items()}, what)
            rows_drawn = (np.arange(len(fields['terminals'])) if t.mode == 0 else t.valid_idxs)[d.idx_pos]
            obs_rows = row_of(np.asarray(got['observations'])[:, -1:] if over.get('frame_stack') else got['observations'])
            assert np.array_equal(obs_rows[~knife], rows_drawn[~knife]), what
        assert kernel_names(handle) == expected, (what, kernel_names(handle), expected)


# ------------------------------------------------ two large cases ------------------------------------------------
LARGE = {
    # ~8M rows, invalid rows ~40 apart with one pair 3 apart: no segment table, gap_shift 4 raised to 6 by the 2^17 cap
    'gap_ranks_8M': dict(rows=8_000_000, lo=30, hi=50, close_pair=True),
    # >= 2^26 + 2^20 valid rows, min gap 16..31: (n_valid >> 4) > 2^22 refuses the segment table
    'gap_ranks_69M': dict(valid=(1 << 26) + (1 << 20), lo=17, hi=32, close_pair=False),
}


def large_lengths(spec):
    rng = np.random.default_rng(9)
    target = spec.get('valid', spec.get('rows'))
    lengths = rng.integers(spec['lo'], spec['hi'] + 1, target // spec['lo'] + 10).astype(np.int64)
    counted = np.cumsum(lengths - 1 if 'valid' in spec else lengths)
    lengths = lengths[:int(np.searchsorted(counted, target)) + 1]
    if spec['close_pair']:
        lengths[1000] = 4                                # two invalid rows 3 valid rows apart
    return lengths


def large_tables(spec):
    """Tables of the large layout from its trajectory lengths alone (no per-row host arrays)."""
    lengths = large_lengths(spec)
    valid = lengths - 1
    t = Tables.__new__(Tables)
    t.why = set()
    t.n_valid = int(valid.sum())
    n_gaps = len(lengths)
    c = np.cumsum(valid)
    min_gap = int(np.min(np.diff(c)))
    t.gap_shift = shift_for(t.n_valid + 1, n_gaps)
    t.why.add('gap_shift capped' if t.gap_shift != _mean_gap_shift(t.n_valid + 1, n_gaps) else 'gap_shift from mean gap')
    t.mode, t.seg_shift = 2, -1
    shift = 4
    while (1 << (shift + 1)) <= min_gap:
        shift += 1
    if min_gap < SEG_MIN_GAP:
        t.why.add('min_gap<16')
    elif (t.n_valid >> shift) > SEG_MAX_BUCKETS:
        t.why.add('n_valid>>shift>2^22')
    else:
        t.mode = 3
    t.lengths, t.c = lengths, c
    return t


@pytest.mark.gpu
@pytest.mark.parametrize('name', list(LARGE))
def test_large_gap_rank_tables(name):
    """Every bucket-boundary position +- 1 and 1M random positions, against valid_idxs[pos] and the trajectory's final row
    in closed form (trajectory t: rows start[t] .. start[t] + L - 1, its last row invalid, final state start[t] + L - 2)."""
    from ogbench_b200 import Dataset, GCDataset

    t = large_tables(LARGE[name])
    lengths = t.lengths
    size = int(lengths.sum())
    starts = np.concatenate([[0], np.cumsum(lengths)[:-1]])
    valids = np.ones(size, np.float32)
    valids[starts + lengths - 1] = 0
    terminals = 1 - valids
    terminals[starts + lengths - 2] = 1
    obs = np.arange(size, dtype=np.int32).view(np.float32)[:, None]
    config = cfg(value_p_curgoal=0.0, value_p_trajgoal=1.0, value_p_randomgoal=0.0, actor_geom_sample=True)
    sampler = GCDataset(Dataset.create(observations=obs, terminals=terminals, valids=valids), config, output='numpy')
    del obs, valids, terminals
    info = table_info(sampler)
    assert (info.valid_mode, info.seg_shift, info.gap_shift, info.n_choices) == (2, -1, t.gap_shift, t.n_valid), name
    b = np.arange((t.n_valid >> t.gap_shift) + 1, dtype=np.int64) << t.gap_shift
    pos = np.concatenate([b - 1, b, b + 1, np.random.default_rng(1).integers(0, t.n_valid, 1 << 20)])
    pos = pos[(pos >= 0) & (pos < t.n_valid)]
    B = len(pos)
    d = Draws(idx_pos=pos)
    d.goals = [GoalDraws(rand_pos=pos, offset=np.full(B, 1 << 40, np.int64), u_traj=np.full(B, 0.5), u_cur=np.full(B, 0.5))] * 2
    got = sampler.sample(B, evaluation=True, draws=d)
    traj = np.searchsorted(t.c, pos, side='right')                      # c[t] = valid rows in trajectories 0..t
    before = np.concatenate([[0], t.c])[traj]
    want_rows = starts[traj] + (pos - before)
    assert np.array_equal(row_of(got['observations']), want_rows), name
    assert np.array_equal(row_of(got['value_goals']), starts[traj] + lengths[traj] - 2), name
    assert np.array_equal(row_of(got['actor_goals']), starts[traj] + lengths[traj] - 2), name
    assert np.array_equal(got['masks'], (want_rows != starts[traj] + lengths[traj] - 2).astype(np.float64)), name
