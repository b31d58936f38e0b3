"""Row gathers (every vector key of GCDataset, HGCDataset, TRL and Dataset.sample) against plain references, at every row
size class, drain kind, rows-per-item value and launch split of the host planner (`classify_rows`, `split_span_jobs` and
`fill_row_tables`, ogb_sampler.cu).

`RowPlan` below restates the planner in Python: the record layout of `ogb_dataset_create`, the key plan, tiny versus span
fields and span merging, stage budget and rows per item, the launch split, the drain kind of every output, fused versus
un-fused launches and the register-staged (LSU) keys.  `test_case_plan_reaches_every_path` (no GPU) checks that the case
list reaches every path; every device case asserts that the launch count and the dominant kernel are the ones the
restatement predicts, so a shape cannot quietly move to another path.

References: small cases are compared bit for bit with the oracle (rng='numpy' under a fixed np.random.seed, and the
Philox draws rebuilt by oracle/philox_np.py for the split cases); large cases read the index vectors (debug bit 0) and
compare every row key with numpy fancy indexing of the host fields, with a canary pass (debug bits 0 and 1) whose key
gaps must stay untouched, and a debug-off pass that must equal it byte for byte.
"""

import ctypes as C
import json
import os
import subprocess
import sys
from collections import defaultdict

import numpy as np
import pytest

from tests.golden.make_golden import cfg, ragged, toy_fields
from tests.gpu_util import device_sampler, oracle_with_draws, to_host

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# ------------------------------------------------ the host planner, restated ------------------------------------------------
REC_MAX_ROW, REC_MAX_BYTES = 2048, 4096             # ogb_dataset_create: kRecordMaxRow, kRecordMaxBytes
ASYNC_MAX_STRIDE = 4096                             # relabel_rows.cuh kAsyncMaxStride
MAX_ROW_JOBS, MAX_ITEMS, MAX_ITEM_OUTS = 24, 64, 192
MAX_TINY_JOBS, MAX_TINY_GROUPS, MAX_TINY_FIELDS = 16, 2, 16
OVERLAP_MIN_ROWS = 32768
SMEM_LIMIT = 225 * 1024
SLOT_IDX, SLOT_NEXT = 0, 1
GC_VALUE_GOAL, GC_ACTOR_GOAL, GC_TRL_MID, GC_TRL_PLUS1 = 2, 3, 4, 5
HGC_HV_GOAL, HGC_HV_NEXT, HGC_LV_NEXT, HGC_HA_GOAL, HGC_HA_NEXT, HGC_LA_GOAL, HGC_LA_NEXT, HGC_LV_GOAL = 2, 3, 4, 5, 6, 7, 8, 9
DENSE16, WORDS, WORDS_UNALIGNED, ELEMS_U16, ELEMS_U8 = 'DENSE16', 'WORDS', 'WORDS_UNALIGNED', 'ELEMS_U16', 'ELEMS_U8'
FUSED, ASYNC, LSU, INDEX = 'relabel_gather_kernel', 'gather_rows_async_kernel', 'gather_rows_kernel', 'relabel_index_kernel'


class Refused(Exception):
    """The planner refuses the batch (OGB_ERR_UNSUPPORTED -> NotImplementedError)."""


def round_up(x, a):
    return (x + a - 1) // a * a


def vec_log2(a, b):
    """largest_vec_log2: the largest power of two <= 16 dividing both."""
    v = 4
    while v > 0 and (a % (1 << v) or b % (1 << v)):
        v -= 1
    return v


def rows_per_item(pitch, budget):
    r = 32
    while r > 1 and r * pitch > budget:
        r //= 2
    return r


def stage_budget(max_pitch):
    return max(6144 if max_pitch > 256 else 4096, max_pitch)


def under(name, prefix):
    return name == prefix or name.startswith(prefix + '/')


def native_fields(fields):
    """Field order and names of the native dataset: pytrees are flattened with sorted keys (datasets._flatten)."""
    from ogbench_b200.datasets import _flatten

    return _flatten(fields) if any(isinstance(v, dict) for v in fields.values()) else dict(fields)


class Field:
    def __init__(self, name, arr):
        self.name = name
        self.n = len(arr)
        self.row = arr.dtype.itemsize * int(np.prod(arr.shape[1:], dtype=np.int64))
        self.stride = self.row if self.row <= 16 else round_up(self.row, 32)
        self.in_record, self.rec_off = False, 0
        self.src = name                                 # host field the rows come from (the shadow: 'observations')


def record_layout(fields, env):
    """ogb_dataset_create: fields of <= 2 KB rows share one record of <= 4 KB, observations first, then by decreasing
    alignment; 32-, 64- or 128-byte multiple strides; the shadow copy of the next row's observation when it is <= 16 B."""
    fl = [Field(k, v) for k, v in fields.items()]
    align = lambda f: 16 if f.row > 16 else next(a for a in (16, 8, 4, 2, 1) if f.row % a == 0)
    order = [] if 'OGB_NO_RECORDS' in env else [f for f in fl if f.row <= REC_MAX_ROW]
    order.sort(key=lambda f: (f.name != 'observations', -align(f)))
    cursor, packed = 0, []
    for f in order:
        off = round_up(cursor, align(f))
        if off + f.row > REC_MAX_BYTES:
            continue
        f.rec_off, f.in_record, cursor = off, True, off + f.row
        packed.append(f)
    stride, used = 0, 0
    if len(packed) < 2:
        for f in packed:
            f.in_record = False
    else:
        used, stride = cursor, 32 if cursor <= 32 else 64 if cursor <= 64 else round_up(cursor, 128)
        for f in packed:
            f.stride = stride
    obs = [f for f in fl if under(f.name, 'observations')]
    if obs and len(obs) == 1 and not any(under(f.name, 'next_observations') for f in fl):
        o = obs[0]
        off = round_up(used, align(o))
        if o.in_record and o.row <= 16 and off + o.row <= stride:
            sh = Field('\x01next_observations', np.zeros((1, 0), np.uint8))
            sh.row, sh.stride, sh.in_record, sh.rec_off, sh.src, sh.n = o.row, stride, True, off, o.name, o.n
            fl.append(sh)
    return fl


class Key:
    def __init__(self, name, field, slot, alias):
        self.name, self.field, self.slot, self.alias = name, field, slot, alias


def key_plan(fl, kind, config, dedup):
    """build_plan: the row keys (name, field, index-vector slot), with aliases (dedup) marked."""
    keys = []
    canon = list(range(10))
    if kind == 'hgc' and dedup:
        value, actor, low = hgc_steps(config)
        if low == value:
            canon[HGC_LV_NEXT] = HGC_HV_NEXT
        if low == actor:
            canon[HGC_LA_NEXT] = HGC_HA_NEXT
    public = [f for f in fl if not f.name.startswith('\x01')]
    obs = [f for f in public if under(f.name, 'observations')]

    def field_key(name, f, slot):
        slot = canon[slot]
        alias = dedup and any(k.field is f and k.slot == slot and not k.alias for k in keys)
        keys.append(Key(name, f, slot, alias))

    def obs_key(name, slot):
        for f in obs:
            field_key(name + f.name[len('observations'):], f, slot)

    def alias(name, target):
        for k in list(keys):
            if under(k.name, target):
                keys.append(Key(name + k.name[len(target):], k.field, k.slot, True))

    for f in public:
        if f is obs[0]:
            obs_key('observations', SLOT_IDX)
        elif not under(f.name, 'observations'):
            field_key(f.name, f, SLOT_IDX)
    if not any(under(f.name, 'next_observations') for f in public):
        shadow = [f for f in fl if f.name.startswith('\x01')]
        if shadow:
            field_key('next_observations', shadow[0], SLOT_IDX)
        else:
            obs_key('next_observations', SLOT_NEXT)
    if kind in ('gc', 'trl'):
        obs_key('value_goals', GC_VALUE_GOAL)
        obs_key('actor_goals', GC_ACTOR_GOAL)
        if kind == 'trl':
            actions = next(f for f in public if f.name == 'actions')
            obs_key('value_goal_observations', GC_VALUE_GOAL)
            obs_key('actor_goal_observations', GC_VALUE_GOAL)
            obs_key('value_midpoint_observations', GC_TRL_MID)
            field_key('value_midpoint_actions', actions, GC_TRL_MID)
            field_key('next_actions', actions, GC_TRL_PLUS1)
            obs_key('value_midpoint_goals', GC_TRL_MID)
            obs_key('value_cur_goals', SLOT_IDX)
            obs_key('value_next_goals', GC_TRL_PLUS1)
    elif kind == 'hgc':
        for name, slot in (('high_value_reps', SLOT_IDX), ('high_value_goals', HGC_HV_GOAL), ('high_value_actions', HGC_HV_NEXT),
                           ('high_value_next_observations', HGC_HV_NEXT), ('low_value_next_observations', HGC_LV_NEXT)):
            obs_key(name, slot)
        if config.get('low_discount') is not None:
            obs_key('low_value_goals', HGC_LV_GOAL)
        alias('value_goals', 'high_value_goals')
        for name, slot in (('high_actor_goals', HGC_HA_GOAL), ('high_actor_actions', HGC_HA_NEXT),
                           ('high_actor_next_observations', HGC_HA_NEXT)):
            obs_key(name, slot)
        alias('high_actor_targets', 'high_actor_actions')
        for name, slot in (('low_actor_goals', HGC_LA_GOAL), ('low_actor_goal_observations', HGC_LA_GOAL),
                           ('low_actor_next_observations', HGC_LA_NEXT)):
            obs_key(name, slot)
    return keys


def hgc_steps(config):
    high = config.get('high_subgoal_steps', config['subgoal_steps'])
    value = high if config.get('value_subgoal_steps') is None else config['value_subgoal_steps']
    actor = high if config.get('actor_subgoal_steps') is None else config['actor_subgoal_steps']
    return value, actor, config.get('low_subgoal_steps', config['subgoal_steps'])


class Span:
    def __init__(self, slot, nbytes, outs):
        self.slot, self.bytes, self.outs = slot, nbytes, outs     # outs: [(Key, byte offset inside the span)]


class RowPlan:
    """classify_rows and split_span_jobs for one sample() call of `total` rows (no image keys)."""

    def __init__(self, fields, kind, config=None, total=1, dedup=True, env=None, philox=True, host_chunks=1):
        env = env or {}
        config = config or {}
        self.fl = record_layout(native_fields(fields), env)
        self.keys = key_plan(self.fl, kind, config, dedup)
        lsu_env = env.get('OGB_GATHER') == 'lsu'
        n = self.fl[0].n
        takes_async = lambda f: f.row > 16 and f.stride <= ASYNC_MAX_STRIDE and n * f.stride < 1 << 36 and not lsu_env
        rows = [k for k in self.keys if not k.alias]
        # fused: vector keys on the cp.async path, and not a big HGC launch (OGB_FUSE=0|1 overrides)
        fuse_env = env.get('OGB_FUSE')
        fuse = ((fuse_env == '1' if fuse_env is not None else (total < OVERLAP_MIN_ROWS or kind != 'hgc'))
                and any(takes_async(k.field) for k in rows))
        self.n_tiny, self.n_tiny_groups, self.n_tiny_fields = 0, 0, 0
        spans, self.lsu = [], []
        record_keys = defaultdict(list)

        def add_tiny(k):
            if k.field.row > 16 or self.n_tiny >= MAX_TINY_JOBS:
                return False
            self.n_tiny += 1
            return True

        for k in rows:
            f = k.field
            if f.in_record and f.stride <= ASYNC_MAX_STRIDE and not lsu_env and n * f.stride < 1 << 36:
                record_keys[k.slot].append(k)
            elif add_tiny(k):
                pass
            elif takes_async(f):
                spans.append(Span(k.slot, round_up(f.row, 16), [(k, 0)]))
            else:
                self.lsu.append(k)
        for slot in sorted(record_keys):
            ks = sorted(record_keys[slot], key=lambda k: k.field.rec_off)
            k0 = 0
            while k0 < len(ks):
                f0 = ks[k0].field
                lo, hi, k1, has_long = f0.rec_off & ~15, f0.rec_off + f0.row, k0 + 1, f0.row > 16
                while k1 < len(ks):
                    fn = ks[k1].field
                    if fn.rec_off > hi + 32:
                        break
                    pitch = round_up(max(hi, fn.rec_off + fn.row) - lo, 16)
                    if 32 // rows_per_item(pitch, stage_budget(pitch)) * (k1 - k0 + 1) > MAX_ITEM_OUTS:
                        break
                    hi, has_long, k1 = max(hi, fn.rec_off + fn.row), has_long or fn.row > 16, k1 + 1
                if has_long:
                    spans.append(Span(slot, round_up(hi - lo, 16), [(k, k.field.rec_off - lo) for k in ks[k0:k1]]))
                else:
                    k = k0
                    while 'OGB_NO_TINY_GROUPS' not in env and k < k1 and self.n_tiny_groups < MAX_TINY_GROUPS:
                        glo, kk = ks[k].field.rec_off & ~15, k
                        while kk < k1:
                            fk = ks[kk].field
                            if (fk.row % 4 or fk.rec_off % 4 or fk.rec_off + fk.row > glo + 32
                                    or (fk.row == 16 and (fk.rec_off - glo) % 16) or self.n_tiny_fields + kk - k >= MAX_TINY_FIELDS):
                                break
                            kk += 1
                        if kk - k < 2:
                            break
                        self.n_tiny_groups += 1
                        self.n_tiny_fields += kk - k
                        k = kk
                    for t in range(k, k1):
                        if not add_tiny(ks[t]):
                            fk = ks[t].field
                            l2 = fk.rec_off & ~15
                            spans.append(Span(slot, round_up(fk.rec_off + fk.row - l2, 16), [(ks[t], fk.rec_off - l2)]))
                k0 = k1
        self.spans = spans
        self.fused = fuse and bool(spans)
        # launch split: the largest prefix of the remaining jobs whose items and outputs fit one launch
        self.launches, self.split_reasons, self.drains = [], set(), set()
        self.rows_per_item, self.chunk_walks = set(), set()
        q = 0
        while q < len(spans):
            q1 = min(len(spans), q + MAX_ROW_JOBS)
            reason = 'jobs' if q1 < len(spans) else None
            while True:
                budget = stage_budget(max(s.bytes for s in spans[q:q1]))
                items = sum(32 // rows_per_item(s.bytes, budget) for s in spans[q:q1])
                outs = sum(32 // rows_per_item(s.bytes, budget) * len(s.outs) for s in spans[q:q1])
                if (items <= MAX_ITEMS and outs <= MAX_ITEM_OUTS) or q1 == q + 1:
                    if items > MAX_ITEMS or outs > MAX_ITEM_OUTS:
                        raise Refused(f'a {spans[q].bytes}-byte row span with {len(spans[q].outs)} keys')
                    break
                reason = 'items' if items > MAX_ITEMS else 'outputs'
                q1 -= 1
            if q1 < len(spans):
                self.split_reasons.add(reason)
            group = spans[q:q1]
            stage = round_up(max(rows_per_item(s.bytes, budget) * s.bytes for s in group), 128)
            for s in group:
                rpi = rows_per_item(s.bytes, budget)
                self.rows_per_item.add((rpi, budget if rpi == 16 else None))
                cpr = s.bytes // 16
                self.chunk_walks.add('cpr>32' if cpr > 32 else 'divides' if 32 % cpr == 0 else 'does not divide')
                for sub in range(0, 32, rpi):
                    for k, soff in s.outs:
                        self.drains.add(self.drain(k.field.row, soff, s.bytes, sub))
            self.launches.append(dict(first=q, items=items, outs=outs, stage=stage,
                                      shape=self.shape(kind, q == 0 and self.fused, philox, stage)))
            q = q1
        # register-staged keys: one launch per element width and 24 keys
        self.lsu_vecs = [vec_log2(k.field.row, k.field.stride) for k in self.lsu]
        n_lsu = sum(-(-self.lsu_vecs.count(v) // MAX_ROW_JOBS) for v in range(5))
        n_chunks = min(host_chunks, 8, total // 16384) if host_chunks > 1 and philox and total >= 2 * 16384 else 1
        self.n_launches = (1 + len(self.launches) - (1 if self.fused else 0) + n_lsu) * n_chunks
        self.dominant = FUSED if self.fused else ASYNC if spans else LSU if self.lsu else INDEX
        self.write_vecs_needed = self.fused and (len(self.launches) > 1 or bool(self.lsu))

    @staticmethod
    def drain(row, soff, pitch, sub):
        if row % 16 == 0 and pitch == row:
            return DENSE16
        if row % 4 == 0 and soff % 4 == 0:
            return WORDS if sub * row % 16 == 0 else WORDS_UNALIGNED
        return ELEMS_U16 if row % 2 == 0 and soff % 2 == 0 else ELEMS_U8

    @staticmethod
    def shape(kind, fused_here, philox, stage):
        if fused_here and kind in ('gc', 'trl') and philox:
            return 220 if 20 * 2 * stage <= 200 * 1024 else 216
        return 310 if not fused_here and stage > 4096 and 10 * 3 * stage <= 200 * 1024 else 308

    def smem(self, launch):
        """Shared memory of one row-gather launch: item and output tables, a tile FIFO per warp, the rings."""
        warps, stages = launch['shape'] % 100, launch['shape'] // 100
        return round_up(launch['items'] * 48 + launch['outs'] * 32 + warps * 16, 128) + warps * stages * launch['stage']

    @property
    def refused_smem(self):
        return any(self.smem(la) > SMEM_LIMIT for la in self.launches)


# ------------------------------------------------ the cases ------------------------------------------------
F32, F64, F16, U8, I32, I64, BOOL = np.float32, np.float64, np.float16, np.uint8, np.int32, np.int64, np.bool_


def make_fields(case):
    """A ragged compact dataset (toy_fields) with the case's observations and extra fields."""
    seed = case['seed']
    n_traj, lo, hi = case.get('traj', (30, 5, 60))
    obs_shape, obs_dtype = case['obs']
    fields = toy_fields(seed, ragged(seed, n_traj, lo, hi), (1,), case.get('act', 4), np.float32)
    n = len(fields['terminals'])
    rng = np.random.default_rng(seed + 1)

    def rand(shape, dtype):
        dt = np.dtype(dtype)
        if dt == np.bool_:
            return rng.integers(0, 2, (n, *shape)).astype(bool)
        if dt.kind in 'ui':
            return rng.integers(0, min(np.iinfo(dt).max, 1 << 30), (n, *shape), endpoint=True).astype(dt)
        return rng.standard_normal((n, *shape)).astype(dt)

    if case.get('leaves'):
        fields['observations'] = {f'leaf_{i}': rand(obs_shape, obs_dtype) for i in range(case['leaves'])}
    else:
        fields['observations'] = rand(obs_shape, obs_dtype)
    for name, (shape, dtype) in case.get('extra', {}).items():
        fields[name] = rand(shape, dtype)
    return fields


def make_config(case):
    kind = case['kind']
    over = dict(case.get('cfg', {}))
    if kind == 'hgc':
        over.setdefault('subgoal_steps', 5)
    if kind == 'trl':   # value goals from the trajectory only (the reference asserts idxs != value goal, datasets.py:257)
        over.update(agent_name='trl', value_p_curgoal=0.0, value_p_trajgoal=1.0, value_p_randomgoal=0.0)
    return cfg(**over)


def plan_of(case, total, env=None, philox=True, host_chunks=1):
    return RowPlan(make_fields(case), case['kind'], make_config(case), total, case.get('dedup', True), env, philox, host_chunks)


def C_(name, kind, obs, seed, **kw):
    return dict(name=name, kind=kind, obs=obs, seed=seed, **kw)


def smalls(k, shape=(1,), dtype=F32):
    return {f'x{i:02d}': (shape, dtype) for i in range(k)}


# Observations of 1-17 bytes next to longer fields (tiny rows drained inside a span), every pitch boundary of the stage
# budget, rows in arrays of their own, odd element counts of every dtype.
ORACLE_CASES = [
    C_('obs1-u8', 'gc', ((1,), U8), 1, extra={'long': ((40,), F32)}, B=31),
    C_('obs6-u8', 'gc', ((6,), U8), 2, extra={'long': ((10,), F64)}, B=33),
    C_('obs12-f32', 'gc', ((3,), F32), 3, extra={'long': ((9,), F16), 'flag': ((3,), BOOL)}, B=33),
    C_('obs17-u8', 'gc', ((17,), U8), 4, extra={'id': ((1,), I64)}, B=33),
    C_('obs18-f16', 'gc', ((9,), F16), 5, extra={'u': ((19,), U8)}, B=31),
    C_('pitch128', 'gc', ((32,), F32), 6, B=1000),
    C_('pitch144', 'gc', ((36,), F32), 7, extra={'i': ((3,), I32)}, B=33),
    C_('pitch256', 'hgc', ((32,), F64), 8, B=33),
    C_('pitch272', 'gc', ((68,), F32), 9, B=31),
    C_('pitch384', 'gc', ((96,), F32), 10, extra={'k': ((2,), I64)}, B=33),
    C_('pitch400', 'hgc', ((100,), F32), 11, B=31),
    C_('pitch768', 'gc', ((192,), F32), 12, B=33),
    C_('pitch784', 'gc', ((392,), F16), 13, B=33),
    C_('pitch1536', 'gc', ((384,), F32), 14, B=33),
    C_('pitch1552', 'gc', ((194,), F64), 15, B=31),
    C_('own2048', 'gc', ((512,), F32), 16, extra={'fill': ((512,), F32)}, B=33),
    C_('own2064', 'gc', ((516,), F32), 17, B=33),
    C_('pitch3072', 'gc', ((768,), F32), 18, B=31),
    C_('pitch3088', 'gc', ((3088,), U8), 19, B=33),
    C_('pitch4096', 'gc', ((1024,), F32), 20, B=33),
    C_('unaligned2404', 'gc', ((601,), F32), 21, B=33),
    C_('lsu', 'gc', ((1025,), F32), 22, extra={'b': ((4097,), U8), 'h': ((2049,), F16), 'd': ((513,), F64), 'w': ((1028,), F32)},
       B=33, traj=(10, 5, 40)),
    C_('plain', 'plain', ((150,), F32), 23, extra={'h': ((9,), F16), 'b': ((17,), U8), 'z': ((20,), BOOL)}, B=1000),
    C_('b1', 'gc', ((29,), F32), 24, B=1),
    C_('hgc-fused', 'hgc', ((96,), F32), 25, extra={'i': ((5,), I32)}, B=1000),
    C_('trl', 'trl', ((45,), F32), 26, B=1000, K=1),
]
# Launches split while the index algebra is fused into the first one: the later launches read the index vectors the
# fused launch stores.
SPLIT_CASES = [
    # 2,400-byte observations: 16 items in each of four slots + the 48-byte record span at IDX (8-float actions,
    # terminals, valids) = 65 items
    C_('split-items-gc', 'gc', ((600,), F32), 31, act=8, B=1000),
    # HGC below 32,768 rows, no key dedup: 9 slots x 8 items
    C_('split-items-hgc', 'hgc', ((300,), F32), 32, B=1000, dedup=False, cfg=dict(subgoal_steps=4)),
    C_('split-items-trl', 'trl', ((600,), F32), 33, act=8, B=257),
    # 1,200-byte observations + 19 small fields: 8 items x 22 outputs at IDX, 200 outputs in all
    C_('split-outputs', 'gc', ((300,), F32), 34, extra=smalls(19), B=1000),
    # a full 4 KB record (observations, actions and two wide fields): the small fields get arrays of their own, one
    # span job each, 26 jobs
    C_('split-jobs', 'gc', ((8,), F32), 35, act=8, extra={'big_a': ((512,), F32), 'big_b': ((496,), F32), **smalls(22, (5,))}, B=500),
    # eight 100-float leaves in the record: 32 items x 8 outputs per slot did not fit one launch
    C_('pytree-8x100', 'gc', ((100,), F32), 36, leaves=8, B=513),
]
# Row counts the oracle is too slow for: index vectors + numpy fancy indexing.  The fused 2 x 20 launch needs more than
# 148 SMs x 20 warps x 32 rows (~95 K rows) for ticket-scheduled tiles; HGC at >= 32,768 rows runs un-fused.
BIG_CASES = [
    C_('big-gc-fused', 'gc', ((29,), F32), 41, B=25000, K=4, traj=(400, 20, 400)),
    C_('big-hgc-unfused', 'hgc', ((96,), F32), 42, B=4096, K=9, traj=(300, 20, 300)),
    C_('big-hgc-unfused-nodedup', 'hgc', ((69,), F32), 43, B=33000, dedup=False, traj=(300, 20, 300)),
    C_('big-split-gc', 'gc', ((600,), F32), 44, act=8, B=20000, K=2),
    C_('big-split-outputs', 'gc', ((300,), F32), 45, extra=smalls(19), B=40000),
    C_('big-lsu', 'gc', ((1025,), F32), 46, extra={'b': ((4097,), U8), 'w': ((1028,), F32)}, B=8000, traj=(10, 5, 40)),
    C_('big-pytree-8x100', 'gc', ((100,), F32), 47, leaves=8, B=20000),
]
ALL_CASES = ORACLE_CASES + SPLIT_CASES + BIG_CASES


def case_total(case):
    return case['B'] * case.get('K', 1)


# ------------------------------------------------ device legs ------------------------------------------------
def batch_info(handle):
    from ogbench_b200 import _native

    n, name, ms = C.c_int32(), C.c_char_p(), C.c_float()
    _native.check(_native.lib().ogb_batch_launches(handle.ptr, C.byref(n)))
    _native.check(_native.lib().ogb_batch_dominant_kernel(handle.ptr, C.byref(name), C.byref(ms)))
    return n.value, name.value.decode()


def check_path(handle, plan, what):
    launches, kernel = batch_info(handle)
    assert (launches, kernel.split('<')[0]) == (plan.n_launches, plan.dominant), (what, launches, kernel, plan.n_launches, plan.dominant)
    return kernel


def assert_same(got, want, what):
    assert set(got) == set(want), (what, set(got) ^ set(want))
    for k in want:
        g, w = np.asarray(got[k]), np.asarray(want[k])
        assert g.dtype == w.dtype and g.shape == w.shape, (what, k, g.dtype, w.dtype, g.shape, w.shape)
        if not np.array_equal(g, w):
            bad = np.nonzero((g != w).reshape(len(w), -1).any(axis=1))[0]
            raise AssertionError(f'{what} {k}: {len(bad)} of {len(w)} rows differ, first {bad[:8].tolist()}')


def sampler_for(case, fields, **kw):
    if case['kind'] == 'plain':
        from ogbench_b200 import Dataset

        ds = Dataset.create(**{k: v.copy() for k, v in fields.items()})
        for name, value in kw.items():
            setattr(ds, name, value)
        return ds
    kind = 'gc' if case['kind'] == 'trl' else case['kind']
    return device_sampler(fields, make_config(case), kind, dedup=case.get('dedup', True), **kw)


def plain_reference(fields, idxs):
    """Dataset.sample (datasets.py:72-83): every field at idxs, next_observations at min(idx + 1, size - 1)."""
    n = len(fields['terminals'])
    out = {k: v[idxs] for k, v in fields.items()}
    out['next_observations'] = fields['observations'][np.minimum(idxs + 1, n - 1)]
    return out


def numpy_leg(case, fields, debug, seed):
    """rng='numpy' against the oracle (or the plain reference) under the same np.random.seed; returns the native batch."""
    B = case['B']
    kind = case['kind']
    if kind == 'plain':
        ds = sampler_for(case, fields, rng='numpy', output='numpy')
        ds._plain_sampler().set_debug(debug)
        np.random.seed(seed)
        want = plain_reference(fields, ds.get_random_idxs(B))
        np.random.seed(seed)
        assert_same(ds.sample(B), want, f'{case["name"]} debug={debug}')
        return ds._plain_sampler().sample_native(B, idxs=ds.get_random_idxs(B))
    sampler = sampler_for(case, fields, rng='numpy', output='numpy')
    sampler._sampler.set_debug(debug)
    okind = 'gc' if kind == 'trl' else kind
    np.random.seed(seed)
    _, want = oracle_with_draws(fields, make_config(case), okind, B)
    np.random.seed(seed)
    got = sampler.sample(B)
    assert_same(to_host(got), want, f'{case["name"]} debug={debug}')
    # the same draws once more through the native batch, for its launch count and dominant kernel
    np.random.seed(seed)
    draws, idxs = sampler._host_draws(B, None, False)
    return sampler._sampler.sample_native(B, idxs=idxs, draws=draws)


def philox_leg(case, fields, debug):
    """On-device draws: the batch equals the oracle fed the numpy restatement of the Philox draws."""
    from oracle import philox_np
    from oracle.replay_oracle import DrawsSource, OracleSampler
    from tests.test_gpu_philox import goal_sets_for

    B, config = case['B'], make_config(case)
    sampler = sampler_for(case, fields, seed=0x5EED, stream_id=5)
    sampler._sampler.set_debug(debug)
    oracle = OracleSampler(fields, config, case['kind'])
    handle = sampler._sampler.sample_native(B)
    got = to_host(sampler._sampler.wrap(handle))
    draws, knife = philox_np.philox_draws(0x5EED, 5, 0, B, len(oracle.valid_table), goal_sets_for(config, case['kind']), True, 0.0)
    want = oracle.sample(B, source=DrawsSource(draws))
    ok = ~knife
    assert ok.mean() > 0.9
    assert_same({k: v[ok] for k, v in got.items()}, {k: v[ok] for k, v in want.items()}, f'{case["name"]} philox debug={debug}')
    return handle


def index_vector(handle, slot, n):
    from ogbench_b200 import _native

    out = np.empty(n, dtype=np.int64)
    _native.check(_native.lib().ogb_batch_index_vector(handle.ptr, slot, out.ctypes.data_as(C.c_void_p)))
    return out


def check_rows_by_index(handle, got, plan, fields, total, what):
    """Every row key of the plan equals the host field at the rows its index vector names; next_observations is the
    observation at min(idx + 1, n - 1) (datasets.py:82), whether it comes from the record's shadow copy or a row gather."""
    flat = native_fields(fields)
    got = {k: np.asarray(v) for k, v in native_fields(got).items()}
    n_rows = len(fields['terminals'])
    vecs = {slot: index_vector(handle, slot, total) for slot in {k.slot for k in plan.keys} | {SLOT_IDX}}
    for k in plan.keys:
        rows = np.minimum(vecs[SLOT_IDX] + 1, n_rows - 1) if k.name.startswith('next_observations') else vecs[k.slot]
        want = flat[k.field.src][rows]
        assert np.array_equal(got[k.name].reshape(want.shape), want), (what, k.name)


# ------------------------------------------------ tests ------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('case', ORACLE_CASES, ids=[c['name'] for c in ORACLE_CASES])
def test_row_sizes_against_the_oracle(case):
    fields = make_fields(case)
    plan = plan_of(case, case_total(case), philox=False)
    handle = numpy_leg(case, fields, 0, case['seed'])
    check_path(handle, plan, case['name'])


@pytest.mark.gpu
@pytest.mark.parametrize('case', SPLIT_CASES, ids=[c['name'] for c in SPLIT_CASES])
def test_split_fused_launches_against_the_oracle(case):
    """Debug off (the fused launch stores the index vectors only because a later launch reads them) and static tiles
    (debug bit 3, which does not set bit 0), in both RNG modes where the oracle restates them."""
    fields = make_fields(case)
    plan = plan_of(case, case_total(case), philox=False)
    assert plan.fused and len(plan.launches) > 1 and plan.write_vecs_needed
    philox = case['kind'] in ('gc', 'hgc') and not case.get('leaves')
    for debug in (0, 8):
        if case.get('leaves'):
            # pytree observations: the oracle restates flat fields only; same draws through debug 1 and the index vectors
            sampler = sampler_for(case, fields, seed=9)
            ref = sampler_for(case, fields, seed=9)
            sampler._sampler.set_debug(debug)
            ref._sampler.set_debug(debug | 1)
            h, hr = sampler._sampler.sample_native(case['B']), ref._sampler.sample_native(case['B'])
            got, want = sampler._sampler.wrap(h), ref._sampler.wrap(hr)
            assert_same(to_host(native_fields(got)), to_host(native_fields(want)), f'{case["name"]} debug={debug}')
            check_rows_by_index(hr, want, plan_of(case, case['B']), fields, case['B'], case['name'])
            check_path(h, plan_of(case, case['B']), case['name'])
            continue
        handle = numpy_leg(case, fields, debug, case['seed'] + debug)
        check_path(handle, plan, case['name'])
        if philox:
            handle = philox_leg(case, fields, debug)
            check_path(handle, plan_of(case, case_total(case)), case['name'])


@pytest.mark.gpu
@pytest.mark.parametrize('case', BIG_CASES + SPLIT_CASES[:2], ids=[c['name'] for c in BIG_CASES + SPLIT_CASES[:2]])
def test_row_keys_by_index_vectors(case):
    """Large launches: a canary pass (debug 3) read against the host fields through the index vectors, with untouched
    gaps, and a debug-off pass of the same draws that must equal it byte for byte."""
    from ogbench_b200 import _native

    fields = make_fields(case)
    B, K = case['B'], case.get('K', 1)
    plan = plan_of(case, B * K)
    canary, plain = sampler_for(case, fields, seed=77), sampler_for(case, fields, seed=77)
    canary._sampler.set_debug(3)
    hc = canary._sampler.sample_native(B, n_batches=K)
    bad = C.c_int64(-1)
    _native.check(_native.lib().ogb_batch_check_gaps(hc.ptr, C.byref(bad)))
    assert bad.value == 0, case['name']
    want = canary._sampler.wrap(hc)
    check_rows_by_index(hc, want, plan, fields, B * K, case['name'])
    hp = plain._sampler.sample_native(B, n_batches=K)
    check_path(hp, plan, case['name'])
    assert_same(to_host(native_fields(plain._sampler.wrap(hp))), to_host(native_fields(want)), case['name'])


@pytest.mark.gpu
def test_host_chunks_equal_the_unchunked_batch():
    """ogb_sampler_set_host_chunks(4) with host output: the rows issued in four chunks equal one launch's."""
    from ogbench_b200 import _native

    case = BIG_CASES[0]
    fields = make_fields(case)
    B, K = case['B'], case.get('K', 1)
    assert plan_of(case, B * K, host_chunks=4).n_launches == 4
    one = sampler_for(case, fields, seed=3, output='numpy')
    four = sampler_for(case, fields, seed=3, output='numpy')
    _native.check(_native.lib().ogb_sampler_set_host_chunks(four._sampler.ptr, 4))
    h1, h4 = one._sampler.sample_native(B, n_batches=K), four._sampler.sample_native(B, n_batches=K)
    check_path(h1, plan_of(case, B * K), 'unchunked')
    check_path(h4, plan_of(case, B * K, host_chunks=4), 'four chunks')
    assert_same(to_host(four._sampler.wrap(h4)), to_host(one._sampler.wrap(h1)), 'host chunks')


@pytest.mark.gpu
def test_eight_leaf_pytree_samples():
    """Eight 100-float observation leaves (3.2 KB, all in the record) sample instead of being refused, and every leaf of
    every observation key is the host leaf at the rows its index vector names."""
    case = SPLIT_CASES[-1]
    fields = make_fields(case)
    sampler = sampler_for(case, fields, seed=4)
    sampler._sampler.set_debug(1)
    handle = sampler._sampler.sample_native(case['B'])
    batch = sampler._sampler.wrap(handle)
    assert sorted(batch['value_goals']) == [f'leaf_{i}' for i in range(8)]
    check_rows_by_index(handle, batch, plan_of(case, case['B']), fields, case['B'], case['name'])
    assert to_host(sampler.sample(7))['actions'].shape == (7, 4)


# ------------------------------------------------ switches ------------------------------------------------
# each forces, for every input, a path that some real inputs take anyway
SWITCHES = [{'OGB_GATHER': 'lsu'}, {'OGB_NO_RECORDS': '1'}, {'OGB_FUSE': '0'}, {'OGB_FUSE': '1'}, {'OGB_NO_TINY_GROUPS': '1'}]
# one split GC case, one C3-like HGC case (384-byte spans, un-fused at >= 32,768 rows), one LSU case
SWITCH_CASES = [SPLIT_CASES[0], C_('c3-like', 'hgc', ((96,), F32), 51, B=1024, K=33, traj=(300, 20, 300)), BIG_CASES[5]]

SWITCH_SCRIPT = r'''
import hashlib, json, sys
sys.path.insert(0, sys.argv[1])
import numpy as np
from tests.test_gpu_rows import SWITCH_CASES, batch_info, make_fields, native_fields, sampler_for, to_host
out = {}
for case in SWITCH_CASES:
    sampler = sampler_for(case, make_fields(case), seed=21)
    try:
        handle = sampler._sampler.sample_native(case['B'], n_batches=case.get('K', 1))
    except NotImplementedError as e:
        out[case['name']] = dict(refused=str(e))
        continue
    batch = to_host(native_fields(sampler._sampler.wrap(handle)))
    out[case['name']] = dict(launches=batch_info(handle)[0],
                             keys={k: hashlib.sha256(np.ascontiguousarray(v).tobytes()).hexdigest() + str(v.shape) + str(v.dtype)
                                   for k, v in batch.items()})
print(json.dumps(out))
'''


def run_switch(env):
    full = {k: v for k, v in os.environ.items() if not k.startswith('OGB_')}
    full.update(env)
    proc = subprocess.run([sys.executable, '-c', SWITCH_SCRIPT, ROOT], env=full, capture_output=True, text=True, timeout=600)
    assert proc.returncode == 0, (env, proc.stderr[-3000:])
    return json.loads(proc.stdout.strip().splitlines()[-1])


@pytest.mark.gpu
def test_measurement_switches_give_identical_batches():
    """Every switch (read once per process, so one process each) returns the default process's batches byte for byte,
    with the launch count the restated planner predicts for it."""
    default = run_switch({})
    for case in SWITCH_CASES:
        assert 'refused' not in default[case['name']], default[case['name']]
    for env in SWITCHES:
        got = run_switch(env)
        for case in SWITCH_CASES:
            plan = plan_of(case, case_total(case), env=env)
            name = case['name']
            assert 'refused' not in got[name], (env, name, got[name])
            assert got[name]['launches'] == plan.n_launches, (env, name, got[name]['launches'], plan.n_launches)
            assert got[name]['keys'] == default[name]['keys'], (env, name)


# ------------------------------------------------ no GPU ------------------------------------------------
def test_case_plan_reaches_every_path():
    """The device cases above cover what they are meant to: every drain kind, rows-per-item value, chunk walk, element
    width of the register-staged kernel, launch split and fused / un-fused HGC."""
    import time

    t0 = time.time()
    plans = {c['name']: plan_of(c, case_total(c), philox=False) for c in ALL_CASES}
    plans.update({c['name'] + '/philox': plan_of(c, case_total(c)) for c in ALL_CASES})
    drains = set().union(*(p.drains for p in plans.values()))
    assert drains == {DENSE16, WORDS, WORDS_UNALIGNED, ELEMS_U16, ELEMS_U8}, drains
    rpi = set().union(*(p.rows_per_item for p in plans.values()))
    assert {(32, None), (16, 4096), (16, 6144), (8, None), (4, None), (2, None), (1, None)} <= rpi, rpi
    walks = set().union(*(p.chunk_walks for p in plans.values()))
    assert walks == {'divides', 'does not divide', 'cpr>32'}, walks
    assert set().union(*(p.lsu_vecs for p in plans.values())) == {0, 1, 2, 3, 4}
    for name in ('split-items-gc', 'split-items-hgc', 'split-items-trl', 'split-outputs', 'split-jobs', 'pytree-8x100',
                 'big-split-gc', 'big-split-outputs', 'big-pytree-8x100'):
        assert plans[name].fused and len(plans[name].launches) > 1 and plans[name].write_vecs_needed, name
    assert plans['split-items-gc'].split_reasons == {'items'} and plans['split-items-gc'].n_launches == 2
    assert plans['split-items-hgc'].split_reasons == {'items'}
    assert plans['split-outputs'].split_reasons == {'outputs'}
    assert plans['split-jobs'].split_reasons == {'jobs'}
    assert not plans['big-hgc-unfused'].fused and not plans['big-hgc-unfused-nodedup'].fused and plans['hgc-fused'].fused
    assert plans['big-gc-fused/philox'].launches[0]['shape'] == 220 and plans['split-items-gc/philox'].launches[0]['shape'] == 220
    # every compiled gather shape is planned by some case: 2 x 16 for a fused GCDataset launch of 6 KB stages, 3 x 10 for an
    # un-fused gather of 6 KB stages
    assert {la['shape'] for p in plans.values() for la in p.launches} == {220, 216, 308, 310}
    # tiny observations drained inside the span of the transition's record
    for name in ('obs1-u8', 'obs6-u8', 'obs12-f32'):
        p = plans[name]
        span_obs = [k for s in p.spans for k, _ in s.outs if k.name == 'observations']
        assert span_obs and span_obs[0].field.row <= 16, name
    # rows in arrays of their own at 2,048 / 2,064 bytes, exactly 4,096 on the cp.async path, LSU beyond
    own = {k.field.row for p in plans.values() for s in p.spans for k, _ in s.outs if not k.field.in_record}
    assert {2048, 2064, 3072, 3088, 4096} <= own, own
    assert {k.field.row for k in plans['lsu'].lsu} == {4097, 4098, 4100, 4104, 4112}
    # the eight-leaf pytree: no observation span holds all eight leaves any more
    assert all(len(s.outs) < 8 for s in plans['pytree-8x100'].spans if s.slot != SLOT_IDX)
    # no case, by default or under any switch, plans a launch over the shared-memory limit (that refusal is internal)
    refused = [name for name, p in plans.items() if p.refused_smem]
    for c in ALL_CASES + SWITCH_CASES:
        fields, config = make_fields(c), make_config(c)
        refused += [(c['name'], tuple(env.items())) for env in SWITCHES
                    if RowPlan(fields, c['kind'], config, case_total(c), c.get('dedup', True), env).refused_smem]
    assert not refused, refused
    assert time.time() - t0 < 10

