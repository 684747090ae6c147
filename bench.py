#!/usr/bin/env python
"""bench.py — ops/sec applied for automerge-classic's Backend.applyChanges path on B200.

  python bench.py --gpus N --steps K --warmup W            (N>1: launched under torchrun, one rank per GPU)
  python bench.py --impl reference --gpus N --steps K --warmup W
  python bench.py ... --dump-outputs DIR   (also writes the patch of the last timed step as DIR/*.npy: patch_arrays)

Workload (BASELINE.json `metric`: "ops/sec applied (1M-op text trace)"; SURVEY.md §8d C3): a makeText
change plus 10 actors x 100 000 single-op changes (70 % insert / 30 % delete, merge every 100 changes)
= 1 000 001 binary changes, ~132 MB, synthetic (seeded generator csrc/tracegen.cc). One *step* =
Backend.applyChanges(init(), all changes) -> incremental patch, on a document that is reset (not
re-allocated) between steps. With N GPUs every rank replays its own independent document (seed + rank,
config C5): no data-path collective, weak scaling; the time of a step is the max over ranks.

  value : ops/s with the change bytes already resident in HBM: the same C-ABI call is handed a DEVICE pointer; time =
          CUDA events on the engine's stream from the first to the last kernel of the call (device->device copy into the
          document's arena, SHA-256, decode, gate, op-set ordering, patch kernels, patch copy-out to pinned host memory)
  e2e   : ops/s through the C ABI (amg_apply_changes_packed) from a pinned HOST buffer to the flat patch in
          host memory, host<->device copies inside the timed region (wall clock around the synchronous call); the upload
          goes in 16 MB pieces and every piece is hashed and decoded while the next one is still crossing PCIe
  e2e_ptr_array: the same through amg_apply_changes with one pageable buffer per change (pointer array), the shape
          Backend.applyChanges(state, Uint8Array[]) has in the reference
  roofline: the column decode kernel (header parse + column expansion fused) re-run on resident data: algorithmic bytes
          of SURVEY.md §8d (encoded bytes + 48 B/op + 8 B/pred + 96 B/change) / CUDA-event time against the measured
          HBM peak; the SHA-256 kernel over the same bytes is ALU-bound and stated next to it (`sha256_kernel`,
          `with_sha256_frac` = both together)
  --workload C3|C4|C2|C2b: the configs of SURVEY.md §8d (C3 = headline); the default run also reports C4 / C2 / C2b
          briefly under config.other_workloads
  cpu_baseline: the oracle (CPU restatement of the reference's algorithm, 1 core) on a bounded prefix
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
if os.environ.get('NCCL_DEBUG', '').upper() in ('', 'VERSION'):
    os.environ['NCCL_DEBUG'] = 'WARN'   # keep stdout to the one JSON line (NCCL prints its version banner there)
# stdout carries exactly one JSON line: whatever native libraries print to file descriptor 1 (NCCL's version banner does,
# whatever NCCL_DEBUG says) goes to stderr instead; the JSON line is written through the saved descriptor
_JSON_OUT = os.fdopen(os.dup(1), 'w')
os.dup2(2, 1)


def _emit(line):
    print(line, file=_JSON_OUT, flush=True)


N_OPS, N_ACTORS = 1_000_000, 10
CPU_SAMPLE_OPS = 200_000
# bounded CPU samples (about 10-30 s of oracle time each): the oracle, like the reference, is super-linear in document length
# (C4: 50k ops 43 s, 100k ops 172 s), so the sample is a prefix and the ops/s it yields flatters the CPU side
CPU_SAMPLE = {'C3': 200_000, 'C4': 30_000, 'C2': 100_000, 'C2b': 100_000}


def read_traffic():
    """DRAM bytes per launch of the decode kernels from the committed ncu capture (None if the file is missing)."""
    try:
        with open(os.path.join(ROOT, 'profiles', 'traffic_r02.json')) as fh:
            return int(json.load(fh)['decode_total_bytes']), 'profiles/traffic_r02.json (ncu --set full of k_decode_tiles, dram__bytes_read.sum + dram__bytes_write.sum, see profiles/README_r02.md)'
    except Exception:
        return None, None


def read_peaks():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as fh:
            return float(json.load(fh)['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    except Exception:
        return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


class ClockSampler:
    """One `nvidia-smi -lms 50` process for the length of the measurement (a fresh nvidia-smi per sample takes longer to
    start than a timed region of ten 8 ms steps lasts)."""

    def __init__(self, index):
        q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
        self.samples, self.marks = [], []
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(index), '--query-gpu=' + q, '--format=csv,noheader,nounits', '-lms', '50'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            parts = [x.strip() for x in line.strip().split(',')]
            if parts and parts[0].isdigit():
                self.samples.append((time.perf_counter(), parts))

    def start(self):
        pass

    def mark(self):
        """start / end of a timed region"""
        self.marks.append(time.perf_counter())

    def stop(self):
        if self.proc:
            time.sleep(0.15)   # one more sample after the last timed step
            self.proc.terminate()
    stop_flag = property(lambda self: False, lambda self, v: self.stop() if v else None)

    def summary(self):
        lo, hi = (self.marks[0], self.marks[-1]) if len(self.marks) >= 2 else (0, float('inf'))
        inside = [p for t, p in self.samples if lo - 0.11 <= t <= hi + 0.16] or [p for _, p in self.samples]
        sm = sorted(int(p[0]) for p in inside)
        reasons = set()
        for p in inside:
            for name, v in zip(['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'], p[2:6]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        mx = [int(p[1]) for p in inside if len(p) > 1 and p[1].isdigit()]
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None, 'reasons': sorted(reasons), 'samples': len(sm),
                'how': 'nvidia-smi -lms 50 running from before the warm-up to after the last timed step; samples inside (or within 0.1 s of) the timed regions'}


def run_reference(args, rank, world):
    """The reference arm: the CPU restatement of the reference backend (oracle/, pinned on the reference's own
    tests) on the host cores. The reference is single-threaded JavaScript; the restatement is single-threaded."""
    if rank != 0:
        return
    import numpy as np
    import oracle
    from automerge_classic_b200 import tracegen
    oracle.build()
    cfg, ops, actors, desc = WORKLOADS[getattr(args, 'workload', 'C3')]
    t = tracegen.generate(cfg, min(CPU_SAMPLE[getattr(args, 'workload', 'C3')], ops), actors)
    times = []
    for i in range(args.warmup + args.steps):
        doc = oracle.OracleDoc()
        t0 = time.perf_counter()
        doc.apply_blob(t.blob.ctypes.data_as(C.c_void_p), t.offsets.ctypes.data_as(C.c_void_p), t.n_changes, want_patch=False)
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            times.append(dt)
    ms = 1e3 * sum(times) / len(times)
    v = t.n_ops / (ms / 1e3)
    sample = 'first %d ops of the %s trace (same generator), applyChanges(init(), all) on 1 core: a PREFIX of the workload (the reference is super-linear in document length), C++ restatement of backend/new.js, not V8' % (t.n_ops, cfg)
    _emit(json.dumps({
        'impl': 'reference', 'metric': 'ops/sec applied (1M-op text trace)' if cfg == 'C3' else 'ops/sec applied (%s)' % cfg, 'value': v, 'unit': 'ops/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'int64', 'data': 'synthetic',
        'config': {'workload': desc + '; reference arm: bounded prefix', 'sample_ops': t.n_ops},
        'cpu_baseline': {'value': v, 'unit': 'ops/s', 'cores': 1, 'kind': 'port', 'sample': sample},
        'e2e': {'value': v, 'unit': 'ops/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}))


WORKLOADS = {
    # name: (trace config, ops, actors, description) — SURVEY.md 8d; C3 is the headline (BASELINE.json configs[2] / metric)
    'C3': ('C3', 1_000_000, 10, 'C3 text trace: makeText + 10 actors x 100k single-op changes, 70% insert / 30% delete (SURVEY.md 8d); one independent document per GPU (C5)'),
    'C4': ('C4', 1_000_000, 100, 'C4 nested maps: 100 actors, 10 000 keys (100 child maps x 100 keys), 10 000 changes x 100 set ops, Zipf keys, same-round writers conflict (SURVEY.md 8d)'),
    'C2': ('C2', 100_000, 1, 'C2 text trace: makeText + 100k single-op insert changes, one actor (SURVEY.md 8d)'),
    'C2b': ('C2b', 100_000, 1, 'C2b: the 100k inserts of C2 in ONE change (bulk decode)'),
}


def bind_to_gpu_numa_node(local):
    """Pins this process (and the pinned buffers it allocates from here on: first touch) to the CPUs of the NUMA node the
    GPU hangs off. Eight ranks staging 130 MB each through one node's memory was what bent the 8-GPU end-to-end curve."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local).pci_bus_id
        dom = torch.cuda.get_device_properties(local).pci_domain_id
        dev = torch.cuda.get_device_properties(local).pci_device_id
        path = '/sys/bus/pci/devices/%04x:%02x:%02x.0/' % (dom, bus, dev)
        node = int(open(path + 'numa_node').read())
        if node < 0:
            return None
        cpus = []
        for part in open('/sys/devices/system/node/node%d/cpulist' % node).read().strip().split(','):
            lo, _, hi = part.partition('-')
            cpus += list(range(int(lo), int(hi or lo) + 1))
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


def measure(args, wl_name, rank, world, local, lib, torch, dist, full, keep_patch=False):
    """K timed steps of one workload. Returns the pieces of the JSON line (with keep_patch, also the bytes of the flat
    patch the last timed step returned)."""
    import numpy as np
    from automerge_classic_b200 import tracegen
    from automerge_classic_b200.engine import GpuBackendDoc, _ErrStruct
    L = lib.L
    cfg, ops, actors, desc = WORKLOADS[wl_name]
    if wl_name == 'C3':
        ops = args.ops
    trace = tracegen.generate(cfg, ops, actors, seed=tracegen.SEED + rank)
    nbytes = int(trace.offsets[-1])
    # the caller's buffers: pinned host memory (e2e: copied to the device inside the timed region, every step) and a
    # device-resident copy of the same bytes (value: inputs already in HBM when the timed region starts)
    pinned = torch.empty(nbytes + 64, dtype=torch.uint8).pin_memory()
    pinned[:nbytes].copy_(torch.from_numpy(trace.blob))
    resident = pinned.to('cuda:%d' % local)
    offs = np.ascontiguousarray(trace.offsets)
    offs_pinned = torch.from_numpy(offs.astype(np.int64)).pin_memory()   # the offsets array travels by DMA as well (pinned like the bytes)
    offs_p = C.c_void_p(offs_pinned.data_ptr())
    doc = GpuBackendDoc(device=local)
    err = _ErrStruct()
    L.amg_reserve(doc.h, C.c_size_t(nbytes + (1 << 20)), C.byref(err))
    state = {}

    def step(ptr, keep=False):
        lib.check(L.amg_reset(doc.h, C.byref(err)), err)
        pp = C.c_void_p()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rc = L.amg_apply_changes_packed(doc.h, C.c_void_p(ptr), offs_p, C.c_size_t(trace.n_changes), 0, 1, C.byref(pp), C.byref(err))
        state['call_ms'] = (time.perf_counter() - t0) * 1e3
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        lib.check(rc, err)
        n = C.c_size_t()
        p = L.amg_patch_bytes(pp, C.byref(n))
        if keep:
            state['patch'] = bytes((C.c_uint8 * n.value).from_address(p))
        L.amg_patch_free(pp)
        return dt, doc.timings(), n.value

    def timed(ptr, steps, keep_last=False):
        wall, dev, ph, pb = [], [], None, 0
        for i in range(steps):
            dt, ph, pb = step(ptr, keep_last and i == steps - 1)
            wall.append(dt)
            dev.append(sum(ph[0:12]) / 1e3)   # CUDA events on the engine's stream, first to last kernel of the call
        return wall, dev, ph, pb

    sampler = ClockSampler(local)
    for _ in range(args.warmup):
        step(resident.data_ptr())
        step(pinned.data_ptr())
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.mark()
    # value: K steps on the device-resident bytes (the call copies them device -> device into the document's arena: that
    # copy, SHA-256, decode, gate, op-set ordering, patch kernels and the patch copy-out are all inside the figure)
    _, dev_res, ph_res, _ = timed(resident.data_ptr(), args.steps)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    launches0 = doc.launches()
    wall, dev_e2e, last_ph, patch_bytes = timed(pinned.data_ptr(), args.steps, keep_last=keep_patch)
    torch.cuda.synchronize()
    sampler.mark()
    if world > 1:
        dist.barrier()
    sampler.stop()
    launches = (doc.launches() - launches0) // max(args.steps, 1)
    t_wall, t_dev = sum(wall) / len(wall), sum(dev_res) / len(dev_res)
    if world > 1:   # a step ends when the slowest rank is done
        tt = torch.tensor([t_wall, t_dev], dtype=torch.float64, device='cuda')
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t_wall, t_dev = float(tt[0]), float(tt[1])
    res = {'trace': trace, 'nbytes': nbytes, 'desc': desc, 't_wall': t_wall, 't_dev': t_dev, 'wall_steps': wall, 'dev_steps': dev_res, 'last_ph': last_ph, 'ph_res': ph_res,
           'patch_bytes': patch_bytes, 'launches': int(launches), 'call_ms': state['call_ms'], 'clocks': sampler.summary(), 'doc': doc, 'pinned': pinned, 'offs': offs, 'offs_pinned': offs_pinned,
           'patch': state.get('patch')}
    if not full:
        del doc
    return res


def ptr_array_e2e(trace, lib, torch, local, steps):
    """The shape Backend.applyChanges(state, Uint8Array[]) produces: n separate, pageable buffers through
    amg_apply_changes (one pointer and one length per change), host copies inside the timed region."""
    from automerge_classic_b200.engine import GpuBackendDoc, _ErrStruct
    L = lib.L
    changes = trace.changes()                                   # n separate bytes objects
    n = len(changes)
    bufs = (C.c_char_p * n)(*changes)
    lens = (C.c_size_t * n)(*[len(c) for c in changes])
    doc, err = GpuBackendDoc(device=local), _ErrStruct()
    L.amg_reserve(doc.h, C.c_size_t(int(trace.offsets[-1]) + (1 << 20)), C.byref(err))
    times = []
    for i in range(steps + 2):
        lib.check(L.amg_reset(doc.h, C.byref(err)), err)
        pp = C.c_void_p()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rc = L.amg_apply_changes(doc.h, bufs, lens, C.c_size_t(n), 0, 1, C.byref(pp), C.byref(err))
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        lib.check(rc, err)
        L.amg_patch_free(pp)
        if i >= 2:
            times.append(dt)
    return sum(times) / len(times)


DUMP_BUDGET = 64_000_000   # bytes --dump-outputs writes at most
DUMP_SEED = 20261017


def _gather(buf, off, length):
    """buf[off[i]:off[i] + length[i]] of every row, back to back."""
    length = length.astype(np.int64)
    idx = np.repeat(off.astype(np.int64) - (np.cumsum(length) - length), length) + np.arange(int(length.sum()))
    return buf[idx]


def _split_ids(name, ids):
    """opIds are (counter << 16 | actor index): two columns, each exact in float64."""
    ids = ids.astype(np.uint64)
    return {name + '_ctr': ids >> np.uint64(16), name + '_actor': ids & np.uint64(0xffff)}


def patch_arrays(raw, budget=DUMP_BUDGET, seed=DUMP_SEED):
    """The flat patch of include/amgpu.h (what amg_apply_changes_packed hands its caller) as named float64 / float32 arrays:
    the header counts, actor table, clock, heads, and the map-property and list-edit records column by column. Payload
    bytes (keys, values) are gathered per record instead of their offsets in the patch buffer, so that two builds that
    compute the same patch dump the same arrays however they lay the buffer out. When the records would take more than
    `budget` bytes, a fixed seeded sample of them is kept, in order; their record numbers are the `*_row` arrays."""
    from automerge_classic_b200.engine import FlatPatch
    fp = FlatPatch(raw)
    h = fp.hdr
    buf = np.frombuffer(raw, dtype=np.uint8)
    out = {'header': np.array([fp.max_op, fp.pending, int(h[3]), int(h[4]), int(h[8]), int(h[10]), int(h[12]), int(h[14]), int(h[16])], dtype=np.float64)}
    ids = [bytes.fromhex(a) for a in fp.actors]
    actors = np.full((len(ids), max([len(a) for a in ids] + [0])), -1.0)
    for i, a in enumerate(ids):
        actors[i, :len(a)] = np.frombuffer(a, dtype=np.uint8)
    out['actors'] = actors
    out['clock'] = np.frombuffer(raw, dtype='<u8', count=2 * int(h[10]), offset=int(h[9])).reshape(-1, 2).astype(np.float64)
    out['deps'] = buf[int(h[11]):int(h[11]) + 32 * int(h[12])].reshape(-1, 32).astype(np.float64)

    p, e = fp.props, fp.edits
    p_action, p_flags = p['flags'] >> 8, p['flags']
    p_counter = (p_action == 1) & (p_flags & 2 != 0)
    p_vlen = np.where((p_action == 1) & (p_flags & 3 == 0), p['valLen'] >> 4, 0)
    props = {**_split_ids('obj', p['obj']), **_split_ids('op', p['opId']), 'key_len': p['keyLen'], 'flags': p_flags, 'val_len': p['valLen'],
             'counter': np.where(p_counter, (p['valOff'].astype(np.uint64) | (p['pad'].astype(np.uint64) << np.uint64(32))).view(np.int64), 0)}
    e_kind = e['kind']
    e_counter = e_kind & 0x1000 != 0
    e_vlen = np.where((e_kind & 0xff != 1) & (e_kind >> 16 == 1) & ~e_counter, e['valLen'] >> 4, 0)
    edits = {**_split_ids('obj', e['obj']), **_split_ids('op', e['opId']), **_split_ids('elem', fp.edit_elem), 'index': e['index'], 'kind': e_kind,
             'val_len': e['valLen'], 'counter': np.where(e_counter, (e['valLen'].astype(np.uint64) | (e['valOff'].astype(np.uint64) << np.uint64(32))).view(np.int64), 0)}
    # payload bytes go out as float32 (4 bytes each), record columns as float64 (8 bytes each, plus the record number)
    tables = [('props', props, [('key', p['keyOff'], p['keyLen']), ('value', p['valOff'], p_vlen)]),
              ('edits', edits, [('value', e['valOff'], e_vlen)])]
    cost = [8 * (len(cols) + 1) + 4 * sum(ln.astype(np.int64) for _, _, ln in pays) for _, cols, pays in tables]
    room = budget - sum(a.nbytes for a in out.values()) - 128 * (len(out) + sum(len(c) + 1 + len(pl) for _, c, pl in tables))
    rng = np.random.default_rng(seed)
    # the smaller table first: it keeps every record if it fits its half of the room, the other table gets the rest
    for left, k in enumerate(sorted(range(len(tables)), key=lambda k: int(cost[k].sum()))):
        (name, cols, pays), c = tables[k], cost[k]
        rows = np.arange(len(c))
        if int(c.sum()) > room // (len(tables) - left):
            order = rng.permutation(len(c))
            rows = np.sort(order[:np.searchsorted(np.cumsum(c[order]), room // (len(tables) - left), side='right')])
        room -= int(c[rows].sum())
        out[name + '_row'] = rows.astype(np.float64)
        for col, v in cols.items():
            out['%s_%s' % (name, col)] = np.asarray(v)[rows].astype(np.float64)
        for pay, off, ln in pays:
            out['%s_%s_bytes' % (name, pay)] = _gather(buf, off[rows], ln[rows]).astype(np.float32)
    return out


def dump_outputs(raw, out_dir):
    """Writes the arrays of patch_arrays that have elements (a workload without list edits, or a patch whose map entries
    carry no value bytes, has nothing to compare there)."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in patch_arrays(raw).items():
        if a.size:
            np.save(os.path.join(out_dir, name + '.npy'), a)


def cpu_sample(wl_name, sample_ops):
    import oracle
    from automerge_classic_b200 import tracegen
    oracle.build()
    cfg, ops, actors, _ = WORKLOADS[wl_name]
    ts = tracegen.generate(cfg, min(sample_ops, ops), actors)
    od = oracle.OracleDoc()
    t0 = time.perf_counter()
    od.apply_blob(ts.blob.ctypes.data_as(C.c_void_p), ts.offsets.ctypes.data_as(C.c_void_p), ts.n_changes, want_patch=False)
    dt = time.perf_counter() - t0
    return {'value': ts.n_ops / dt, 'unit': 'ops/s', 'cores': 1, 'kind': 'port',
            'sample': 'first %d ops of the same %s workload (a prefix: the reference is super-linear in document length), oracle restatement of backend/new.js (C++, not V8), 1 core, %.1f s' % (ts.n_ops, wl_name, dt)}


def main():
    import faulthandler
    # a hung native call must not eat the GPU budget silently: after this many seconds the Python stacks go to stderr and the
    # process exits
    faulthandler.dump_traceback_later(int(os.environ.get('AMG_BENCH_WATCHDOG_S', '900')), exit=True)
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='amgpu')
    ap.add_argument('--ops', type=int, default=N_OPS)
    ap.add_argument('--workload', default='C3', choices=sorted(WORKLOADS))
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-extras', action='store_true', help='headline figures only (no other routes / workloads / pointer-array entry)')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the patch the last timed step returned as DIR/<name>.npy (see patch_arrays; '
                                                         'at most 64 MB, a fixed seeded sample of the records if the patch is larger)')
    args = ap.parse_args()
    rank, world, local = int(os.environ.get('RANK', 0)), int(os.environ.get('WORLD_SIZE', 1)), int(os.environ.get('LOCAL_RANK', 0))
    if args.impl == 'reference':
        return run_reference(args, rank, world)

    import numpy as np
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device — the engine has no CPU fallback')
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa_node(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    from automerge_classic_b200 import build
    if rank == 0:
        build.build_all()
    if world > 1:
        dist.barrier()
    from automerge_classic_b200.engine import GpuBackendDoc, default_library, _ErrStruct
    lib = default_library()
    L = lib.L
    err = _ErrStruct()

    m = measure(args, args.workload, rank, world, local, lib, torch, dist, full=True, keep_patch=bool(args.dump_outputs))
    if rank == 0 and args.dump_outputs:
        dump_outputs(m['patch'], args.dump_outputs)
    trace, doc, nbytes = m['trace'], m['doc'], m['nbytes']
    t_wall, t_dev, last_ph = m['t_wall'], m['t_dev'], m['last_ph']
    total_ops = trace.n_ops * world
    blob_ptr, offs = C.c_void_p(m['pinned'].data_ptr()), m['offs']
    extras = rank == 0 and not args.no_extras

    # decode roofline: re-run the decode kernels on the resident batch
    roofline = None
    if rank == 0:
        ms_sha, ms_parse, ms_dec, algo = C.c_float(), C.c_float(), C.c_float(), C.c_uint64()
        rc = L.amg_bench_decode(doc.h, 20, C.byref(ms_sha), C.byref(ms_parse), C.byref(ms_dec), C.byref(algo), C.byref(err))
        peak, peak_src = read_peaks()
        traffic, traffic_src = read_traffic()
        if rc == 0:
            # the HBM-bound part of the decode: header parse + column expansion (one fused kernel). SHA-256 over the same
            # bytes is ALU-bound (64 rounds per 64-byte block) and is reported next to it, not folded into the HBM figure.
            t_dec = (ms_parse.value + ms_dec.value) / 1e3
            kernel_name = 'column decode = k_decode_tiles (fused header parse + column expansion, bulk-staged through shared memory; one launch over the batch, one over the inflated changes) + k_decode_direct (changes outside their tile, totals) + DecodeColumnKernel (changes of more than 16 ops)'
            ach = algo.value / t_dec / 1e9
            n_blocks = (trace.blob.size + 64 * trace.n_changes) / 64.0          # ~ message blocks incl. padding
            roofline = {'bound': 'hbm', 'kernel': kernel_name,
                        'achieved': ach, 'peak': peak, 'unit': 'GB/s', 'frac': ach / peak, 'traffic': traffic, 'traffic_source': traffic_src, 'peak_source': peak_src,
                        'algorithmic_bytes_per_launch': int(algo.value),
                        'ms': {'decode_tiles': ms_parse.value, 'decode_large_changes': ms_dec.value},
                        'sha256_kernel': {'bound': 'alu', 'ms': ms_sha.value, 'bytes_hashed': int(trace.blob.size),
                                          'gb_per_s': trace.blob.size / (ms_sha.value / 1e3) / 1e9 if ms_sha.value else None,
                                          'blocks_per_s': n_blocks / (ms_sha.value / 1e3) if ms_sha.value else None},
                        'with_sha256_gbs': algo.value / ((ms_sha.value + ms_parse.value + ms_dec.value) / 1e3) / 1e9,
                        'with_sha256_frac': algo.value / ((ms_sha.value + ms_parse.value + ms_dec.value) / 1e3) / 1e9 / peak}
        else:
            roofline = {'bound': 'hbm', 'achieved': None, 'peak': peak, 'unit': 'GB/s', 'frac': None, 'traffic': None, 'error': err.msg.decode()}

    # the other routes of SURVEY §8d, once each on rank 0 (wall clock through the C ABI): (ii) loadChanges + getPatch,
    # (iii) save, then load + getPatch of the saved document
    other = None
    if extras:
        try:
            def wall(fn):
                torch.cuda.synchronize(); t0 = time.perf_counter(); r = fn(); torch.cuda.synchronize(); return r, time.perf_counter() - t0
            lib.check(L.amg_reset(doc.h, C.byref(err)), err)
            _, t_lc = wall(lambda: doc.apply_packed_flat(blob_ptr, offs, trace.n_changes, want_patch=False))
            _, t_gp = wall(doc.get_patch_flat)
            _, t_gpw = wall(doc.get_patch_flat)
            saved, t_sv = wall(doc.save)
            d2, t_ld = wall(lambda: GpuBackendDoc(saved, device=local))
            _, t_gp2 = wall(d2.get_patch_flat)
            del d2
            other = {'loadChanges_plus_getPatch_ops_per_s': trace.n_ops / (t_lc + t_gp), 'loadChanges_ms': t_lc * 1e3, 'getPatch_ms': t_gp * 1e3, 'getPatch_warm_ms': t_gpw * 1e3,
                     'save_ms': t_sv * 1e3, 'saved_document_bytes': len(saved),
                     'load_plus_getPatch_ops_per_s': trace.n_ops / (t_ld + t_gp2), 'load_ms': t_ld * 1e3, 'getPatch_after_load_ms': t_gp2 * 1e3,
                     'note': 'single invocation each, host buffers in and out'}
        except Exception as e:   # never lose the headline line over the extras
            other = {'error': repr(e)[:200]}
    e2e_ptr = None
    if extras:
        try:
            t_ptr = ptr_array_e2e(trace, lib, torch, local, min(args.steps, 3))
            e2e_ptr = {'value': trace.n_ops / t_ptr, 'unit': 'ops/s', 'ms_per_step': t_ptr * 1e3,
                       'entry': 'amg_apply_changes: %d separate pageable buffers (pointer + length each), what Backend.applyChanges(state, Uint8Array[]) hands to the addon' % trace.n_changes}
        except Exception as e:
            e2e_ptr = {'error': repr(e)[:200]}
    del doc
    others = None
    if extras and args.workload == 'C3' and world == 1:
        others = {}
        short = argparse.Namespace(**vars(args)); short.steps = min(args.steps, 3); short.warmup = 3
        for name in ('C4', 'C2', 'C2b'):
            try:
                r = measure(short, name, rank, world, local, lib, torch, dist, full=False)
                others[name] = {'value': r['trace'].n_ops / r['t_dev'], 'e2e': r['trace'].n_ops / r['t_wall'], 'unit': 'ops/s', 'ops': r['trace'].n_ops, 'changes': r['trace'].n_changes,
                                'change_bytes': r['nbytes'], 'device_ms_per_step': r['t_dev'] * 1e3, 'wall_ms_per_step': r['t_wall'] * 1e3, 'gpu_launches': r['launches'], 'workload': r['desc']}
            except Exception as e:
                others[name] = {'error': repr(e)[:200]}

    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        cpu = cpu_sample(args.workload, CPU_SAMPLE[args.workload])

    if rank == 0 and os.environ.get('AMG_BENCH_MARKS'):
        buf = C.create_string_buffer(4096)
        print('marks: (see amg_debug_marks)', file=sys.stderr)
    if rank == 0:
        names = ['upload_hash_decode', 'inflate_finish_decode', 'gate', 'actors_finalize', 'opset', 'patch_groups_props', 'patch_list_index', 'patch_edits_copyout', 'heads_commit']
        _emit(json.dumps({
            'metric': 'ops/sec applied (1M-op text trace)' if args.workload == 'C3' else 'ops/sec applied (%s)' % args.workload, 'value': total_ops / t_dev, 'unit': 'ops/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': t_wall * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'int64', 'data': 'synthetic',
            'config': {'workload': m['desc'],
                       'ops_per_gpu': trace.n_ops, 'changes_per_gpu': trace.n_changes, 'change_bytes_per_gpu': nbytes, 'parallelism': 'replicas x%d' % world, 'numa_node': numa,
                       'l2': 'inputs (%.0f MB) + working tables exceed the 126 MB L2; document reset every step' % (nbytes / 1e6),
                       'value_definition': 'change bytes resident in HBM (device pointer handed to amg_apply_changes_packed); CUDA events on the engine stream from the first to the last kernel of the call, patch copied to pinned host memory',
                       'e2e_definition': 'same call with the bytes in pinned HOST memory: wall clock around the synchronous call, H2D upload and patch D2H inside',
                       'device_ms_per_step': t_dev * 1e3, 'wall_ms_steps': [round(x * 1e3, 3) for x in m['wall_steps']], 'call_return_ms_last_step': round(m['call_ms'], 3), 'abi_call_ms_last_step': round(last_ph[23], 3), 'device_ms_steps': [round(x * 1e3, 3) for x in m['dev_steps']],
                       'phase_ms_last_step_e2e': dict(zip(names, [round(x, 3) for x in last_ph[:9]])),
                       'phase_ms_last_step_resident': dict(zip(names, [round(x, 3) for x in m['ph_res'][:9]])),
                       'host_marks_ms': [round(x, 3) for x in last_ph[12:22]], 'other_paths': other, 'other_workloads': others},
            'e2e': {'value': total_ops / t_wall, 'unit': 'ops/s', 'h2d_bytes_per_step': nbytes + 8 * (trace.n_changes + 1), 'd2h_bytes_per_step': m['patch_bytes']},
            'e2e_ptr_array': e2e_ptr,
            'gpu_launches': m['launches'], 'roofline': roofline, 'cpu_baseline': cpu, 'clocks': m['clocks']}))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
