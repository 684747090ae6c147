"""Host-logic tests of the replay pipeline WITHOUT a GPU: the engine's kernel functors are compiled
with -DAMG_EMU (tests/_emu/build.sh) and executed as serial loops, so the orchestration in
csrc/engine_impl.cuh and the per-item kernel logic can be checked against the oracle in this
GPU-less build container. This is a development aid: the emulation library is never loaded by the
product package, and none of these tests stands in for the `-m gpu` parity tests, which run the
nvcc-built kernels through libamgpu.so on a B200.
"""
import os
import subprocess

import pytest

import parity_checks
import replay
from automerge_classic_b200.backend import RangeError as FacadeRangeError

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope='module')
def emu_doc():
    subprocess.check_call([os.path.join(HERE, '_emu', 'build.sh')])
    from automerge_classic_b200 import build
    build.build_tracegen()
    from automerge_classic_b200.engine import doc_class_for
    return doc_class_for(os.path.join(HERE, '_emu', 'libamgpu_emu.so'))


def _all_cases():
    out = []
    for f in ('new_backend_test.json', 'backend_test.json'):
        out += [pytest.param(t, id=t['name'][-70:]) for t in replay.load(f) if 'skipped' not in t]
    return out


@pytest.mark.parametrize('test', _all_cases())
def test_reference_fixture_emu(emu_doc, test):
    from automerge_classic_b200.engine import AmgError
    r = replay.Replayer(emu_doc, (AmgError, ValueError, TypeError, RuntimeError, FacadeRangeError), structural=False)
    fails = r.run_test(test)
    assert not fails, '\n'.join(fails[:5])


@pytest.mark.parametrize('cfg,n,a', [('C1', 0, 0), ('C2', 400, 0), ('C2b', 700, 0), ('C2b', 6000, 0), ('C3', 3000, 10), ('C3', 900, 3), ('C4', 2000, 4), ('C4', 10000, 100)])
def test_trace_parity_emu(emu_doc, oracle_mod, cfg, n, a):
    parity_checks.check_trace_parity(emu_doc, oracle_mod, cfg, n, a)


@pytest.mark.parametrize('n,a,chunk', [(60, 2, 1000), (300, 3, 7), (400, 4, 50), (200, 1, 3), (450, 5, 1)])
def test_rich_list_emu(emu_doc, oracle_mod, n, a, chunk):
    compared = sum(parity_checks.check_rich_list(emu_doc, oracle_mod, seed, n, a, chunk) for seed in range(1, 7))
    assert compared >= 4


@pytest.mark.parametrize('cfg,n,a', [('C1', 0, 0), ('C2', 300, 0), ('C2b', 500, 0), ('C3', 1500, 5), ('C4', 1200, 4), ('C6', 300, 3), ('C7', 300, 3)])
def test_decoded_rows_emu(emu_doc, oracle_mod, cfg, n, a):
    assert parity_checks.check_decoded_rows_trace(emu_doc, oracle_mod, cfg, n, a) > 0


@pytest.mark.parametrize('seed', [11, 10, 3, 101, 7])
def test_decoded_rows_corrupted_emu(emu_doc, oracle_mod, seed):
    parity_checks.check_decode_corrupted(emu_doc, oracle_mod, seed=seed, cases=200)   # seed 10: an unknown GROUP_CARD column in the key group


def test_utf16_key_order_emu(emu_doc, oracle_mod):
    parity_checks.check_utf16_keys(emu_doc, oracle_mod)


def test_deflate_variants_emu(emu_doc, oracle_mod):
    parity_checks.check_deflate_variants(emu_doc, oracle_mod)


@pytest.mark.parametrize('n,a,chunk', [(80, 2, 1000), (300, 3, 5), (500, 4, 40), (200, 1, 1)])
def test_counters_emu(emu_doc, oracle_mod, n, a, chunk):
    for seed in range(1, 6):
        parity_checks.check_counters(emu_doc, oracle_mod, seed, n, a, chunk)


@pytest.mark.parametrize('cfg,n,a', [('C1', 0, 0), ('C2', 400, 0), ('C2b', 700, 0), ('C3', 3000, 10), ('C4', 2000, 4), ('C6', 400, 3), ('C7', 500, 3)])
def test_save_emu(emu_doc, oracle_mod, cfg, n, a):
    parity_checks.check_save(emu_doc, oracle_mod, cfg, n, a)


@pytest.mark.parametrize('cfg,n,a', [('C1', 0, 0), ('C2', 400, 0), ('C6', 300, 1), ('C7', 300, 1)])
def test_save_after_load_emu(emu_doc, oracle_mod, cfg, n, a):
    parity_checks.check_save_after_load(emu_doc, oracle_mod, cfg, n, a)


@pytest.mark.parametrize('n,a,chunk', [(80, 2, 1000), (300, 3, 5), (400, 4, 40), (200, 1, 1)])
def test_list_counters_emu(emu_doc, oracle_mod, n, a, chunk):
    compared = sum(parity_checks.check_rich_list(emu_doc, oracle_mod, seed, n, a, chunk, cfg='C8') for seed in range(1, 9))
    assert compared >= 5


def test_full_size_properties_emu(emu_doc):
    parity_checks.check_full_size_properties(emu_doc, n_ops=20000, n_actors=5, calls=7)


def test_pointer_array_entry_emu(emu_doc, oracle_mod):
    parity_checks.check_pointer_array_entry(emu_doc, oracle_mod)


def test_incremental_calls_emu(emu_doc, oracle_mod):
    parity_checks.check_incremental_calls(emu_doc, oracle_mod)


def test_out_of_order_emu(emu_doc, oracle_mod):
    parity_checks.check_out_of_order(emu_doc, oracle_mod)


def test_errors_atomic_emu(emu_doc):
    parity_checks.check_errors_atomic(emu_doc)


@pytest.mark.parametrize('cfg,n,a', [('C2', 600, 0), ('C3', 6000, 3), ('C1', 0, 0)])
def test_load_saved_document_emu(emu_doc, oracle_mod, cfg, n, a):
    parity_checks.check_load(emu_doc, oracle_mod, cfg, n, a)


def test_load_rust_document_emu(emu_doc):
    parity_checks.check_rust_document(emu_doc)


@pytest.mark.parametrize('seed', [1, 2, 3])
def test_column_decoders_emu(emu_doc, seed):
    parity_checks.check_column_decoders(emu_doc, seed, 120)


def test_load_parallel_columns_emu(emu_doc, oracle_mod, monkeypatch):
    monkeypatch.setenv('AMG_PAR_DOC_MIN', '1')   # every document takes the parallel column decoders (doccols.cuh)
    parity_checks.check_load_parallel_columns(emu_doc, oracle_mod, [('C2', 600, 0), ('C3', 6000, 3), ('C4', 3000, 4), ('C6', 500, 3), ('C7', 400, 3), ('C8', 400, 3)])
    parity_checks.check_rust_document(emu_doc)
    parity_checks.check_save_after_load(emu_doc, oracle_mod, 'C6', 300, 1)


@pytest.mark.parametrize('cfg,n,a', [('C1', 0, 0), ('C2', 300, 0), ('C2b', 400, 0), ('C3', 600, 3), ('C3', 3000, 10), ('C4', 1500, 4), ('C6', 300, 3), ('C7', 300, 3), ('C8', 300, 3)])
def test_history_after_load_emu(emu_doc, cfg, n, a):
    parity_checks.check_history_after_load(emu_doc, cfg, n, a)


def test_history_after_load_late_cut_emu(emu_doc):
    parity_checks.check_history_after_load(emu_doc, 'C3', 1000, 4, frac=0.9)


def test_empty_batch_emu(emu_doc):
    from automerge_classic_b200 import tracegen
    g = emu_doc()
    p0 = g.apply_changes([])                       # an empty array of changes is legal (backend.js:27-32)
    assert p0['diffs']['props'] == {} and p0['maxOp'] == 0
    g.apply_changes(tracegen.generate('C2', 50, 0).changes())
    before = g.save()
    p1 = g.apply_changes([])
    assert p1['diffs']['props'] == {} and g.save() == before


@pytest.mark.parametrize('cfg,n,a', [('C2', 300, 0), ('C3', 600, 3), ('C3', 2000, 4), ('C4', 1500, 4), ('C6', 300, 3), ('C7', 300, 3), ('C8', 300, 3)])
def test_history_against_oracle_emu(emu_doc, oracle_mod, cfg, n, a):
    parity_checks.check_history_against_oracle(emu_doc, oracle_mod, cfg, n, a)


def test_corrupt_documents_emu(emu_doc):
    stats = parity_checks.check_corrupt_documents(emu_doc)
    assert stats['loaded'] + stats['refused'] == 600


def test_block_boundary_cases_emu(emu_doc, oracle_mod):
    assert parity_checks.check_block_boundary_cases(emu_doc, oracle_mod)


def test_full_size_oracle_fingerprint_emu(emu_doc):
    # BASELINE.json's full size on the emulation build: bulk / chunked / loaded routes agree and save() has the oracle's digest
    parity_checks.check_full_size_properties(emu_doc)


@pytest.mark.parametrize('seed', [7, 8])
def test_out_of_order_random_emu(emu_doc, oracle_mod, seed):
    assert parity_checks.check_out_of_order_random(emu_doc, oracle_mod, seed, sessions=12) > 0


def test_local_changes_random_emu(emu_doc, oracle_mod):
    assert parity_checks.check_local_changes_random(emu_doc, oracle_mod, range(25)) == 25


@pytest.mark.parametrize('seed', [31, 32, 33, 34, 36])
def test_out_of_order_waiting_copies_emu(emu_doc, oracle_mod, seed):
    # (seed 35 runs into the duplicated-successor quirk of the reference, DESIGN.md section 5)
    assert parity_checks.check_out_of_order_random(emu_doc, oracle_mod, seed, sessions=15, waiting_copies=True) > 0


def test_load_without_head_indexes_emu(emu_doc, oracle_mod):
    parity_checks.check_load_without_head_indexes(emu_doc, oracle_mod)


def test_value_validation_emu(emu_doc, oracle_mod):
    parity_checks.check_value_validation(emu_doc, oracle_mod)


def test_duplicated_successor_pinned_emu(emu_doc, oracle_mod):
    parity_checks.check_duplicated_successor_pin(emu_doc, oracle_mod)


def test_unknown_columns_emu(emu_doc, oracle_mod):
    parity_checks.check_unknown_columns(emu_doc, oracle_mod)


def test_random_sweep_small_emu(emu_doc):
    """tools/sweep_emu.py, 60 random small trace configurations (C3 - C8): every patch, getPatch, op table, decoded rows and
    save() identical to the oracle's."""
    import sys
    root = os.path.dirname(HERE)
    out = subprocess.run([sys.executable, os.path.join(root, 'tools', 'sweep_emu.py'), '60', '99'], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and 'sweep: 60 cases identical' in out.stdout and ' 0 mismatches' in out.stdout, out.stdout[-600:] + out.stderr[-300:]


def test_deflate_fuzz_emu(emu_doc, oracle_mod):
    parity_checks.check_deflate_fuzz(emu_doc, oracle_mod, 400)


def test_apply_corrupted_emu(emu_doc, oracle_mod):
    both, refused, engine_only = parity_checks.check_apply_corrupted(emu_doc, oracle_mod, 40)
    assert both > 5 and refused > 5


DUMP_SCRIPT = r'''
import os, sys, numpy as np
sys.path.insert(0, %(root)r)
import bench                     # (bench.py sends file descriptor 1 to stderr: run in a process of its own)
raw = open(%(raw)r, 'rb').read()
bench.dump_outputs(raw, os.path.join(%(out)r, 'full'))
for d in ('a', 'b'):
    os.makedirs(os.path.join(%(out)r, d))
    for name, a in bench.patch_arrays(raw, budget=20000).items():
        np.save(os.path.join(%(out)r, d, name + '.npy'), a)
'''


def test_bench_dump_outputs_emu(emu_doc, tmp_path):
    """bench.py --dump-outputs: the arrays carry the flat patch's records and value bytes; under a smaller budget they are a
    seeded sample of the records that fits it and is the same on every run."""
    import sys
    import numpy as np
    from automerge_classic_b200 import tracegen
    t = tracegen.generate('C3', 3000, 3)
    fp = emu_doc().apply_packed_flat(t.blob, t.offsets, t.n_changes)
    (tmp_path / 'patch.bin').write_bytes(fp.raw)
    script = tmp_path / 'dump.py'
    script.write_text(DUMP_SCRIPT % {'root': os.path.dirname(HERE), 'raw': str(tmp_path / 'patch.bin'), 'out': str(tmp_path)})
    out = subprocess.run([sys.executable, str(script)], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]

    def load(d):
        return {f[:-4]: np.load(os.path.join(tmp_path, d, f)) for f in os.listdir(tmp_path / d)}
    full, a, b = load('full'), load('a'), load('b')
    assert all(v.dtype in (np.float32, np.float64) and v.size for v in full.values())
    assert 'props_key_bytes' in full and 'props_value_bytes' not in full   # the makeText entry has a key and no value bytes
    assert full['header'][0] == fp.max_op and np.array_equal(full['edits_row'], np.arange(len(fp.edits)))
    assert np.array_equal((full['edits_op_ctr'] * 65536 + full['edits_op_actor']).astype(np.uint64), fp.edits['opId'])
    text = [o for c in fp.to_patch(False)['diffs']['props'].values() for o in c.values()][0]
    chars = ''.join(v for e in text['edits'] for v in ([e['value']['value']] if e['action'] == 'insert' else e.get('values', [])))
    assert bytes(full['edits_value_bytes'].astype(np.uint8)).decode() == chars
    assert sum(os.path.getsize(os.path.join(tmp_path, 'a', f)) for f in os.listdir(tmp_path / 'a')) <= 20000
    assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a)
    rows = a['edits_row'].astype(np.int64)
    assert 0 < len(rows) < len(fp.edits) and np.array_equal(a['edits_index'], fp.edits['index'][rows])
