"""recorded outputs of the comparisons with the unmodified reference (dgkuester/iqwaveform), for machines where the
reference is not installed.

Each test that compares this project with the reference computes its own side first and passes it to `recorded()`.
Where the reference cannot be imported, `recorded()` checks those outputs, bit for bit, against the SHA-256 digest
stored for the test in tests/golden/reference_digests.json and returns True; the test then stops there.  Where the
reference is installed, `recorded()` returns False and the test compares with the live reference as before.

    IQW_RECORD_REFERENCE_DIGESTS=1 python -m pytest tests/test_oracle_vs_reference.py tests/test_io_host.py

rewrites the digests from a run on this machine (keep the file only if that run passed; with the reference installed
it also checks every recorded output against the reference).  A digest covers dtype, shape and every bit of an
array, so a stored digest is a bitwise comparison at 64 hex characters per test.

The reference, and the oracle with it, runs its FFTs on os.cpu_count() // 2 threads, and the thread count changes
the last bits of some transforms.  The file therefore also stores the CPU count of the machine that recorded it, and
a check against the digests runs the oracle with that count (`recorded_cpu_count()`).
"""
import atexit
import hashlib
import json
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'reference_digests.json')
RECORD = bool(os.environ.get('IQW_RECORD_REFERENCE_DIGESTS'))


def _load():
    if not os.path.exists(PATH):
        return {}
    with open(PATH) as f:
        return json.load(f)


_table = _load()


def _feed(h, obj):
    if isinstance(obj, (np.ndarray, np.generic)) and np.asarray(obj).dtype != object:
        a = np.ascontiguousarray(obj)
        h.update(f'array {a.dtype.str} {a.shape}|'.encode())
        h.update(a.tobytes())
    elif isinstance(obj, np.ndarray):
        _feed(h, obj.tolist())
    elif isinstance(obj, (list, tuple)):
        h.update(f'{type(obj).__name__} {len(obj)}|'.encode())
        for o in obj:
            _feed(h, o)
    elif isinstance(obj, dict):
        h.update(f'dict {len(obj)}|'.encode())
        for k in sorted(obj, key=repr):
            _feed(h, k)
            _feed(h, obj[k])
    elif hasattr(obj, 'columns') and hasattr(obj, 'index'):          # pandas DataFrame
        _feed(h, ('DataFrame', obj.values, obj.columns.values, obj.index.values))
    else:
        h.update(f'{type(obj).__name__} {obj!r}|'.encode())


def digest(*outputs) -> str:
    h = hashlib.sha256()
    _feed(h, outputs)
    return h.hexdigest()


def _test_id():
    # "tests/test_x.py::test_y[params] (call)" -> "test_x.py::test_y[params]"
    return os.environ['PYTEST_CURRENT_TEST'].rsplit(' ', 1)[0].split('/')[-1]


def recorded(ref, *outputs) -> bool:
    """this project's side of one test against the reference.  True: the reference (`ref`) is not installed and the
    outputs equal the recorded ones bit for bit.  False: `ref` is the live reference; compare with it."""
    key, d = _test_id(), digest(*outputs)
    if RECORD:
        _table[key] = d
        return ref is None
    if ref is not None:
        return False
    assert key in _table, f'no recorded reference digest for {key} in {PATH}'
    assert d == _table[key], f'{key}: outputs differ from the recorded reference outputs'
    return True


def recorded_cpu_count() -> int:
    return _table['_cpu_count']


def _save():
    _table['_cpu_count'] = os.cpu_count() or 1
    with open(PATH, 'w') as f:
        json.dump(dict(sorted(_table.items())), f, indent=0)
        f.write('\n')


if RECORD:
    atexit.register(_save)
