"""tests/test_gpu_pair_r32.py against the emulated library (tests/test_library_on_cpu.py):
the 32-byte-record list kernel, its eligibility and its fallbacks run on the CPU, at a
smaller dam break."""
import pytest

from test_library_on_cpu import _call, _id, emulated_library  # noqa: F401  (the fixture)

CASES = [
    ('test_gpu_pair_r32', 'test_r32_matches_the_48_byte_path', {'monkeypatch': None, 'dx': 0.08}),
] + [('test_gpu_pair_r32', 'test_r32_fallbacks_are_the_48_byte_path', {'monkeypatch': None, 'case': c, 'dx': 0.08})
     for c in ('h', 'm', 'classes', 'update_h')] + [
    ('test_gpu_pair_r32', 'test_r32_periodic', {'monkeypatch': None, 'n': 8}),
]


@pytest.mark.parametrize('t', CASES, ids=_id)
def test_pair_r32_on_the_emulated_library(emulated_library, t):  # noqa: F811
    _call(t, emulated_library)
