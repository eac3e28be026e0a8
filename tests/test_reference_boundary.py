"""CPU-side boundary check made with the reference's own symbol list (no GPU, no compute calls): the symbol list the
ABI tests use is the one python/cwipc/util.py of the reference binds (tests/golden/reference_bound_symbols.txt), not a
hand-typed copy that could drift from it."""
import os

from test_abi_exports import REFERENCE_BOUND_SYMBOLS, declared_functions

BOUND = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_bound_symbols.txt")


def reference_bound_symbols():
    return [l.strip() for l in open(BOUND) if l.strip() and not l.startswith("#")]


def test_bound_symbols_are_the_ones_the_reference_binds(lib):
    """Every `_cwipc_util_dll_reference.<name>.argtypes = ...` of python/cwipc/util.py:387-550 resolves in our library,
    and the hand-typed list of test_abi_exports.py is exactly that set (+ cwipc_write, which only the C++ apps use)."""
    bound = sorted(set(reference_bound_symbols()))
    assert len(bound) > 50
    missing = [name for name in bound if not hasattr(lib, name)]
    assert not missing, f"library lacks symbols the reference binds at load time: {missing}"
    declared = set(declared_functions())
    assert not [name for name in bound if name not in declared]
    assert set(bound) == set(REFERENCE_BOUND_SYMBOLS) - {"cwipc_write"}
