"""The C-ABI shared library loads and exports every symbol include/regnn_b200.h declares, and the
ctypes signature table covers exactly that set (no compute calls: there is no GPU here)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, 'include', 'regnn_b200.h')


def declared_symbols():
    text = open(HEADER).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(regnn_\w+)\s*\(', text)))


@pytest.fixture(scope='module')
def lib():
    from re_gnn_b200 import build, _lib
    build.build_library()       # no-op when the .so is newer than the sources
    return _lib.load()


def test_header_declares_expected_entry_points():
    syms = declared_symbols()
    for s in ('regnn_csr_build', 'regnn_etype_permute', 'regnn_wdeg_norm_fwd', 'regnn_wdeg_norm_bwd',
              'regnn_spmm_fwd', 'regnn_spmm_bwd_w', 'regnn_gat_fwd', 'regnn_gat_bwd_stats', 'regnn_gat_bwd_edges', 'regnn_gat_bwd_reduce',
              'regnn_gatv2_fwd', 'regnn_gatv2_bwd_edges_blocks', 'regnn_gatv2_bwd_edges', 'regnn_gatv2_bwd_dst'):
        assert s in syms


def test_library_exports_every_declared_symbol(lib):
    for s in declared_symbols():
        assert hasattr(lib, s), 'libregnn_b200.so does not export %s' % s


def test_ctypes_table_matches_header(lib):
    from re_gnn_b200 import _lib
    assert sorted(_lib.SIGNATURES) == declared_symbols()
    text = re.sub(r'/\*.*?\*/', '', open(HEADER).read(), flags=re.S)
    for name, (_, argtypes) in _lib.SIGNATURES.items():
        m = re.search(r'\b%s\s*\((.*?)\)\s*;' % name, text, flags=re.S)
        assert m, name
        params = m.group(1).strip()
        n = 0 if params in ('', 'void') else len(params.split(','))
        assert n == len(argtypes), '%s: header has %d parameters, ctypes table %d' % (name, n, len(argtypes))


def test_status_strings_and_version(lib):
    assert lib.regnn_version() >= 100
    assert lib.regnn_status_string(0) == b'ok'
    assert lib.regnn_status_string(-2) == b'unsupported shape'
    assert lib.regnn_max_partial_blocks() == 4736
    assert lib.regnn_csr_build_workspace_bytes(10, 0) > 0


def test_argument_validation_without_a_gpu(lib):
    """Entry points validate before touching the device: bad arguments come back as status codes."""
    assert lib.regnn_csr_build(None, None, -1, 0, None, None, None, None, None, None, None, None, 0, None) == -1
    assert lib.regnn_etype_permute(None, None, None, 5, 300, None, None, None, None) == -2
    assert b'num_relations' in lib.regnn_last_error_string()
    assert lib.regnn_spmm_fwd(None, None, None, None, 1.0, 0, None, None, None, 4, None, 4, 0, 0, 4, None, None, None, None) == -1


def test_missing_library_fails_loudly(monkeypatch):
    from re_gnn_b200 import _lib
    monkeypatch.setattr(_lib, '_lib', None)
    monkeypatch.setattr(_lib, 'LIB_PATH', '/nonexistent/libregnn_b200.so')
    with pytest.raises(RuntimeError, match='no CPU or eager fallback'):
        _lib.load()


def test_struct_layouts_match_the_c_header(tmp_path):
    """The header compiles as plain C and the ctypes mirrors of its structs have the C compiler's layout."""
    import subprocess
    from re_gnn_b200 import _lib
    src = tmp_path / 'layout.c'
    src.write_text('''#include <stdio.h>
#include <stddef.h>
#include "regnn_b200.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(regnn_rowsplit_t), offsetof(regnn_rowsplit_t, frag_begin),
         offsetof(regnn_rowsplit_t, num_long), offsetof(regnn_rowsplit_t, threshold), sizeof(regnn_peer_rows_t),
         offsetof(regnn_peer_rows_t, num_ranks), offsetof(regnn_peer_rows_t, rows_per_rank),
         offsetof(regnn_peer_rows_t, col_offset));
  return 0;
}
''')
    exe = tmp_path / 'layout'
    subprocess.run(['gcc', '-std=c99', '-Wall', '-Werror', '-I', os.path.join(ROOT, 'include'), str(src), '-o', str(exe)],
                   check=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    rs, pr = _lib.RowSplit, _lib.PeerRows
    want = [ctypes.sizeof(rs), rs.frag_begin.offset, rs.num_long.offset, rs.threshold.offset, ctypes.sizeof(pr),
            pr.num_ranks.offset, pr.rows_per_rank.offset, pr.col_offset.offset]
    assert got == want


def test_scatter_entry_points_validate_arguments(lib):
    """The peer-memory variants reject a missing peer table / a shape the narrow-row kernel cannot take before any launch."""
    from re_gnn_b200 import _lib
    assert lib.regnn_spmm_fwd_scatter(None, None, None, None, 1.0, 0, None, None, None, 4, 8, 4, None, None, None, None,
                                      None, 0, None) == -1
    assert b'peer' in lib.regnn_last_error_string()
    assert lib.regnn_rows_to_slabs(None, 4, 8, 4, 2, 0, None, None) == -1
    peers = _lib.PeerRows(1, 2, 4, 6, 0)   # ld 6 is not a multiple of 4 floats
    assert lib.regnn_spmm_bwd_fused_scatter(None, None, None, None, 1.0, 1, None, 3, None, 4, None, 4, 8, 4, None, None,
                                            None, None, 0, None, None, None, None, ctypes.byref(peers), None) == -1


def test_every_entry_point_is_called_from_one_wrapper():
    """ops.py's contract, one Python function per C-ABI entry point: each regnn_* name passed to ``_lib.call`` appears
    in exactly one call of the package, so a change to an entry point's arguments, buffers or launch count has one
    place to go."""
    import collections
    import glob
    counts, calls = collections.Counter(), 0
    for path in glob.glob(os.path.join(ROOT, 're_gnn_b200', '*.py')):
        with open(path) as f:
            text = f.read()
        calls += text.count('_lib.call(')
        counts.update(re.findall(r"_lib\.call\(\s*'(regnn_\w+)'", text))
    assert counts and sum(counts.values()) == calls, 'every _lib.call names its entry point as a literal'
    shared = {name: c for name, c in counts.items() if c > 1}
    assert not shared, shared


def test_integration_doc_lists_every_entry_point():
    """INTEGRATION.md maps every exported symbol to the reference call site it replaces."""
    text = open(os.path.join(ROOT, 'INTEGRATION.md')).read()
    missing = [s for s in declared_symbols() if s not in text]
    assert not missing, missing
