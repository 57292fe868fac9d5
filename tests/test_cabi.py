"""CPU-side checks of the C ABI: the library loads and exports every symbol include/vlfb.h declares."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, 'include', 'vlfb.h')).read()
    return sorted(set(re.findall(r'\b(vlfb_[a-z0-9_]+)\s*\(', src)))


def test_library_exports_every_declared_symbol():
    from vlfb import libvlfb
    lib = libvlfb.load()
    names = _declared()
    assert len(names) >= 30
    for n in names:
        assert hasattr(lib, n), n
    assert sorted(libvlfb.SIGNATURES) == names
    assert lib.vlfb_version() == 100


def test_argument_validation_without_gpu():
    from vlfb import libvlfb
    lib = libvlfb.load()
    assert lib.vlfb_gemm(None, None) == -1
    assert b'bad argument' in lib.vlfb_last_error()
    p = libvlfb.GemmParams()
    p.a.ptr = p.b.ptr = p.d = 256                       # never dereferenced: validation fails first
    p.M, p.N, p.K, p.batch, p.taps, p.split_k, p.engine = 128, 128, 128, 1, 1, 1, 7
    assert lib.vlfb_gemm(ctypes.byref(p), None) == -1 and b'engine' in lib.vlfb_last_error()
    p.engine, p.tile_n = 0, 48
    assert lib.vlfb_gemm(ctypes.byref(p), None) == -1 and b'tile_n' in lib.vlfb_last_error()
    p.tile_n, p.flags, p.relu_bits_out = 0, 0, 256                    # sign bits without VLFB_EPI_RELU
    assert lib.vlfb_gemm(ctypes.byref(p), None) == -1 and b'relu_bits_out' in lib.vlfb_last_error()
    assert lib.vlfb_relu_fwd(None, None, 4, None) == -1


def test_struct_layout_matches_header(tmp_path):
    """sizeof / offsetof of the C structs, as the C compiler sees include/vlfb.h, equal the ctypes mirror."""
    import subprocess
    from vlfb import libvlfb as L
    fields = ['a', 'b', 'g', 'M', 'split_k', 'd', 'ldd', 'alpha', 'col_scale', 'residual', 'relu_mask', 'flags',
              'workspace', 'workspace_bytes', 'engine', 'tile_n', 'pair', 'stream_k', 'relu_mask_bits', 'relu_bits_out']
    src = tmp_path / 'layout.c'
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "vlfb.h"\nint main(void) {\n'
                   '  printf("%zu %zu %zu %zu\\n", sizeof(vlfb_conv_geom_t), sizeof(vlfb_operand_t), sizeof(vlfb_gemm_params_t), sizeof(vlfb_gemm_plan_t));\n'
                   + ''.join('  printf("%%zu\\n", offsetof(vlfb_gemm_params_t, %s));\n' % f for f in fields)
                   + '  return 0;\n}\n')
    exe = tmp_path / 'layout'
    subprocess.check_call(['gcc', '-I', os.path.join(ROOT, 'include'), str(src), '-o', str(exe)])
    out = subprocess.check_output([str(exe)]).decode().split()
    sizes, offs = [int(v) for v in out[:4]], [int(v) for v in out[4:]]
    assert sizes == [ctypes.sizeof(L.ConvGeom), ctypes.sizeof(L.Operand), ctypes.sizeof(L.GemmParams), ctypes.sizeof(L.GemmPlan)]
    assert offs == [getattr(L.GemmParams, f).offset for f in fields]


def test_wt_job_layout(tmp_path):
    """The device job table of vlfb_weight_transpose_multi is written from numpy: 40-byte records."""
    import subprocess
    src = tmp_path / 'job.c'
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "vlfb.h"\nint main(void) {\n'
                   '  printf("%zu %zu %zu %zu %zu\\n", sizeof(vlfb_wt_job_t), offsetof(vlfb_wt_job_t, wt), '
                   'offsetof(vlfb_wt_job_t, scale), offsetof(vlfb_wt_job_t, Co), offsetof(vlfb_wt_job_t, block_begin));\n'
                   '  return 0;\n}\n')
    exe = tmp_path / 'job'
    subprocess.check_call(['gcc', '-I', os.path.join(ROOT, 'include'), str(src), '-o', str(exe)])
    assert subprocess.check_output([str(exe)]).decode().split() == ['40', '8', '16', '24', '36']



def test_gemm_plan_query():
    """Host-only: the tiling / schedule the tensor-core GEMM would use (vlfb_gemm_plan).  The res4/res5 layers of a
    2-clip batch have M = 6272 = 49 row tiles of 128: with 128 x 256 tiles they fill 98 of 148 SMs (round 1).  CTA
    pairs (cta_group::2, 256-row tiles) halve the operand bytes per SM and stream-K gives every pair the same number
    of K chunks whatever the tile count."""
    import ctypes as C
    from vlfb import libvlfb as L
    lib = L.load()
    ws_bytes = lib.vlfb_gemm_workspace_bytes()
    assert ws_bytes >= 16384 * 4 + 148 * 2 * 128 * 256 * 4

    def plan(M, N, K, split=1, taps=1, flags=0, ws=True, **opts):
        p = L.GemmParams()
        p.M, p.N, p.K, p.batch, p.taps, p.split_k, p.flags = M, N, K, 1, taps, split, flags
        if ws:
            p.workspace, p.workspace_bytes = 4096, ws_bytes      # host-only query: the pointer is never dereferenced
        for k, v in opts.items():
            setattr(p, k, v)
        out = L.GemmPlan()
        assert lib.vlfb_gemm_plan(C.byref(p), 148, C.byref(out)) == 0
        return out

    r5 = plan(6272, 512, 4608, pair=1, stream_k=1)               # res5 branch2b on pairs + stream-K (opt-in)
    assert (r5.tile_n, r5.pair, r5.stream_k, r5.units, r5.tiles) == (256, 1, 1, 74, 50)
    r4 = plan(6272, 256, 2304, pair=1, stream_k=1)               # res4 branch2b: 25 pair tiles over 74 pairs
    assert (r4.tile_n, r4.pair, r4.stream_k, r4.units) == (256, 1, 1, 74)
    nows = plan(6272, 512, 4608, ws=False, pair=1, stream_k=1)   # no workspace -> no fix-up schedule
    assert nows.stream_k == 0 and nows.pair == 1
    off = plan(6272, 512, 4608)                                  # default: the static tile loop on single CTAs
    assert (off.tile_n, off.pair, off.stream_k, off.tiles, off.units) == (256, 0, 0, 98, 98)
    big = plan(200704, 256, 64)                                  # res2 1x1: thousands of tiles, static loop
    assert big.stream_k == 0 and big.tile_n == 256
    forced = plan(6272, 512, 4608, tile_n=192, pair=-1, stream_k=-1)
    assert (forced.tile_n, forced.tiles) == (192, 147)
    for M, N, K in [(4, 80, 2560), (3136, 784, 256), (512, 4608, 6272), (64, 224, 802816), (1, 300, 512)]:
        o = plan(M, N, K, split=0, flags=L.EPI_ATOMIC)
        assert o.tile_n % 32 == 0 and 32 <= o.tile_n <= 256 and o.split_k >= 1
        assert o.tile_n & (o.tile_n - 1) == 0
        assert o.tile_n == 32 or N > o.tile_n // 2               # never pad N by 2x or more
        assert o.tiles == -(-M // (256 if o.pair else 128)) * -(-N // o.tile_n) * o.split_k
        assert not (o.stream_k and o.split_k != 1)
        assert o.split_k == 1                                    # with a workspace: no order-dependent K slices
    # conv1-style weight gradient (one tile, K ~ 8e5): stream-K pieces summed in a fixed order in the workspace; without
    # a workspace, or with stream-K refused, plain (atomic) split-K spreads the reduction instead
    w = plan(64, 224, 802816, split=0, flags=L.EPI_ATOMIC)
    assert (w.split_k, w.stream_k, w.units) == (1, 1, 148)
    assert plan(64, 224, 802816, split=0, flags=L.EPI_ATOMIC, ws=False).split_k > 1
    assert plan(64, 224, 802816, split=0, flags=L.EPI_ATOMIC, stream_k=-1).split_k > 1
    assert lib.vlfb_gemm_plan(None, 148, None) == -1


def test_colsum_workspace_query():
    """Host-only: colsum needs no workspace when one slab of rows suffices (rows <= 64), else one partial sum per slab
    and column.  Slabs: about two waves of 32-column blocks on 148 SMs, at least 64 rows each."""
    from vlfb import libvlfb as L
    lib = L.load()
    for rows in (1, 63, 64, 65, 128, 129, 1000, 50000, 70000, 1 << 20):
        for cols in (1, 20, 80, 157, 512, 2048, 9440, 9441, 20000):
            slabs = max(1, min(-(-296 // -(-cols // 32)), -(-rows // 64)))
            want = 0 if slabs == 1 else slabs * cols * 4
            assert lib.vlfb_colsum_workspace_bytes(rows, cols) == want, (rows, cols)
            if rows <= 64:
                assert want == 0
    assert lib.vlfb_colsum_workspace_bytes(65, 1) == 2 * 4
    assert lib.vlfb_colsum_workspace_bytes(0, 80) == 0 and lib.vlfb_colsum_workspace_bytes(100, 0) == 0


def test_fbo_bank_scan_split_table_properties():
    """Host-only: the split of a RoI's L bank rows over CTAs never leaves an empty split, covers all rows, and the
    workspace query matches it (csrc/fbo.cu vlfb_fbo_bank_scan_splits)."""
    from vlfb import libvlfb as L
    lib = L.load()
    for D, rows_per_tile in [(1024, 8), (2048, 8), (4096, 4)]:
        for R in (1, 2, 3, 4, 16, 37, 64, 255, 256, 1000):
            for Lb in (1, 2, 7, 8, 9, 60, 300, 301, 1200, 3600):
                s = lib.vlfb_fbo_bank_scan_splits(R, Lb, D)
                per = -(-Lb // s)
                assert 1 <= s <= 1024 and (s - 1) * per < Lb <= s * per, (R, Lb, D, s)
                assert s <= -(-Lb // rows_per_tile), 'a split holds at least one tile of rows'
                assert lib.vlfb_fbo_bank_scan_workspace(R, Lb, D) == (R * s * D + R * s * 2) * 4
    for bad in [(0, 300, 2048), (4, 0, 2048), (4, 300, 512), (4, 300, 2047)]:
        assert lib.vlfb_fbo_bank_scan_splits(*bad) == 0 and lib.vlfb_fbo_bank_scan_workspace(*bad) == 0
    # many RoIs: enough CTAs for two per SM without splitting rows needlessly
    assert lib.vlfb_fbo_bank_scan_splits(1000, 17, 2048) <= 3
