"""Decode-time JPEG block scalers (SURVEY.md section 8(f) item 1; c_components/lib/codecs_jpeg_idct_fast.c).

The oracle for this row is the REFERENCE ITSELF: oracle/_ref/libidct_ref.so is that C file compiled unmodified (oracle/Makefile),
and tests/golden/idct_golden.npz holds its outputs for two committed planes of blocks (tests/golden/make_idct_golden.py).
CPU: the reference's known answer (188), _ref against the committed vectors where _ref is built, and the product's tables (the
literals extracted from the C file, evaluated by a plain host loop) against both.  GPU: the kernel through the C ABI, bit-exact
against the committed vectors."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = np.load(os.path.join(ROOT, "tests", "golden", "idct_golden.npz"))
VARIANTS = [(s, n) for s in (0, 1) for n in range(1, 8)]


def test_reference_known_answer_and_committed_vectors():
    """c_components/tests/test_idct_scaling.rs:4-18: alternating 0/255 through flow_scale_spatial_srgb_1x1 -> 188"""
    assert GOLD["out_1_1"][0, 2] == 188
    if not oracle.idct_ref_available():
        pytest.skip("oracle/_ref not built (no reference tree on this machine)")
    blk = np.tile(np.array([0, 255], np.uint8), 32).reshape(8, 8)
    assert oracle.flow_scale_spatial_ref(blk, 1, True)[0, 0] == 188
    for s, n in VARIANTS:
        assert np.array_equal(oracle.flow_scale_spatial_ref(GOLD["plane"], n, bool(s)), GOLD[f"out_{s}_{n}"]), (s, n)
        assert np.array_equal(oracle.flow_scale_spatial_ref(GOLD["random_plane"], n, bool(s)), GOLD[f"random_{s}_{n}"]), (s, n)


def test_product_tables_reproduce_the_reference(tmp_path):
    so = str(tmp_path / "libidct_tables_eval.so")
    subprocess.run(["g++", "-O2", "-shared", "-fPIC", "-o", so, os.path.join(ROOT, "tests", "cpu_emu", "idct_tables_eval.cc")], check=True)
    L = C.CDLL(so)
    L.idct_tables_eval.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint32, C.c_int, C.c_int]
    L.idct_tables_eval.restype = None

    def ev(p, n, s):
        out = np.zeros((p.shape[0] // 8 * n, p.shape[1] // 8 * n), np.uint8)
        L.idct_tables_eval(p.ctypes.data, p.strides[0], p.shape[1] // 8, p.shape[0] // 8, out.ctypes.data, out.strides[0], n, s)
        return out
    p = np.ascontiguousarray(GOLD["plane"])
    r = np.ascontiguousarray(GOLD["random_plane"])
    for s, n in VARIANTS:
        assert np.array_equal(ev(p, n, s), GOLD[f"out_{s}_{n}"]), (s, n)
        assert np.array_equal(ev(r, n, s), GOLD[f"random_{s}_{n}"]), (s, n)
    if oracle.idct_ref_available():                                   # a larger random plane against the reference itself
        big = np.random.default_rng(5).integers(0, 256, (256, 320), dtype=np.uint8)
        for s, n in VARIANTS:
            assert np.array_equal(ev(big, n, s), oracle.flow_scale_spatial_ref(big, n, bool(s))), (s, n)


@pytest.mark.gpu
def test_gpu_block_scalers_bit_exact():
    import torch
    import imageflow_b200 as ifb
    assert ifb.device_count() > 0 and torch.cuda.is_available()
    p = np.ascontiguousarray(GOLD["plane"])
    for s, n in VARIANTS:                                             # host-buffer drop-in against the committed vectors
        assert np.array_equal(ifb.flow_scale_spatial(p, n, bool(s)), GOLD[f"out_{s}_{n}"]), (s, n)
    # device-resident, odd block counts (33 x 5 blocks: two CTAs per block row), padded pitches
    big = np.ascontiguousarray(GOLD["random_plane"])
    b = ifb.Batch(0)
    st = torch.cuda.current_stream().cuda_stream
    tin = torch.zeros((40, 320), dtype=torch.uint8, device="cuda")
    tin[:, :264] = torch.from_numpy(big).cuda()
    for s, n in VARIANTS:
        tout = torch.zeros((5 * n, 256), dtype=torch.uint8, device="cuda")
        b.block_scale(tin.data_ptr(), 320, 33, 5, tout.data_ptr(), 256, n, bool(s), stream=st)
        torch.cuda.synchronize()
        got = tout[:, :33 * n].cpu().numpy()
        assert np.array_equal(got, GOLD[f"random_{s}_{n}"]), (s, n)
        assert np.array_equal(got, ifb.flow_scale_spatial(big, n, bool(s))), (s, n)
    with pytest.raises(ifb.FlowError):
        ifb.flow_scale_spatial(p, 8)
    b.close()
