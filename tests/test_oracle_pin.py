"""Pins the CPU oracle (oracle/clip_oracle.c + oracle.py) before it is trusted as the checker:
  1. against golden embeddings the REFERENCE produced (tests/golden/*.npz, made by oracle/_ref);
  2. against the reference's embeddings of inputs outside those fixtures, un-normalised (tests/golden/reference_runs.npz);
  3. its block quantizer against the reference's quantized model files (sha256 of the whole GGUF).
Tolerances: the oracle reproduces every rounding point of the reference, so only summation order differs; quantized
paths re-quantize activations per layer, which turns ulp-level differences into occasional +-1 flips (observed 1e-5)."""
import os

import numpy as np
import pytest

import oracle as orc
import synth_gguf as sg
from _util import FTYPES, check_sha, golden, model_file, one_minus_cos, reference_runs, token_seqs

PIN_TOL = {"f32": 1e-5, "f16": 1e-5, "q4_0": 5e-4, "q4_1": 5e-4, "q5_0": 5e-4, "q5_1": 5e-4, "q8_0": 5e-4}


@pytest.mark.parametrize("ft", list(FTYPES))
def test_oracle_matches_reference_golden_tiny(prod, ft):
    g = golden("tiny")
    path = model_file("tiny", ft, prod)
    check_sha(path, g["sha_" + ft])
    m = orc.OracleModel(path)
    imgs = sg.synth_images(int(g["n_img"]), 64, int(g["img_seed"]))
    seqs = token_seqs(int(g["n_txt"]), int(g["tok_seed"]))
    oi = np.stack([m.encode_image(im) for im in imgs[:2]])
    ot = np.stack([m.encode_text(s) for s in seqs[:4]])
    assert one_minus_cos(oi, g["img_" + ft][:2]).max() <= PIN_TOL[ft]
    assert one_minus_cos(ot, g["txt_" + ft][:4]).max() <= PIN_TOL[ft]


@pytest.mark.parametrize("geom,ft", [("tiny-gelu", "f16"), ("tiny-gelu", "q4_0"), ("small-p14", "f16"), ("small-p14", "q8_0")])
def test_oracle_matches_reference_golden_variants(prod, geom, ft):
    g = golden(geom)
    path = model_file(geom, ft, prod)
    check_sha(path, g["sha_" + ft])
    m = orc.OracleModel(path)
    img = sg.synth_images(int(g["n_img"]), sg.GEOMETRIES[geom].image_size, int(g["img_seed"]))[0]
    seq = token_seqs(int(g["n_txt"]), int(g["tok_seed"]))[0]
    assert one_minus_cos(m.encode_image(img), g["img_" + ft][0]) <= PIN_TOL[ft]
    assert one_minus_cos(m.encode_text(seq), g["txt_" + ft][0]) <= PIN_TOL[ft]


LIVE_FTYPES = ["f16", "q4_1", "q5_0"]


def live_inputs():
    """Inputs of test_oracle_matches_live_reference: seeds none of the golden fixtures above use."""
    return sg.synth_images(2, 64, 31337), [sg.synth_tokens(1, n, 7 * n)[0] for n in (4, 50)]


@pytest.mark.parametrize("ft", LIVE_FTYPES)
def test_oracle_matches_live_reference(prod, ft):
    """Un-normalised embeddings of fresh inputs against the reference's (recorded by tests/golden/make_ref_golden.py)."""
    path = model_file("tiny", ft, prod)
    check_sha(path, golden("tiny")["sha_" + ft])
    imgs, seqs = live_inputs()
    g = reference_runs()
    r = {"img": g["pin_img_" + ft], "txt": g["pin_txt_" + ft]}
    m = orc.OracleModel(path)
    for i in range(2):
        oi, ot = m.encode_image(imgs[i], normalize=False), m.encode_text(seqs[i], normalize=False)
        assert one_minus_cos(oi, r["img"][i]) <= PIN_TOL[ft]
        assert one_minus_cos(ot, r["txt"][i]) <= PIN_TOL[ft]
        assert abs(np.linalg.norm(oi) / np.linalg.norm(r["img"][i]) - 1) < 1e-2


@pytest.mark.parametrize("ft", ["q4_0", "q4_1", "q5_0", "q5_1", "q8_0"])
def test_oracle_quantizer_reproduces_reference_blocks(prod, ft):
    """orc_quantize_row == the reference's quantize_row_*_reference: re-quantising the f16 weights with the oracle
    gives byte-identical tensor payloads to the file whose sha256 the reference-made fixture records."""
    g = golden("tiny")
    qpath, fpath = model_file("tiny", ft, prod), model_file("tiny", "f16", prod)
    check_sha(qpath, g["sha_" + ft])
    gq, gf = orc.GGUF(qpath), orc.GGUF(fpath)
    n = 0
    for name in ["v.blk.3.attn_q.weight", "t.blk.11.ffn_up.weight", "visual_projection.weight", "v.position_embd.weight"]:
        w = gf.tensors[name].f32()
        assert orc.quantize_rows(FTYPES[ft], w) == bytes(gq.tensors[name].data), name
        n += 1
    assert n == 4


def test_oracle_dequant_matches_format_definition():
    """Hand-built q4_0 / q8_0 blocks with known values (ggml.c:1496-1512, 1599-1605)."""
    import ctypes as C
    blk = np.zeros(18, np.uint8)
    blk[0:2] = np.array([0.5], np.float16).view(np.uint8)
    blk[2:] = np.arange(16, dtype=np.uint8) | ((15 - np.arange(16, dtype=np.uint8)) << 4)
    out = np.empty(32, np.float32)
    assert orc.lib().orc_dequantize_row(orc.Q4_0, blk.ctypes.data, out.ctypes.data_as(C.POINTER(C.c_float)), 32) == 0
    assert np.array_equal(out[:16], (np.arange(16) - 8) * 0.5) and np.array_equal(out[16:], (15 - np.arange(16) - 8) * 0.5)
    b8 = np.zeros(34, np.uint8)
    b8[0:2] = np.array([0.25], np.float16).view(np.uint8)
    b8[2:] = np.arange(-16, 16, dtype=np.int8).view(np.uint8)
    assert orc.lib().orc_dequantize_row(orc.Q8_0, b8.ctypes.data, out.ctypes.data_as(C.POINTER(C.c_float)), 32) == 0
    assert np.array_equal(out, np.arange(-16, 16) * 0.25)
