"""Shared helpers for the test-suite: model files from seeds, golden fixtures, tolerances."""
import os

import numpy as np

import binding as bd
import synth_gguf as sg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
FTYPES = {"f32": 0, "f16": 1, "q4_0": 2, "q4_1": 3, "q5_0": 6, "q5_1": 7, "q8_0": 8}
SEED = 1234
TOK_LENS = [77, 5, 2, 33, 16, 77, 9, 64]

# tolerances from BASELINE.json north_star: 1 - cos <= 1e-3 for f16 (and f32), <= 1e-2 for q4_0 (applied to all q*)
TOL = {"f32": 1e-3, "f16": 1e-3, "q4_0": 1e-2, "q4_1": 1e-2, "q5_0": 1e-2, "q5_1": 1e-2, "q8_0": 1e-2}


def golden(geom):
    p = os.path.join(GOLDEN, "%s-s%d.npz" % (geom, SEED))
    if not os.path.exists(p):
        return None
    z = np.load(p)
    return {k: z[k] for k in z.files}


def reference_runs():
    """What the reference returned for the inputs of the embedding and scoring tests (tests/golden/make_ref_golden.py)."""
    z = np.load(os.path.join(GOLDEN, "reference_runs.npz"))
    return {k: z[k] for k in z.files}


def model_file(geom: str, ftype: str, prod: "bd.ClipLib") -> str:
    """(geom, SEED, ftype) -> path; f16/f32 written from the seed, q* made with the PRODUCT's clip_model_quantize
    (byte-identical to the reference's: tests/test_host_side.py)."""
    path = sg.model_path(geom, SEED, ftype)
    if not os.path.exists(path):
        if ftype in ("f32", "f16"):
            sg.write_model(path, sg.GEOMETRIES[geom], SEED, FTYPES[ftype])
        else:
            src = model_file(geom, "f16", prod)
            assert prod.quantize(src, path + ".tmp", FTYPES[ftype]), prod.last_error()
            os.replace(path + ".tmp", path)
    return path


_sha_cache = {}


def check_sha(path, expect):
    """The file must be the one the golden vectors were produced from."""
    key = (path, os.path.getmtime(path))
    if key not in _sha_cache:
        _sha_cache[key] = sg.sha256_file(path)
    assert _sha_cache[key] == str(expect), "model file %s drifted from the golden fixture (generator changed?)" % path


def token_seqs(n, tok_seed=99):
    return [sg.synth_tokens(1, TOK_LENS[i % len(TOK_LENS)], tok_seed + i)[0] for i in range(n)]


def one_minus_cos(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    num = (a * b).sum(-1)
    den = np.linalg.norm(a, axis=-1) * np.linalg.norm(b, axis=-1)
    return 1.0 - num / den
