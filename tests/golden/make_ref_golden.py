"""Records what the REFERENCE ITSELF (oracle/_ref, built by oracle/Makefile) returns for the inputs of the tests that compare with
it beyond the other fixtures, so that those tests run wherever the product runs:

  reference_runs.json  the image decoder tests of tests/test_host_side.py, each run once with the reference library standing in
                       for the recording (every file it writes must decode to the same pixels in both libraries, as before); the
                       tokens and preprocessed floats of test_tokenizer_and_preprocess_match_live_reference;
  reference_runs.npz   un-normalised embeddings for tests/test_oracle_pin.py and the scoring results (clip_compare_text_and_image,
                       clip_zero_shot_label_image) for tests/test_gpu_scoring.py.

Run after build() in the build container, with the reference's sample JPEGs copied to tests/golden/jpeg/ref_*.jpg:
    python tests/golden/make_ref_golden.py
"""
import json
import os
import pathlib
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in ("clip.cpp_b200", "oracle", "tests"):
    sys.path.insert(0, os.path.join(ROOT, p))
import binding as bd                # noqa: E402
import ref_run                      # noqa: E402
import test_gpu_scoring as tsc      # noqa: E402
import test_host_side as ths        # noqa: E402
import test_oracle_pin as tpin      # noqa: E402
from _util import model_file        # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")


class Recorder:
    """Stands in for test_host_side._ReferenceDecodes: decodes each file with the reference, checks the product agrees, records it."""

    def __init__(self, ref, rows, pin_files):
        self.ref, self.rows, self.pin_files = ref, rows, pin_files

    def check(self, path, got):
        want = ths._load_file(self.ref, path)
        assert want is not None and got is not None and np.array_equal(got, want), (path, len(self.rows))
        self.rows.append([ths._sha(open(path, "rb").read()) if self.pin_files else None, ths._sha(want.tobytes())])

    def done(self):
        pass


def record_decodes(prod, ref):
    decodes = {}
    tests = {"png_pil": ths.test_png_decode_matches_live_reference, "png_modes": ths.test_png_every_colour_type_depth_and_interlace,
             "bmp_pnm": ths.test_bmp_and_pnm_variants, "gif": ths.test_gif_first_frame, "jpeg_pil": ths.test_jpeg_decode_matches_live_reference}
    for name, fn in tests.items():
        rows = decodes[name] = []
        ths._reference_decodes = lambda test, pin_files=False, rows=rows: Recorder(ref, rows, pin_files)
        with tempfile.TemporaryDirectory() as td:
            fn(prod, pathlib.Path(td))
        print("%-10s %d files" % (name, len(rows)))
    return decodes


def main():
    assert ref_run.available(), "build oracle/_ref first (build() or make -C oracle ref)"
    prod, ref = bd.ClipLib(bd.PRODUCT_LIB), bd.ClipLib(ref_run.REF_LIB)
    out = {"source": "oracle/_ref/libclip_ref.so (the unmodified reference), tests/golden/make_ref_golden.py"}
    out["decodes"] = record_decodes(prod, ref)

    model = model_file("tiny", "f16", prod)
    ctx = ref.load(model, 0)
    out["tokenize_preprocess"] = {"model_sha": ths.sg.sha256_file(model),
                                  "tokens": [[int(v) for v in ref.tokenize(ctx, t)] for t in ths.LIVE_TEXTS],
                                  "preprocess_sha256": ths._sha(ref.preprocess(ctx, ths._synth_u8(*ths.LIVE_IMAGE)).tobytes())}
    ref.free(ctx)
    with open(os.path.join(GOLDEN, "reference_runs.json"), "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)

    arrays = {}
    imgs, seqs = tpin.live_inputs()
    for ft in tpin.LIVE_FTYPES:
        r = ref_run.run_reference(model_file("tiny", ft, prod), imgs, seqs, n_threads=2, normalize=False)
        arrays["pin_img_" + ft], arrays["pin_txt_" + ft] = r["img"], r["txt"]
    for ft in ("f16", "q4_0"):
        r = ref_run.run_reference(model_file("tiny", ft, prod), u8_image=tsc._u8(*tsc.SCORING_IMAGE), texts=tsc.TEXTS, n_threads=4)
        arrays["cmp_" + ft], arrays["zsl_scores_" + ft], arrays["zsl_idx_" + ft] = r["cmp"], r["zsl_scores"], r["zsl_idx"]
    np.savez_compressed(os.path.join(GOLDEN, "reference_runs.npz"), **arrays)
    print("wrote reference_runs.json and reference_runs.npz:", sorted(arrays))


if __name__ == "__main__":
    main()
