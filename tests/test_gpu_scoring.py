"""Scoring entry points of the C ABI on the GPU: clip_compare_text_and_image (clip.cpp:1534-1571) and clip_zero_shot_label_image
(clip.cpp:1624-1659) against what the reference returned (tests/golden/reference_runs.npz), the device similarity / softmax / top-k
kernels against numpy restatements of softmax_with_sorting (clip.cpp:1591-1622), the batched zero-shot call, the device-resident
text entry point, and pinned vs pageable caller buffers."""
import ctypes as C

import numpy as np
import pytest

import synth_gguf as sg
from _util import check_sha, golden, model_file, one_minus_cos, reference_runs, token_seqs

pytestmark = pytest.mark.gpu

TEXTS = ["a photo of a cat", "a photo of a dog", "red apple", "two cars on the road", "the sky", "it's 12 o'clock"]
SCORING_IMAGE = (120, 90, 5)        # nx, ny, seed of _u8


def _u8(nx, ny, seed):
    rng = np.random.default_rng(seed)
    base = rng.integers(0, 256, (ny // 8 + 2, nx // 8 + 2, 3)).astype(np.float32)
    img = np.kron(base, np.ones((8, 8, 1), np.float32))[:ny, :nx] + rng.normal(0, 10, (ny, nx, 3))
    return np.clip(img, 0, 255).astype(np.uint8)


def _softmax_sorted(s):
    """softmax_with_sorting's arithmetic (clip.cpp:1599-1607) with a stable, index-ascending tie order."""
    s = np.asarray(s, np.float32)
    e = (np.exp(s.astype(np.float64)) + 1e-9).astype(np.float32)
    p = (e.astype(np.float64) / e.astype(np.float64).sum(-1, keepdims=True)).astype(np.float32)
    order = np.argsort(-p, axis=-1, kind="stable")
    return np.take_along_axis(p, order, -1), order


# |score - reference| bounds: the two embeddings may each differ by the north-star tolerance (1 - cos <= 1e-3 / 1e-2, i.e. an angle
# of sqrt(2 tol)); measured differences are 100x smaller, the bounds below are what the tolerance implies for a unit-vector dot product
SCORE_TOL = {"f16": 5e-3, "q4_0": 1e-1}


@pytest.mark.parametrize("ft", ["f16", "q4_0"])
def test_compare_and_zero_shot_label_match_live_reference(prod, ft):
    path = model_file("tiny", ft, prod)
    check_sha(path, golden("tiny")["sha_" + ft])
    u8 = _u8(*SCORING_IMAGE)
    g = reference_runs()
    ref = {k: g[k + "_" + ft] for k in ("cmp", "zsl_scores", "zsl_idx")}
    ctx = prod.load(path, 0)
    try:
        got_cmp = np.array([prod.compare_text_and_image(ctx, t, u8) for t in TEXTS], np.float32)
        sc, ix = prod.zero_shot_label_image(ctx, u8, TEXTS)
    finally:
        prod.free(ctx)
    print(ft, "compare max |d|", np.abs(got_cmp - ref["cmp"]).max(), "zsl max |dp|", np.abs(np.sort(sc) - np.sort(ref["zsl_scores"])).max())
    assert np.abs(got_cmp - ref["cmp"]).max() <= SCORE_TOL[ft]
    assert abs(sc.sum() - 1.0) < 1e-5 and np.all(np.diff(sc) <= 0)
    # probabilities per LABEL (undo both sorts), then the ranking wherever the reference's gaps exceed the tolerance
    p_got, p_ref = np.empty(len(TEXTS)), np.empty(len(TEXTS))
    p_got[ix], p_ref[ref["zsl_idx"]] = sc, ref["zsl_scores"]
    assert np.abs(p_got - p_ref).max() <= SCORE_TOL[ft]
    gaps = np.abs(np.diff(ref["zsl_scores"]))
    if gaps.min() > 4 * np.abs(p_got - p_ref).max():
        assert np.array_equal(ix, ref["zsl_idx"])


def _dev(prod, ctx, a):
    p = prod.lib.clip_b200_device_malloc(ctx, a.nbytes)
    assert p and prod.lib.clip_b200_memcpy_h2d(ctx, p, a.ctypes.data, a.nbytes)
    return p


@pytest.mark.parametrize("n_img,n_txt,k", [(5, 6, 6), (37, 1000, 5), (3, 4096, 4096), (2, 5000, 7), (4, 9000, 1024), (2, 5000, 3000)])
def test_zero_shot_batch_device_topk(prod, n_img, n_txt, k):
    """similarity + softmax + top-k on the device vs numpy; covers one sort slice, several slices + merge stages, the full ranking
    of one slice and the host-ranked fallback (k > 1024 with several slices)."""
    path = model_file("tiny", "q8_0", prod)
    ctx = prod.load(path, 0)
    d = prod.vision_hparams(ctx).projection_dim
    rng = np.random.default_rng(n_txt + k)
    img = (rng.standard_normal((n_img, d)) * 0.3).astype(np.float32)
    txt = (rng.standard_normal((n_txt, d)) * 0.3).astype(np.float32)
    try:
        d_i, d_t = _dev(prod, ctx, img), _dev(prod, ctx, txt)
        scores, idx = np.empty((n_img, k), np.float32), np.empty((n_img, k), np.int32)
        assert prod.lib.clip_b200_zero_shot_batch(ctx, d_i, n_img, d_t, n_txt, scores.ctypes.data_as(C.POINTER(C.c_float)),
                                                  idx.ctypes.data_as(C.POINTER(C.c_int)), k), prod.last_error()
        prod.lib.clip_b200_device_free(ctx, d_i)
        prod.lib.clip_b200_device_free(ctx, d_t)
    finally:
        prod.free(ctx)
    s = (img.astype(np.float64) @ txt.astype(np.float64).T).astype(np.float32)
    p_sorted, order = _softmax_sorted(s)
    assert np.allclose(scores, p_sorted[:, :k], rtol=2e-4, atol=1e-9)
    # identical ranking, except that labels whose probabilities agree to rounding may swap places
    p_full = (np.exp(s.astype(np.float64)) + 1e-9) / (np.exp(s.astype(np.float64)) + 1e-9).sum(1, keepdims=True)
    r, c = np.nonzero(idx != order[:, :k])
    for ri, ci in zip(r, c):
        assert np.isclose(p_full[ri, idx[ri, ci]], p_full[ri, order[ri, ci]], rtol=2e-4), (ri, ci)
    assert len(r) <= 0.02 * idx.size + 2
    assert (np.sort(idx, 1)[:, 1:] != np.sort(idx, 1)[:, :-1]).all()           # no index reported twice


@pytest.mark.parametrize("nq,ndb,k", [(1, 300, 10), (3, 20000, 10), (70, 4097, 1)])
def test_topk_search_raw_similarity(prod, nq, ndb, k):
    """nearest neighbours by raw dot product (the image-search use: examples/image-search/search.cpp:114-158)"""
    path = model_file("tiny", "q8_0", prod)
    ctx = prod.load(path, 0)
    d = prod.vision_hparams(ctx).projection_dim
    rng = np.random.default_rng(ndb)
    q = rng.standard_normal((nq, d)).astype(np.float32)
    db = rng.standard_normal((ndb, d)).astype(np.float32)
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    db /= np.linalg.norm(db, axis=1, keepdims=True)
    db[123 % ndb] = q[0]                                  # a planted exact match must come out first
    try:
        d_q, d_db = _dev(prod, ctx, q), _dev(prod, ctx, db)
        scores, idx = np.empty((nq, k), np.float32), np.empty((nq, k), np.int32)
        assert prod.lib.clip_b200_topk_search(ctx, d_q, nq, d_db, ndb, k, scores.ctypes.data_as(C.POINTER(C.c_float)),
                                              idx.ctypes.data_as(C.POINTER(C.c_int))), prod.last_error()
    finally:
        prod.free(ctx)
    s = q.astype(np.float64) @ db.astype(np.float64).T
    order = np.argsort(-s, axis=1, kind="stable")[:, :k]
    assert idx[0, 0] == 123 % ndb and abs(scores[0, 0] - 1.0) < 1e-5
    assert np.allclose(scores, np.take_along_axis(s, order, 1), atol=2e-6)
    agree = (idx == order).mean()
    assert agree > 0.95, agree                               # fp32 vs fp64 may swap near-equal neighbours


def test_zero_shot_images_single_gpu_equals_composition(prod):
    path = model_file("tiny", "f16", prod)
    ctx = prod.load(path, 0)
    try:
        imgs = sg.synth_images(7, 64, 21)
        labels = token_seqs(11, 300)
        for normalize in (False, True):
            sc, ix = prod.zero_shot_images(ctx, imgs, labels, 4, normalize=normalize)
            iv = prod.image_batch_encode(ctx, imgs, normalize=normalize)
            tv = prod.text_batch_encode(ctx, labels, normalize=normalize)
            p, order = _softmax_sorted(iv @ tv.T)
            assert np.array_equal(ix, order[:, :4])
            assert np.allclose(sc, p[:, :4], rtol=1e-4)
    finally:
        prod.free(ctx)


def test_text_encode_device_matches_host_entry(prod):
    path = model_file("tiny", "q4_0", prod)
    ctx = prod.load(path, 0)
    try:
        lens = np.array([77, 5, 2, 33, 16, 40], np.int32)
        T = 77
        ids = np.zeros((len(lens), T), np.int32)
        seqs = []
        for i, n in enumerate(lens):
            s = sg.synth_tokens(1, int(n), 50 + i)[0]
            ids[i, :n] = s
            seqs.append(s)
        host = prod.text_batch_encode(ctx, seqs)
        d = host.shape[1]
        d_ids, d_lens = _dev(prod, ctx, ids), _dev(prod, ctx, lens)
        d_out = prod.lib.clip_b200_device_malloc(ctx, host.nbytes)
        assert prod.lib.clip_b200_text_encode_device(ctx, d_ids, d_lens, len(lens), T, d_out, True), prod.last_error()
        got = np.empty_like(host)
        assert prod.lib.clip_b200_memcpy_d2h(ctx, got.ctypes.data, d_out, got.nbytes)
        assert one_minus_cos(got, host).max() < 1e-6         # padding to 77 instead of 80-rounded lengths: same rows, same math
        # bad arguments are refused, not clamped into garbage
        assert not prod.lib.clip_b200_text_encode_device(ctx, d_ids, d_lens, len(lens), 0, d_out, True)
        assert not prod.lib.clip_b200_text_encode_device(ctx, d_ids, d_lens, len(lens), 78, d_out, True)
        assert not prod.lib.clip_b200_text_encode_device(ctx, None, d_lens, len(lens), T, d_out, True)
        assert d * 0 == 0
    finally:
        prod.free(ctx)


def test_pinned_and_pageable_inputs_agree(prod):
    """clip_image_batch_encode from pinned buffers (direct async copies) and from pageable ones (what clip_image_preprocess
    returns; gathered into the library's pinned arena by host threads) must give identical bits."""
    path = model_file("tiny", "q4_0", prod)
    ctx = prod.load(path, 0)
    prod.lib.clip_b200_set_micro_batch(ctx, 48, 0)           # 3 passes, both staging buffers and their reuse
    try:
        n = 130
        imgs = sg.synth_images(n, 64, 9)
        pageable = prod.image_batch_encode(ctx, imgs)
        hp = prod.lib.clip_b200_host_malloc(imgs.nbytes)
        assert hp
        pinned_view = np.ctypeslib.as_array(C.cast(hp, C.POINTER(C.c_float)), shape=imgs.shape)
        pinned_view[:] = imgs
        pinned = prod.image_batch_encode(ctx, pinned_view)
        prod.lib.clip_b200_host_free(hp)
        assert np.array_equal(pageable, pinned)
    finally:
        prod.free(ctx)


def test_stopwatch_marks_are_per_context(prod):
    path = model_file("tiny", "q4_0", prod)
    a, b = prod.load(path, 0), prod.load(path, 0)
    try:
        assert prod.lib.clip_b200_mark(a, 0)
        prod.image_batch_encode(a, sg.synth_images(4, 64, 1))
        assert prod.lib.clip_b200_mark(a, 1)
        assert prod.lib.clip_b200_mark_elapsed_ms(a, 0, 1) > 0
        assert prod.lib.clip_b200_mark_elapsed_ms(b, 0, 1) == -1.0          # b never recorded: slots are not shared
    finally:
        prod.free(a)
        prod.free(b)
