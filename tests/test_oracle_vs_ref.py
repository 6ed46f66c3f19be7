"""Pin the plain-C restatement (oracle/lightctr_oracle.c) bit-for-bit against the unmodified reference.

What the reference computed in each comparison (oracle/_ref/libref.so, run by tests/golden/make_vs_ref_golden.py) is stored in
tests/golden/vs_ref.npz: float results as bit patterns, large arrays as SHA-256 digests, FM_Predict's printed line as text.  The
reference's data files are stored byte for byte (train_sparse.csv.xz, test_sparse.csv.xz), so the oracle parses the text the
reference parsed.  CPU-only."""
import hashlib
import lzma
import os
import shutil

import numpy as np
import pytest

from golden_util import GOLDEN, load_csr

GAUSS_CASES = ((1, 4096, 8), (3, 1001, 16), (9, 10, 4))


@pytest.fixture(scope="module")
def ref_out():
    with np.load(os.path.join(GOLDEN, "vs_ref.npz")) as z:
        return {k: z[k] for k in z.files}


@pytest.fixture(scope="module")
def data_files(tmp_path_factory):
    d = tmp_path_factory.mktemp("ref_data")
    out = []
    for name in ("train_sparse.csv", "test_sparse.csv"):
        with lzma.open(os.path.join(GOLDEN, name + ".xz"), "rb") as src, open(d / name, "wb") as dst:
            shutil.copyfileobj(src, dst)
        out.append(str(d / name))
    return out


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def test_rand_stream_matches_glibc(oracle_api):
    import ctypes
    libc = ctypes.CDLL("libc.so.6")
    L = oracle_api.lib()
    for seed in (1, 7, 12345, 0):
        libc.srand(seed)
        L.orc_srand(seed)
        a = [libc.rand() for _ in range(1000)]
        b = [L.orc_rand() for _ in range(1000)]
        assert a == b


def test_gauss_init_bit_exact(oracle_api, ref_out):
    for seed, n, k in GAUSS_CASES:
        ref = ref_out["gauss_%d_%d_%d" % (seed, n, k)]
        L = oracle_api.lib()
        L.orc_srand(seed)
        L.orc_gauss_reset()
        mine = np.zeros(n, np.float32)
        L.orc_init_V(mine, n, k)
        assert np.array_equal(ref, mine.view(np.uint32))


def test_dot_and_sigmoid_bit_exact(oracle_api, ref_out):
    rng = np.random.default_rng(0)
    L = oracle_api.lib()
    ref_dot = iter(ref_out["dot_bits"])
    for n in (1, 3, 4, 7, 8, 9, 10, 15, 16, 17, 31, 32, 33, 64, 100, 255):
        for _ in range(20):
            x = rng.standard_normal(n).astype(np.float32)
            y = rng.standard_normal(n).astype(np.float32)
            assert next(ref_dot) == np.float32(L.orc_dot(x, y, n)).view(np.uint32)
    xs = list(np.linspace(-20, 20, 4001, dtype=np.float32)) + [16.0, -16.0, 16.000002, -16.000002]
    for x, a in zip(xs, ref_out["sigmoid_bits"], strict=True):
        assert a == np.float32(L.orc_sigmoid(float(x))).view(np.uint32)


def test_loader_bit_exact(oracle_api, ref_out, data_files):
    d_ref = load_csr("train_sparse_csr.npz", field_cnt=68)  # the reference's own parse of the same file
    d = oracle_api.load(data_files[0], field_cnt=68)
    assert (d.rows, d.nnz, d.feature_cnt, d.field_cnt) == (1000, 281975, 233789, 68)
    assert (d.rows, d.nnz, d.feature_cnt, d.field_cnt) == tuple(ref_out["ffm_data_dims"])
    assert d_ref.feature_cnt == d.feature_cnt and d_ref.field_cnt == d.field_cnt
    for a, b in ((d.row_ptr, d_ref.row_ptr), (d.fid, d_ref.fid), (d.field, d_ref.field), (d.val, d_ref.val),
                 (d.label[:d.rows], d_ref.label)):
        assert np.array_equal(a, b)


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def test_fm_training_bit_exact(oracle_api, ref_out, data_files):
    k = 8
    train, test_path = data_files
    ds = oracle_api.load(train)
    Wi, Vi = oracle_api.init_params(1, ds.feature_cnt, k)
    assert _sha(Vi) == ref_out["fm_sha_V0"] and _sha(Wi) == ref_out["fm_sha_W0"]
    o = oracle_api.FMOracle(ds, k, Wi, Vi)
    for e in range(6):
        lo, ao = o.epoch()
        assert ref_out["fm_loss_bits"][e] == np.float32(lo).view(np.uint32), (e, lo)
        assert float(ref_out["fm_acc"][e]) == ao
    assert _sha(o.W) == ref_out["fm_sha_W"]
    assert _sha(o.V) == ref_out["fm_sha_V"]
    assert _sha(o.sumVX) == ref_out["fm_sha_S"]
    # FM_Predict with its quirks (predict/fm_predict.cpp)
    text = str(ref_out["fm_predict_text"])
    test = oracle_api.load_test(test_path, ds.feature_cnt)
    pctr, loss, correct, auc = oracle_api.predict(test, 0, k, o.W, o.V, o.sumVX, False)
    assert test.rows == 200
    ref_loss = float(text.split("likelihood = ")[1].split()[0])
    ref_acc = float(text.split("correct = ")[1].split()[0])
    ref_auc = float(text.split("auc = ")[1].split()[0])
    assert ref_loss in (float("%.6g" % loss), float("%.5g" % loss))
    assert float("%.5g" % (np.float32(correct) / np.float32(test.rows))) == pytest.approx(ref_acc, rel=1e-6)
    assert float("%.4f" % auc) == ref_auc


def test_ffm_training_bit_exact(oracle_api, ref_out, data_files):
    k, Fc = 4, 68
    train, test_path = data_files
    ds = oracle_api.load(train, field_cnt=Fc)
    Wi, Vi = oracle_api.init_params(1, ds.feature_cnt, k, Fc)
    assert _sha(Vi) == ref_out["ffm_sha_V0"]
    o = oracle_api.FFMOracle(ds, k, Wi, Vi)
    for e in range(3):
        lo, ao = o.epoch()
        assert ref_out["ffm_loss_bits"][e] == np.float32(lo).view(np.uint32), (e, lo)
        assert float(ref_out["ffm_acc"][e]) == ao
    assert _sha(o.W) == ref_out["ffm_sha_W"]
    assert _sha(o.V) == ref_out["ffm_sha_V"]
    text = str(ref_out["ffm_predict_text"])
    test = oracle_api.load_test(test_path, ds.feature_cnt)
    pctr, loss, correct, auc = oracle_api.predict(test, Fc, k, o.W, o.V, None, True)
    # cout keeps setprecision(5) from an earlier Predict() in the reference's process (fm_predict.cpp:73-74)
    ref_loss = float(text.split("likelihood = ")[1].split()[0])
    assert ref_loss in (float("%.6g" % loss), float("%.5g" % loss))
    assert float("%.4f" % auc) == float(text.split("auc = ")[1].split()[0])


def test_nfm_training_bit_exact(oracle_api, ref_out, data_files):
    k, H = 10, 32
    ds = oracle_api.load(data_files[0])
    o = oracle_api.NFMOracle(ds, k, H, seed=1)
    assert np.array_equal(ref_out["nfm_fc0_w_bits"], _bits(o.mlp.arrays("weight", 0)))
    assert np.array_equal(ref_out["nfm_fc0_mask"], o.mlp.arrays("mask", 0))
    for e in range(3):
        lo, ao = o.epoch()
        assert ref_out["nfm_loss_bits"][e] == np.float32(lo).view(np.uint32), (e, lo)
        assert float(ref_out["nfm_acc"][e]) == pytest.approx(ao, abs=1e-7)
    assert _sha(o.W) == ref_out["nfm_sha_W"]
    assert _sha(o.V) == ref_out["nfm_sha_V"]
    assert np.array_equal(ref_out["nfm_fc1_w_bits"], _bits(o.mlp.arrays("weight", 1)))
    assert np.array_equal(ref_out["nfm_fc1_b_bits"], _bits(o.mlp.arrays("bias", 1)))


def test_optimizer_units_bit_exact(oracle_api, ref_out):
    rng = np.random.default_rng(5)
    L = oracle_api.lib()
    n = 5000
    import ctypes as C

    def check(name, arrays):
        assert [_sha(x) for x in arrays] == list(ref_out["opt_%d_%s" % (trial, name)]), (trial, name)

    for trial in range(3):
        w = rng.standard_normal(n).astype(np.float32)
        g = (rng.standard_normal(n) * (rng.random(n) < 0.7)).astype(np.float32)
        s1 = np.abs(rng.standard_normal(n)).astype(np.float32) * (trial > 0)
        s2 = np.abs(rng.standard_normal(n)).astype(np.float32) * (trial > 0)
        b = [x.copy() for x in (s1, w, g)]
        L.orc_adagrad(n, b[1], b[2], b[0], 1000, 0.05)
        check("adagrad", b)
        b = [x.copy() for x in (s1, w, g)]
        L.orc_rmsprop(n, b[1], b[2], b[0], 1000, 0.05, 0.99)
        check("rmsprop", b)
        b = [x.copy() for x in (s1, s2, w, g)]
        L.orc_adadelta(n, b[2], b[3], b[0], b[1], 1000, 0.8)
        check("adadelta", b)
        b = [x.copy() for x in (s1, s2, w, g)]
        L.orc_ftrl(n, b[2], b[3], b[0], b[1], 0)
        check("ftrl", b)
        b = [x.copy() for x in (s1, s2, w, g)]
        it = C.c_size_t(trial * 3)
        L.orc_adam(n, b[2], b[3], b[0], b[1], C.byref(it), 1000, 0.05, 0.8, 0.999)
        check("adam", b)
