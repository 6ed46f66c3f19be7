"""Generate the fixtures of tests/test_oracle_vs_ref.py from the UNMODIFIED reference compiled in place (oracle/_ref/libref.so):

    python tests/golden/make_vs_ref_golden.py <reference checkout>

- train_sparse.csv.xz, test_sparse.csv.xz: the reference's data/train_sparse.csv and data/test_sparse.csv, byte for byte
  (xz-compressed), so that the oracle's parsers read the same text the reference reads;
- vs_ref.npz: what the reference computes in each comparison of the test -- float results as their uint32 bit patterns,
  large arrays (parameters after training, optimizer outputs) as the SHA-256 of their bytes, and the text FM_Predict prints.

Every call below mirrors one test, in the test file's order (FM_Predict leaves its cout precision to the FFM one)."""
import hashlib
import lzma
import os
import shutil
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import api  # noqa: E402

GAUSS_CASES = ((1, 4096, 8), (3, 1001, 16), (9, 10, 4))
DOT_NS = (1, 3, 4, 7, 8, 9, 10, 15, 16, 17, 31, 32, 33, 64, 100, 255)
SIGMOID_X = list(np.linspace(-20, 20, 4001, dtype=np.float32)) + [16.0, -16.0, 16.000002, -16.000002]


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def bits(x):
    return np.ascontiguousarray(x, np.float32).view(np.uint32)


def dot_inputs():
    rng = np.random.default_rng(0)
    for n in DOT_NS:
        for _ in range(20):
            yield rng.standard_normal(n).astype(np.float32), rng.standard_normal(n).astype(np.float32)


def optimizer_inputs():
    """-> per trial (w, g, s1, s2), the n = 5000 vectors of test_optimizer_units_bit_exact"""
    rng = np.random.default_rng(5)
    n = 5000
    for trial in range(3):
        w = rng.standard_normal(n).astype(np.float32)
        g = (rng.standard_normal(n) * (rng.random(n) < 0.7)).astype(np.float32)
        s1 = np.abs(rng.standard_normal(n)).astype(np.float32) * (trial > 0)
        s2 = np.abs(rng.standard_normal(n)).astype(np.float32) * (trial > 0)
        yield trial, w, g, s1, s2


def main(ref_root):
    data = os.path.join(ref_root, "data")
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "oracle", "ref", "REF=" + ref_root])
    for name in ("train_sparse.csv", "test_sparse.csv"):
        with open(os.path.join(data, name), "rb") as src, lzma.open(os.path.join(HERE, name + ".xz"), "wb", preset=9) as dst:
            shutil.copyfileobj(src, dst)
    train, test = os.path.join(data, "train_sparse.csv"), os.path.join(data, "test_sparse.csv")
    R = api.ref()
    out = {}

    for seed, n, k in GAUSS_CASES:
        v = np.zeros(n, np.float32)
        R.ref_gauss_fill(seed, n, k, v)
        out["gauss_%d_%d_%d" % (seed, n, k)] = bits(v)
    out["dot_bits"] = np.array([np.float32(R.ref_dot(x, y, len(x))).view(np.uint32) for x, y in dot_inputs()], np.uint32)
    out["sigmoid_bits"] = np.array([np.float32(R.ref_sigmoid(float(x))).view(np.uint32) for x in SIGMOID_X], np.uint32)

    # loader: the reference's parse of train_sparse.csv is tests/golden/train_sparse_csr.npz; confirm it still is
    t = api.RefTrainer("ffm", train, 4, field_cnt=68)
    d = t.data()
    z = np.load(os.path.join(HERE, "train_sparse_csr.npz"))
    assert np.array_equal(d.row_ptr, z["row_ptr"]) and np.array_equal(d.fid, z["fid"]) and np.array_equal(d.field, z["field"])
    assert np.array_equal(d.label, z["label"]) and np.all(d.val == 1.0) and len(z["val"]) == 0
    out["ffm_data_dims"] = np.array([d.rows, d.nnz, d.feature_cnt, d.field_cnt], np.int64)
    t.close()
    # the predict comparisons read the oracle's parse of test_sparse.csv: the committed one must be it
    zt = np.load(os.path.join(HERE, "test_sparse_csr.npz"))
    dt = api.load_test(test, int(out["ffm_data_dims"][2]))
    assert np.array_equal(dt.row_ptr, zt["row_ptr"]) and np.array_equal(dt.fid, zt["fid"])

    def curve(t, epochs):
        c = [t.epoch() for _ in range(epochs)]
        return bits([x[0] for x in c]), np.array([x[1] for x in c], np.float32)

    t = api.RefTrainer("fm", train, 8, seed=1, proc_cnt=1)
    W0, V0, _ = t.params()
    out["fm_sha_W0"], out["fm_sha_V0"] = sha(W0), sha(V0)
    out["fm_loss_bits"], out["fm_acc"] = curve(t, 6)
    W, V, S = t.params()
    out["fm_sha_W"], out["fm_sha_V"], out["fm_sha_S"] = sha(W), sha(V), sha(S)
    out["fm_predict_text"] = t.predict(test)
    t.close()

    t = api.RefTrainer("ffm", train, 4, seed=1, proc_cnt=1, field_cnt=68)
    _, V0, _ = t.params()
    out["ffm_sha_V0"] = sha(V0)
    out["ffm_loss_bits"], out["ffm_acc"] = curve(t, 3)
    W, V, _ = t.params()
    out["ffm_sha_W"], out["ffm_sha_V"] = sha(W), sha(V)
    out["ffm_predict_text"] = t.predict(test)
    t.close()

    t = api.RefTrainer("nfm", train, 10, seed=1, hidden=32)
    w, _, m = t.fc(0, 10, 32)
    out["nfm_fc0_w_bits"], out["nfm_fc0_mask"] = bits(w), m
    out["nfm_loss_bits"], out["nfm_acc"] = curve(t, 3)
    W, V, _ = t.params()
    out["nfm_sha_W"], out["nfm_sha_V"] = sha(W), sha(V)
    w, b, _ = t.fc(1, 32, 1)
    out["nfm_fc1_w_bits"], out["nfm_fc1_b_bits"] = bits(w), bits(b)
    t.close()

    for trial, w, g, s1, s2 in optimizer_inputs():
        n = len(w)
        a = [x.copy() for x in (s1, w, g)]
        R.ref_adagrad_update(n, 1000, 0.05, a[0], a[1], a[2])
        out["opt_%d_adagrad" % trial] = [sha(x) for x in a]
        a = [x.copy() for x in (s1, w, g)]
        R.ref_rmsprop_update(n, 1000, 0.05, 0.99, a[0], a[1], a[2])
        out["opt_%d_rmsprop" % trial] = [sha(x) for x in a]
        a = [x.copy() for x in (s1, s2, w, g)]
        R.ref_adadelta_update(n, 1000, 0.8, a[0], a[1], a[2], a[3])
        out["opt_%d_adadelta" % trial] = [sha(x) for x in a]
        a = [x.copy() for x in (s1, s2, w, g)]
        R.ref_ftrl_update(n, a[0], a[1], a[2], a[3])
        out["opt_%d_ftrl" % trial] = [sha(x) for x in a]
        a = [x.copy() for x in (s1, s2, w, g)]
        R.ref_adam_update(n, 1000, 0.05, 0.8, 0.999, trial * 3, a[0], a[1], a[2], a[3])
        out["opt_%d_adam" % trial] = [sha(x) for x in a]

    np.savez_compressed(os.path.join(HERE, "vs_ref.npz"), **{k: np.asarray(v) for k, v in out.items()})
    print("wrote", sorted(out))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
