"""CPU-only checks: the C-ABI library loads and exports every symbol include/crnn_ctc.h declares; the host-side
mirror of the reference API (config, factory, network surface, feed validation, accuracy) behaves like the reference.
No compute calls (no GPU here)."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_functions():
    src = open(os.path.join(ROOT, "include", "crnn_ctc.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(crnn_[a-z0-9_]+)\s*\(", src)))


def test_library_builds_and_exports_every_declared_symbol():
    import __graft_entry__ as g
    g.build()
    from lstm_ctc_ocr_b200 import _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    names = _header_functions()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), f"{n} declared in crnn_ctc.h but not exported"
        assert n in _lib.SIGNATURES, f"{n} has no ctypes signature"
    assert set(_lib.SIGNATURES) == set(names)
    L = _lib.load()
    assert L.crnn_version() >= 100
    assert L.crnn_status_string(1) == b"CRNN_INVALID_VALUE"


def test_no_gpu_means_loud_failure_not_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from lstm_ctc_ocr_b200 import CrnnError, engine
    from lstm_ctc_ocr_b200.session import Session
    with pytest.raises(CrnnError):
        engine.CrnnModel()
    with pytest.raises(CrnnError):
        Session()


def test_product_package_never_imports_oracle():
    pkg = os.path.join(ROOT, "lstm_ctc_ocr_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dp, f)).read()
                assert "oracle" not in txt.replace("oracle/", "").lower() or "import oracle" not in txt and "from oracle" not in txt, f


def test_factory_contract():
    from lstm_ctc_ocr_b200.lib.networks.factory import get_network
    tr, te = get_network("LSTM_train"), get_network("LSTM_test")
    for attr in ("data", "labels", "time_step_len", "labels_len", "keep_prob", "layers"):
        assert hasattr(tr, attr)
    assert not hasattr(te, "labels") and not hasattr(te, "labels_len")
    with pytest.raises(KeyError):
        get_network("LSTM_bogus")
    assert tr.get_output("logits").kind == "logits"
    assert tr.get_output("time_step_len") is tr.time_step_len
    with pytest.raises(KeyError):
        tr.get_output("nope")
    loss, dec = tr.build_loss()
    assert loss.kind == "loss" and dec.kind == "dense_decoded"
    with pytest.raises(KeyError):
        te.build_loss()                      # LSTM_test has no 'labels' layer (reference: get_output raises)


def test_reference_style_setup_chain_declares_the_compiled_network_and_anything_else_fails_loudly():
    """A `setup()` written in the reference's layer DSL (the chain of lib/networks/LSTM_train.py:22-38: feed / conv_single /
    max_pool / reshape_squeeze_layer / bi_lstm with the reference's argument order, defaults and names) runs unchanged on this
    Network and yields the same layer table as the shipped classes; a chain that differs from the topology compiled into
    libcrnnctc.so -- another width, a missing pool, a dropout, an off-path layer -- raises instead of computing something else."""
    from lstm_ctc_ocr_b200.lib.lstm.config import cfg
    from lstm_ctc_ocr_b200.lib.networks.LSTM_train import LSTM_train
    from lstm_ctc_ocr_b200.lib.networks.network import UnsupportedGraph
    from lstm_ctc_ocr_b200.lib.networks.factory import get_network

    def chain(net, conv2_out=128, with_pool3=True, pad5="VALID"):
        c = (net.feed("data")
             .conv_single(3, 3, 64, 1, 1, name="conv1", c_i=cfg.NCHANNELS)
             .max_pool(2, 2, 2, 2, padding="VALID", name="pool1")
             .conv_single(3, 3, conv2_out, 1, 1, name="conv2")
             .max_pool(2, 2, 2, 2, padding="VALID", name="pool2")
             .conv_single(3, 3, 256, 1, 1, name="conv3_1")
             .conv_single(3, 3, 256, 1, 1, name="conv3_2")
             .max_pool(1, 2, 1, 2, padding="VALID", name="pool2")
             .conv_single(3, 3, 512, 1, 1, name="conv4_1", bn=True)
             .conv_single(3, 3, 512, 1, 1, name="conv4_2", bn=True))
        if with_pool3:
            c = c.max_pool(1, 2, 1, 2, padding="VALID", name="pool3")
        c.conv_single(2, 2, 512, 1, 1, padding=pad5, name="conv5", relu=False).reshape_squeeze_layer(d=512, name="reshaped_layer")
        net.feed("reshaped_layer", "time_step_len").bi_lstm(cfg.TRAIN.NUM_HID, cfg.TRAIN.NUM_LAYERS, name="logits")

    class Mine(LSTM_train):
        variant = {}

        def setup(self):
            chain(self, **self.variant)

    net = Mine()
    ref = get_network("LSTM_train")
    assert sorted(net.layers) == sorted(ref.layers) and [op for op, _ in net._declared] == [op for op, _ in ref._declared]
    assert net._declared == ref._declared
    loss, dense = net.build_loss()
    assert loss.kind == "loss" and dense.kind == "dense_decoded" and net.get_output("logits").kind == "logits"
    for variant in (dict(conv2_out=96), dict(with_pool3=False), dict(pad5="SAME")):
        Mine.variant = variant
        with pytest.raises(UnsupportedGraph):
            Mine()
    Mine.variant = {}

    class Short(LSTM_train):
        def setup(self):
            self.feed("data").conv_single(3, 3, 64, 1, 1, name="conv1", c_i=cfg.NCHANNELS)
    with pytest.raises(UnsupportedGraph):
        Short().build_loss()                                         # a chain that stops early cannot be run
    n = get_network("LSTM_test")
    with pytest.raises(UnsupportedGraph):
        n.feed("conv5").dropout(0.5, name="dropout_layer")           # LSTM_train.py:35 is commented out in the reference
    with pytest.raises(UnsupportedGraph):
        n.feed("conv5").fc(10, name="fc")                            # off-path layer of the reference's DSL
    with pytest.raises(AttributeError):
        n.not_a_layer
    with pytest.raises(RuntimeError):
        n2 = get_network("LSTM_test"); n2.inputs = []; n2.max_pool(2, 2, 2, 2, name="p")   # no input fed (network.py:24-25)
    with pytest.raises(AssertionError):
        get_network("LSTM_test").feed("data").conv_single(3, 3, 64, 1, 1, name="conv1", c_i=1, padding="FULL")


def test_config_merge_and_set(tmp_path):
    from lstm_ctc_ocr_b200.lib.lstm import config as C
    assert C.cfg.NCLASSES == 64 and C.cfg.TRAIN.NUM_HID == 512 and C.cfg.POOL_SCALE == 4
    y = tmp_path / "lstm.yml"
    y.write_text("EXP_DIR: lstm_ctc\nTRAIN:\n  SOLVER: Adam\n  LEARNING_RATE: 0.0001\n  WEIGHT_DECAY: 0.00001\n  STEPSIZE: 2000\n")
    C.cfg_from_file(str(y))
    assert C.cfg.TRAIN.LEARNING_RATE == 1e-4 and C.cfg.TRAIN.WEIGHT_DECAY == 1e-5 and C.cfg.EXP_DIR == "lstm_ctc"
    C.cfg_from_list(["TRAIN.BATCH_SIZE", "32", "EXP_DIR", "foo"])
    assert C.cfg.TRAIN.BATCH_SIZE == 32 and C.cfg.EXP_DIR == "foo"
    bad = tmp_path / "bad.yml"
    bad.write_text("NOT_A_KEY: 1\n")
    with pytest.raises(KeyError):
        C.cfg_from_file(str(bad))
    bad.write_text("TRAIN:\n  STEPSIZE: abc\n")
    with pytest.raises(ValueError):
        C.cfg_from_file(str(bad))
    enc, dec = C.get_encode_decode_dict()
    assert enc["0"] == 1 and enc["Z"] == 62 and dec[11] == "a" and dec[0] == ""
    C.cfg.TRAIN.BATCH_SIZE = 64
    C.cfg.EXP_DIR = "default"


def test_shipped_run_configuration_holds_the_reference_hyper_parameters():
    """lstm_ctc_ocr_b200/lstm/lstm.yml (what train.sh / test.sh pass to --cfg) merges cleanly and carries the values the reference
    trains with (its lstm/lstm.yml: Adam, lr 1e-4, gamma 1.0 every 2000, wd 1e-5, display 100, snapshot 2000)."""
    import copy
    from lstm_ctc_ocr_b200.lib.lstm import config as C
    saved = copy.deepcopy(dict(C.cfg))
    try:
        C.cfg_from_file(os.path.join(ROOT, "lstm_ctc_ocr_b200", "lstm", "lstm.yml"))
        t = C.cfg.TRAIN
        assert (t.SOLVER, t.LEARNING_RATE, t.MOMENTUM, t.GAMMA, t.STEPSIZE, t.WEIGHT_DECAY) == ("Adam", 1e-4, 0.9, 1.0, 2000, 1e-5)
        assert (t.DISPLAY, t.SNAPSHOT_ITERS, t.SYNC_BN, t.BATCH_SIZE) == (100, 2000, True, 64)
        assert (C.cfg.EXP_DIR, C.cfg.LOG_DIR, C.cfg.NET_NAME, C.cfg.GPU_ID, C.cfg.DECODER) == ("lstm_ctc", "lstm_ctc", "LSTM", 0, "greedy")
    finally:
        for k, v in saved.items():
            C.cfg[k] = C.AttrDict(v) if isinstance(v, dict) else v
    for script in ("train.sh", "test.sh"):
        assert os.access(os.path.join(ROOT, script), os.X_OK)


def test_feed_validation():
    from lstm_ctc_ocr_b200.session import Session
    v = Session.validate_feed
    data = np.zeros((2, 88, 32), np.float32)
    ok = dict(tsl=np.array([21, 10], np.int32), labels=np.array([1, 2, 3], np.int32), labels_len=np.array([2, 1], np.int32))
    v(data, ok["tsl"], ok["labels"], ok["labels_len"])
    with pytest.raises(ValueError):
        v(np.zeros((2, 90, 32), np.float32), ok["tsl"], None, None)            # W % 4
    with pytest.raises(ValueError):
        v(data, np.array([22, 10], np.int32), None, None)                      # len > T = 21
    with pytest.raises(ValueError):
        v(data, ok["tsl"], np.array([1, 2, 63], np.int32), ok["labels_len"])   # 63 is never a target
    with pytest.raises(ValueError):
        v(data, ok["tsl"], np.array([0, 2, 3], np.int32), ok["labels_len"])    # 0 = blank
    with pytest.raises(ValueError):
        v(data, ok["tsl"], ok["labels"], np.array([2, 2], np.int32))           # sum mismatch


def test_accuracy_matches_oracle_definition():
    from lstm_ctc_ocr_b200.lib.lstm.utils.training import accuracy_calculation
    from oracle import crnn_oracle as O
    org = [[1, 2, 3], [4, 5], [6]]
    dec = np.array([[1, 2, 3, 0], [4, 0, 0, 0], [6, 0, 0, 0]])
    assert accuracy_calculation(org, dec, isPrint=False) == O.accuracy_calculation(org, dec) == 2 / 3


def test_synthetic_matches_oracle_generators():
    from lstm_ctc_ocr_b200 import synthetic
    from oracle import crnn_oracle as O
    a = synthetic.synth_batch(5, 40, seed=9, widths=[40, 33, 17, 40, 8])
    b = O.synth_batch(5, 40, seed=9, widths=[40, 33, 17, 40, 8])
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    pa, pb = synthetic.init_params(3), O.init_params(3, dtype=np.float32)
    assert list(pa) == list(pb) == [s[0] for s in O.param_specs()]
    for k in pa:
        assert np.array_equal(pa[k], pb[k]), k
    assert sum(v.size for v in pa.values()) == 7158592          # SURVEY §8(a)


def test_golden_fixture_is_reproducible_from_seeds():
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(ROOT, "tests", "golden", "make_golden.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    _, _, digest = mg.inputs()
    g = np.load(os.path.join(ROOT, "tests", "golden", "crnn_n4_w88.npz"))
    assert str(g["digest"]) == digest
    # oracle (fp64) still reproduces the committed outputs
    from oracle import crnn_oracle as O
    params, (data, lab, ll, tsl), _ = mg.inputs()
    p64 = O.to_torch({k: v.astype(np.float64) for k, v in params.items()})
    logits = O.forward(p64, data, tsl).numpy()
    assert np.allclose(logits, g["logits"], atol=1e-5)
    costs, _ = O.ctc_loss_np(logits, lab, ll, tsl)
    assert np.allclose(costs, g["costs"], rtol=1e-9)


def test_eval_line_preparation_and_cli_flags():
    from lstm_ctc_ocr_b200.lib.lstm.test import decodeRes, prepare_line
    from lstm_ctc_ocr_b200.lstm import test_net, train_net
    img = (np.arange(32 * 85) % 256).astype(np.uint8).reshape(32, 85)
    data, tsl = prepare_line(img)
    assert data.shape == (1, 88, 32) and data.dtype == np.float32            # right-padded to a multiple of 4
    assert tsl.tolist() == [85 // 4 - 1] and np.all(data[0, 85:] == 0)
    assert np.allclose(data[0, :85, :], img.T / 255.0)
    assert "".join(decodeRes([1, 0, 11, 37, 0])) == "0aA"
    a = train_net.parse_args(["--network=LSTM_train", "--cfg=./lstm/lstm.yml", "--restore=0", "--set", "TRAIN.BATCH_SIZE", "32"])
    assert a.network_name == "LSTM_train" and a.restore == 0 and a.set_cfgs == ["TRAIN.BATCH_SIZE", "32"] and a.max_iters == 1000000
    b = test_net.parse_args(["--network=LSTM_test", "--testDir", "x"])
    assert b.test_dir == "x" and b.restore == 1


def test_data_layer_batch_contract():
    """lib/lstm/utils/gen.py: groupBatch restates gen.py:41-67 -- resize to height 32 keeping aspect (nw = int(32/h*w)),
    time_step = nw//4 - 1, right-pad with 0.0 to a multiple of 4, /255, transpose to [W, 32]; get_batch yields the 4-tuple."""
    from lstm_ctc_ocr_b200.lib.lstm.utils import gen
    from lstm_ctc_ocr_b200.lib.lstm.config import cfg
    rng = np.random.default_rng(0)
    imgs = [rng.integers(1, 256, size=(60, 160), dtype=np.uint8), rng.integers(1, 256, size=(60, 100), dtype=np.uint8),
            rng.integers(1, 256, size=(32, 57), dtype=np.uint8)]
    batch, lab, ll, ts = gen.groupBatch(imgs, ["ab1", "Zz", "0"])
    nws = [int(32 / 60 * 160), int(32 / 60 * 100), 57]                       # 85, 53, 57
    W = int(np.ceil(max(nws) / 4) * 4)                                        # 88 (the stock captcha case, SURVEY section 2 #7)
    assert W == 88 and all(b.shape == (W, cfg.NUM_FEATURES) and b.dtype == np.float32 for b in batch)
    assert ts == [nw // 4 - 1 for nw in nws] == [20, 12, 13]
    assert ll == [3, 2, 1] and lab == [gen.encode_maps[c] for c in "ab1Zz0"] and min(lab) >= 1 and max(lab) <= 62
    for b, nw in zip(batch, nws):
        assert float(b.max()) <= 1.0 and float(b.min()) >= 0.0
        assert not b[nw:].any() and b[:nw].any()                              # exact zeros right of the resized image
    # the unresized third image: [W,32] is the transpose of the [32,W] pixel grid / 255
    assert np.allclose(batch[2][:57], imgs[2].astype(np.float32).T / 255.0)
    # generator contract (render or contract-identical fallback): N arrays [W,32], flat labels, lengths, time steps <= W/4-1
    for render in (False, True):
        img_list, flat, lens, steps = next(gen.get_batch(num_workers=2, batch_size=5, render=render))
        assert len(img_list) == 5 and len(lens) == 5 and len(steps) == 5 and len(flat) == sum(lens)
        Wb = img_list[0].shape[0]
        assert Wb % 4 == 0 and all(a.shape == (Wb, 32) for a in img_list) and max(steps) <= Wb // 4 - 1
        assert all(cfg.MIN_LEN <= l <= cfg.MAX_LEN for l in lens) and 1 <= min(flat) and max(flat) <= 62


# ---------------------------------------------------------------------------------------------------------------------------
# beam-search decoder (host side of the C ABI: runs without a GPU) vs the oracle's restatement of TF's CTCBeamSearchDecoder
# ---------------------------------------------------------------------------------------------------------------------------
def _beam(x, il, **kw):
    from lstm_ctc_ocr_b200 import engine
    out, out_len, nlp = engine.ctc_beam_search(x, il, **kw)
    return [out[i, :out_len[i]].tolist() for i in range(len(il))], nlp


def test_beam_search_rule_table():
    """Same rule table as tests/test_oracle.py::test_beam_search_restatement_rule_table_and_defined_deviation (network.py:656)."""
    def onehot(seq):
        x = np.zeros((len(seq), 1, 64), np.float32)
        for t, a in enumerate(seq):
            x[t, 0, a] = 8.0
        return x
    beam = lambda seq, **kw: _beam(onehot(seq), [len(seq)], **kw)[0][0]
    assert beam([1, 2, 3, 4]) == [1, 2, 3, 4]
    assert beam([63, 63, 63]) == []
    assert beam([5, 5, 63, 5, 0, 7], merge_repeated=False) == [5, 5, 7]
    assert beam([5, 5, 63, 5, 0, 7]) == [5, 7]                   # merge_repeated collapses the decoded double 5
    assert beam([3, 63, 3, 63, 4]) == [3, 4]
    assert beam([0, 1, 0, 2], strip=-1) == [0, 1, 0, 2]          # class 0 is an ordinary label to the decoder; the solver strips it


@pytest.mark.parametrize("kind,seed", [("peaked", 2), ("soft", 5), ("flat", 7)])
def test_beam_search_matches_oracle_restatement(kind, seed):
    """crnn_ctc_beam_search == oracle.beam_search_decode (width 100, blank 63, merge_repeated) on peaked, soft and flat
    frames with ragged lengths, including zero-length utterances; log-probability of the best prefix is finite."""
    from oracle import crnn_oracle as O
    def _peaked_lines(n, T, seed, margin=6.0):        # frames peaked at a path with CTC blanks (0), decoder blanks (63), repeats
        r = np.random.default_rng(seed)
        path = r.choice(64, size=(T, n), p=np.r_[0.25, np.full(62, 0.65 / 62), 0.10])
        rep = r.random((T, n)) < 0.3
        for t in range(1, T):
            path[t] = np.where(rep[t], path[t - 1], path[t])
        y = r.standard_normal((T, n, 64))
        y[np.arange(T)[:, None], np.arange(n)[None, :], path] += margin
        return y
    rng = np.random.default_rng(seed)
    T, N = 19, 10
    if kind == "peaked":
        x = _peaked_lines(N, T, seed=seed)
    elif kind == "soft":
        x = _peaked_lines(N, T, seed=seed, margin=2.0)
    else:
        x = rng.standard_normal((T, N, 64)) * 0.3
    x = x.astype(np.float32)
    il = rng.integers(0, T + 1, size=N).astype(np.int32)
    il[0] = T; il[1] = 0
    for merge in (True, False):
        ref = O.beam_search_decode(x, il, beam_width=100, merge_repeated=merge)
        got, nlp = _beam(x, il, beam_width=100, merge_repeated=merge)
        assert got == ref, (kind, merge)
        assert np.isfinite(nlp).all() and nlp[1] == 0.0
    # a narrow beam still agrees with the oracle at the same width (exercises the full-list eviction path)
    assert _beam(x, il, beam_width=3)[0] == O.beam_search_decode(x, il, beam_width=3)


@pytest.mark.parametrize("seed", range(6))
def test_beam_search_ties_and_narrow_beams_match_oracle(seed):
    """The decoder keeps the beam in a heap, visits only the classes that can still enter a full list and creates children on
    demand; TF's results depend on visiting ORDER (which of several equal totals is the bottom, a branch evicted mid-frame
    still being expanded unless its parent's visit wipes it), so the restatement is compared on the inputs where order shows:
    quantised logits (exact ties), all-equal frames, few classes, beam widths 1..7 that evict constantly, both merge modes."""
    from oracle import crnn_oracle as O
    rng = np.random.default_rng(100 + seed)
    C = int(rng.choice([3, 6, 17]))
    T, N = int(rng.integers(4, 15)), 8
    kind = seed % 3
    if kind == 0:
        x = np.round(rng.standard_normal((T, N, C)) * 2) / 2
    elif kind == 1:
        x = rng.integers(0, 2, size=(T, N, C)).astype(np.float64) * float(rng.choice([1, 5]))
        x[T // 2] = 0.0                                           # an all-equal frame
    else:
        x = rng.standard_normal((T, N, C)) * float(rng.choice([0.3, 3.0]))
    x = x.astype(np.float32)
    il = rng.integers(0, T + 1, size=N).astype(np.int32)
    il[0] = T
    for bw in (1, 2, 3, 5, 7, 100):
        for merge in (True, False):
            ref = O.beam_search_decode(x, il, beam_width=bw, merge_repeated=merge, strip=-1)
            assert _beam(x, il, beam_width=bw, merge_repeated=merge, strip=-1)[0] == ref, (C, T, bw, merge)


def test_beam_search_reproduces_tensorflows_own_known_answer():
    """crnn_ctc_beam_search on the vector TensorFlow's ctc_decoder_ops_test.py::testCTCDecoderBeamSearch pins
    (tests/golden/third_party_kats.py): top path [1, 0] at beam_width 2 (6 classes, blank 5, unnormalised log p + 2), the
    most probable labelling [0, 1, 0] at every other width.  The product decoder against a number held by the project it
    replaces (network.py:656), not against the oracle."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("third_party_kats", os.path.join(ROOT, "tests", "golden", "third_party_kats.py"))
    K = importlib.util.module_from_spec(spec); spec.loader.exec_module(K)
    x, il = K.beam_case()
    x = x.astype(np.float32)
    assert _beam(x, il, beam_width=K.BEAM_WIDTH, merge_repeated=True, strip=-1)[0] == [K.BEAM_TOP_PATHS[0]]
    for bw in (1, 3, 100):
        assert _beam(x, il, beam_width=bw, merge_repeated=True, strip=-1)[0] == [K.BEAM_TOP_PATHS[1]]


def test_beam_search_rejects_bad_lengths():
    from lstm_ctc_ocr_b200 import engine
    from lstm_ctc_ocr_b200._lib import CrnnError
    x = np.zeros((4, 2, 64), np.float32)
    with pytest.raises(CrnnError):
        engine.ctc_beam_search(x, [5, 1])


# ---------------------------------------------------------------------------------------------------------------------------
# data path, SURVEY 8(f)2: width-bucketing sampler, rank-distinct streams, prefetching feeder (gen.py:112-128 replacement)
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("render", [True, False])
def test_bucket_sampler_contract(render):
    """BASELINE configs[3]: every batch comes from ONE bucket of W in {80,160,256}, is padded to that width, and every line's
    true width lies in (previous bucket, W] (rendered: resized width; synthetic: SURVEY 8(d), at least one line of width W)."""
    from lstm_ctc_ocr_b200.lib.lstm.utils import gen
    s = gen.BucketSampler(batch_size=12, render=render, seed=5, rank=0, world=1)
    for k, W in zip(range(3), gen.BUCKETS):
        assert s.bucket_of(k) == W and s.bucket_of(k + 3) == W
        imgs, flat, lens, steps = s.batch(k)
        lo = max([b for b in gen.BUCKETS if b < W] or [0])
        assert len(imgs) == 12 and all(a.shape == (W, 32) and a.dtype == np.float32 for a in imgs)
        assert len(flat) == sum(lens) and 1 <= min(flat) and max(flat) <= 62
        assert max(steps) <= W // 4 - 1
        widths = [int(np.nonzero(a.any(axis=1))[0].max()) + 1 for a in imgs]        # last non-zero column + 1
        if render:
            assert all(lo // 4 - 1 <= st <= W // 4 - 1 for st in steps)
            assert all(w <= W for w in widths) and max(widths) > lo
        else:
            assert max(steps) == W // 4 - 1 and all(lo < w <= W for w in widths)
    # deterministic: batch k is a pure function of (seed, k, rank, world)
    a, b = s.batch(4), gen.BucketSampler(batch_size=12, render=render, seed=5, rank=0, world=1).batch(4)
    assert all(np.array_equal(x, y) for x, y in zip(a[0], b[0])) and a[1:] == b[1:]


def test_data_parallel_ranks_draw_different_batches():
    """ADVICE r1 (gen.py:82): the synthetic fallback seeded every rank identically.  batch k of rank r now uses seed
    base + k*world + r: ranks differ, and the union over ranks at step k never repeats a batch of another step."""
    from lstm_ctc_ocr_b200.lib.lstm.utils import gen
    for render in (False, True):
        b0 = gen.make_batch(0, 6, render, seed=3, rank=0, world=2)
        b1 = gen.make_batch(0, 6, render, seed=3, rank=1, world=2)
        assert b0[1] != b1[1]
    seeds = {gen.batch_seed(k, 3, r, 4) for k in range(50) for r in range(4)}
    assert len(seeds) == 200
    g0 = gen.generator(batch_size=4, render=False, seed=3, rank=0, world=2)
    g1 = gen.generator(batch_size=4, render=False, seed=3, rank=1, world=2)
    assert next(g0)[1] != next(g1)[1]


def test_prefetch_feeder_delivers_the_stream_in_order():
    """PrefetchFeeder (stands in for GeneratorEnqueuer + multiprocessing.Queue, gen.py:112-128): render processes, batches
    delivered in order as views of a ring of slots; a view stays intact until `depth` further batches were taken."""
    from lstm_ctc_ocr_b200.lib.lstm.utils import gen
    arg_fn = lambda k: dict(k=k, batch_size=6, render=True, seed=11, rank=0, world=1, bucket=gen.BUCKETS[k % 3])
    ref = [gen.make_batch(**arg_fn(k)) for k in range(7)]
    for workers in (0, 2):
        f = gen.PrefetchFeeder(arg_fn, num_workers=workers, depth=3, max_width=256, batch_size=6)
        try:
            held = []
            for k in range(7):
                view, lab, ll, tsl = next(f)
                assert isinstance(view, np.ndarray) and view.shape == (6, gen.BUCKETS[k % 3], 32) and view.flags.c_contiguous
                assert np.array_equal(view, np.stack(ref[k][0]))
                for got, want in zip((lab, ll, tsl), ref[k][1:]):             # int32 arrays of the data layer's lists
                    assert isinstance(got, np.ndarray) and got.dtype == np.int32 and got.tolist() == list(want)
                held.append((k, view))
                for kk, v in held[-3:]:                                         # the last `depth` views are still valid
                    assert np.array_equal(v, np.stack(ref[kk][0]))
        finally:
            f.close()
    # the reference entry point: get_batch(num_workers=N, batch_size=B) -> iterator of data-layer tuples
    it = gen.get_batch(num_workers=2, batch_size=5, render=True, seed=11)
    try:
        imgs, flat, lens, steps = next(it)
        assert len(imgs) == 5 and len(flat) == sum(lens) and len(steps) == 5
    finally:
        if hasattr(it, "close"):
            it.close()


def test_prefetch_feeder_peek_does_not_reorder_or_skip():
    """peek() (what Session.attach_feeder uses to start the next batch's host->device copy early) hands back the batch the next
    next() delivers; `delivered` counts what the consumer holds."""
    from lstm_ctc_ocr_b200.lib.lstm.utils import gen
    arg_fn = lambda k: dict(k=k, batch_size=4, render=False, seed=5, rank=0, world=1, bucket=gen.BUCKETS[k % 3])
    ref = [gen.make_batch(**arg_fn(k)) for k in range(6)]
    f = gen.PrefetchFeeder(arg_fn, num_workers=0, depth=2, max_width=256, batch_size=4, pinned=False, keep=2)
    try:
        assert f.delivered == 0
        for k in range(6):
            if k % 2 == 0:
                pv = f.peek()
                assert f.peek() is pv and f.delivered == k
            view, lab, ll, tsl = next(f)
            assert f.delivered == k + 1
            assert np.array_equal(np.asarray(view), np.stack(ref[k][0])) and list(lab) == list(ref[k][1])
            if k % 2 == 0:
                assert view is pv[0]
    finally:
        f.close()


def test_host_copy_pool_moves_every_byte_for_any_size_and_thread_count():
    """crnn_host_copy: the persistent thread pool behind crnn_forward_pageable (pageable numpy batch -> page-locked staging).  No GPU
    needed.  Sizes around the share / page boundaries, thread counts beyond the pool size, many back-to-back calls (a lost wake-up
    would hang here under the test timeout, not on the GPU box)."""
    from lstm_ctc_ocr_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(0)
    src = rng.integers(0, 255, size=(40 << 20) + 77, dtype=np.uint8)
    dst = np.zeros_like(src)
    sizes = [0, 1, 4095, 4096, (1 << 20) - 1, 1 << 20, (1 << 20) + 1, 3 * (1 << 20) + 4097, (33 << 20) + 5, src.size]
    for rep in range(3):
        for n in sizes:
            for threads in (1, 2, 3, 8, 16, 64):
                dst[:n + 16] = 0 if n + 16 <= dst.size else 0
                assert lib.crnn_host_copy(dst.ctypes.data, src.ctypes.data, n, threads) == 0
                assert np.array_equal(dst[:n], src[:n]) and (n + 16 > dst.size or not dst[n:n + 16].any()), (n, threads)
    for i in range(400):                                                        # back-to-back small-large alternation
        n = int(rng.integers(1 << 20, 6 << 20))
        t = int(rng.integers(2, 12))
        dst[:n] = 0
        assert lib.crnn_host_copy(dst.ctypes.data, src.ctypes.data, n, t) == 0
        assert dst[n - 1] == src[n - 1] and dst[0] == src[0] and dst[n // 2] == src[n // 2]


# ---------------------------------------------------------------------------------------------------------------------------
# bench.py contract pieces that run without a GPU
# ---------------------------------------------------------------------------------------------------------------------------
def test_bench_reference_arm_prints_the_contract_line_and_ours_refuses_without_a_gpu():
    """`bench.py --impl reference` (the CPU port of the reference path, rank 0 only) prints ONE JSON line with the main arm's
    metric / unit / workload keys, `impl`, `cpu_baseline` and a zero-copy `e2e`; a non-zero rank prints nothing and exits 0;
    the product arm exits non-zero on a box without CUDA instead of measuring a fallback."""
    import json
    import subprocess
    import sys
    import torch
    bench = os.path.join(ROOT, "bench.py")
    env = dict(os.environ, OMP_NUM_THREADS="4")
    p = subprocess.run([sys.executable, bench, "--impl", "reference", "--workload", "c1shape", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, env=env, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "text-line images/sec (fwd+CTC loss)" and d["unit"] == "images/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["n_gpus"] == 1 and d["steps"] == 1
    assert d["config"]["batch_per_gpu"] == 32 and d["config"]["width"] == 100 and d["config"]["T"] == 24
    assert d["config"]["reference_sample_per_step"] == 32
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == d["value"] and cb["cores"] >= 1 and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # under torchrun only rank 0 works
    p = subprocess.run([sys.executable, bench, "--impl", "reference", "--workload", "c1shape", "--steps", "1", "--warmup", "1", "--gpus", "2"],
                       capture_output=True, text=True, env=dict(env, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2"), timeout=600)
    assert p.returncode == 0 and not [l for l in p.stdout.splitlines() if l.startswith("{")]
    if not torch.cuda.is_available():
        p = subprocess.run([sys.executable, bench, "--steps", "1", "--warmup", "1"], capture_output=True, text=True, env=env, timeout=600)
        assert p.returncode != 0 and "no CPU fallback" in (p.stderr + p.stdout)


def test_bench_refuses_fewer_than_one_timed_step():
    import subprocess
    import sys
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0", "--dump-outputs", "unused"],
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 2 and "--steps must be at least 1" in p.stderr


def build_c_abi_smoke(tmp_path):
    """gcc -std=c99 tests/c_abi/abi_smoke.c against include/crnn_ctc.h and the in-tree libcrnnctc.so; returns the binary's path."""
    import subprocess
    from lstm_ctc_ocr_b200 import _lib
    _lib.load()                                                     # builds the library if it is stale
    libdir = os.path.join(ROOT, "lstm_ctc_ocr_b200")
    exe = str(tmp_path / "abi_smoke")
    cmd = ["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I" + os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "c_abi", "abi_smoke.c"), "-o", exe, "-L" + libdir, "-lcrnnctc", "-lm", "-Wl,-rpath," + libdir]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr[-3000:]
    return exe


def test_c_abi_is_usable_from_plain_c(tmp_path):
    """The drop-in boundary is a C ABI: a C99 translation unit that includes only include/crnn_ctc.h compiles warning-free,
    links against libcrnnctc.so and drives the GPU-free entry points (status strings, host beam search on TensorFlow's known
    answer, host copy pool); crnn_model_create fails with a status + message where there is no CUDA device."""
    import subprocess
    import torch
    exe = build_c_abi_smoke(tmp_path)
    p = subprocess.run([exe] + (["--gpu"] if torch.cuda.is_available() else []), capture_output=True, text=True, timeout=300)
    assert p.returncode == 0 and "FAIL" not in p.stdout and p.stdout.count("ok ") >= 8, p.stdout + p.stderr
    # crnn_config as the C compiler lays it out == the ctypes mirror the Python side passes to crnn_model_create
    from lstm_ctc_ocr_b200._lib import CrnnConfig
    import ctypes
    layout = [int(v) for v in next(l for l in p.stdout.splitlines() if l.startswith("layout crnn_config")).split()[2:]]
    assert layout == [ctypes.sizeof(CrnnConfig)] + [getattr(CrnnConfig, f).offset for f, _ in CrnnConfig._fields_], layout


def test_ctypes_binding_matches_the_header_prototypes():
    """Every prototype of include/crnn_ctc.h against the argtypes / restype table of lstm_ctc_ocr_b200/_lib.py: same set of names,
    same number of parameters, and per parameter the same class (pointer / int / float / size_t / int64) -- a drifted binding would
    otherwise only show up as garbage arguments on the GPU box."""
    import ctypes
    from lstm_ctc_ocr_b200 import _lib
    src = open(os.path.join(ROOT, "include", "crnn_ctc.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    src = re.sub(r"typedef\s+\w[\w\s\*]*\(\s*\*\s*\w+\s*\)\s*\([^;]*\)\s*;", "", src)         # callback typedefs are not entry points
    protos = dict((m.group(2), (m.group(1).strip(), m.group(3))) for m in
                  re.finditer(r"(?m)^\s*((?:const\s+)?[\w]+\s*\**)\s*(crnn_[a-z0-9_]+)\s*\(([^;{]*)\)\s*;", src))
    assert set(protos) == set(_lib.SIGNATURES), sorted(set(protos) ^ set(_lib.SIGNATURES))

    def kind_of_c(decl):
        decl = decl.strip()
        if "*" in decl or "[" in decl or re.search(r"\b(crnn_stream_t|crnn_\w+_fn)\b", decl):
            return "ptr"
        base = re.sub(r"\bconst\b", "", decl).split()
        t = base[0] if base else decl
        return {"int": "int", "float": "float", "size_t": "size_t", "int64_t": "int64"}.get(t, t)

    def kind_of_ctypes(t):
        if t in (ctypes.c_void_p, ctypes.c_char_p) or isinstance(t, type(ctypes.POINTER(ctypes.c_int))) and issubclass(t, ctypes._Pointer):
            return "ptr"
        return {ctypes.c_int: "int", ctypes.c_float: "float", ctypes.c_size_t: "size_t", ctypes.c_int64: "int64"}[t]

    for name, (ret, params) in protos.items():
        res, args = _lib.SIGNATURES[name]
        plist = [p for p in (q.strip() for q in params.split(",")) if p and p != "void"]
        assert len(plist) == len(args), (name, plist, args)
        for i, (p, a) in enumerate(zip(plist, args)):
            assert kind_of_c(p) == kind_of_ctypes(a), (name, i, p, a)
        assert kind_of_c(ret + " x") == kind_of_ctypes(res), (name, ret, res)


def test_warpctc_tensorflow_import_name_resolves_to_the_drop_in():
    """`import warpctc_tensorflow` (the reference's binding import, network.py:6) finds the shim at the repository root; `ctc`
    takes the reference's keyword names (network.py:653-654) and refuses to run without a GPU instead of falling back."""
    import inspect
    import torch
    import warpctc_tensorflow
    from lstm_ctc_ocr_b200 import warpctc
    from lstm_ctc_ocr_b200._lib import CrnnError
    assert warpctc_tensorflow.ctc is warpctc.ctc
    params = list(inspect.signature(warpctc_tensorflow.ctc).parameters)
    assert params == ["activations", "flat_labels", "label_lengths", "input_lengths", "blank_label"]
    assert inspect.signature(warpctc_tensorflow.ctc).parameters["blank_label"].default == 0
    if not torch.cuda.is_available():
        with pytest.raises(CrnnError):
            warpctc_tensorflow.ctc(activations=np.zeros((3, 1, 64), np.float32), flat_labels=[1], label_lengths=[1], input_lengths=[3])
