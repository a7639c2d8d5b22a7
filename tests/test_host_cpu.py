"""Host-side logic of the polus-shaped API (no GPU): utils/core/data/schedulers/labels/callbacks/bucket plan.
Several cases mirror the reference's own unit tests (tests/test_utils.py, tests/test_core.py, tests/test_data.py)."""
import json
import os

import numpy as np
import pytest


# ------------------------------------------------------------------ utils (reference tests/test_utils.py)
def test_singleton_identity():
    from polus_b200.utils import Singleton

    class A(metaclass=Singleton):
        pass

    class B(metaclass=Singleton):
        pass
    assert A() is A() and B() is B() and A() is not B()


def test_flatten_dict_cases():
    from polus_b200.utils import flatten_dict
    assert flatten_dict({"a": 1, "b": {"c": 2, "d": {"e": 3}}}) == {"a": 1, "c": 2, "e": 3}
    assert flatten_dict({}) == {}
    # duplicate key: the later occurrence overrides (reference tests/test_utils.py:26-55)
    assert flatten_dict({"a": 1, "b": {"a": 2}}) == {"a": 2}
    assert flatten_dict({"b": {"a": 2}, "a": 1}) == {"a": 1}


def test_is_jsonable_and_tensor_roundtrip():
    from polus_b200.utils import complex_json_deserializer, complex_json_serializer, is_jsonable, merge_dicts, unique
    assert is_jsonable({"a": [1, 2, "x"]}) and not is_jsonable({"a": {1, 2}})
    mask = np.ones((4, 4), np.float32)
    mask[1, 3] = 0
    data = {"model": {"mask_impossible_transitions": mask, "hidden": 128}, "name": "m"}
    back = complex_json_deserializer(json.loads(json.dumps(complex_json_serializer(data))))
    assert back["name"] == "m" and back["model"]["hidden"] == 128
    assert np.array_equal(back["model"]["mask_impossible_transitions"], mask)
    assert merge_dicts({"a": 1}, {"b": 2}, {"a": 3}) == {"a": 3, "b": 2}
    assert unique([1, 2, 2, 3, 1]) == [1, 2, 3]
    with pytest.raises(ValueError):
        complex_json_serializer({"x": object()})


def test_jit_flag_roundtrip(monkeypatch):
    from polus_b200.core import get_jit_compile, set_jit_compile
    monkeypatch.delenv("POLUS_JIT", raising=False)
    assert get_jit_compile() is False  # default (reference tests/test_core.py)
    set_jit_compile(True)
    assert get_jit_compile() is True
    set_jit_compile(False)
    assert get_jit_compile() is False


def test_execute_if():
    from polus_b200.core import execute_if

    class X:
        flag = True

        @execute_if("flag")
        def f(self):
            return 1
    x = X()
    assert x.f() == 1
    x.flag = False
    assert x.f() is None


# ------------------------------------------------------------------ data (reference tests/test_data.py:28-80)
def _gen(n=1000):
    def source_generator():
        for i in range(n):
            yield {"id": i, "text": np.full(4, i, np.int32)}
    return source_generator


def test_dataloader_order_count_and_dataset_verbs():
    from polus_b200.data import DataLoader
    dl = DataLoader(_gen())
    assert [s["id"] for s in dl] == list(range(1000))
    assert dl.get_n_samples() == 1000
    ds = dl.to_tfDataset()
    assert dl.shapes["text"] == (4,) and dl.shapes["id"] == ()
    assert [int(s["id"]) for s in ds] == list(range(1000))
    b = list(ds.batch(128, drop_remainder=True))
    assert len(b) == 7 and b[0]["text"].shape == (128, 4) and b[0]["id"][5] == 5
    assert len(list(ds.batch(128))) == 8
    mapped = ds.map(lambda d: (d["text"].astype(np.float32), d["id"])).batch(10)
    x, y = next(iter(mapped))
    assert x.shape == (10, 4) and x.dtype == np.float32 and list(y) == list(range(10))
    shuffled = [int(s["id"]) for s in ds.shuffle(1000, seed=0)]
    assert sorted(shuffled) == list(range(1000)) and shuffled != list(range(1000))
    assert ds.batch(100).cardinality() == -2  # unknown: generator-backed, like tf.data


def test_dynamic_shape_inference():
    from polus_b200.core import find_dtype_and_shapes

    def g():
        for i in range(1, 20):
            yield {"x": np.zeros((i, 3), np.float32)}
    dt, sh = find_dtype_and_shapes(g(), k=10)
    assert sh["x"] == (None, 3) and dt["x"] == np.float32
    with pytest.raises(ValueError):
        find_dtype_and_shapes(iter([1, 2, 3]), k=2)


def test_shard_rule_is_i_mod_n_before_batching():
    """polus/data.py:94-96: sample i -> rank i mod N, applied before the user batches."""
    from polus_b200.data import Dataset
    ds = Dataset.from_generator(lambda: iter(range(10)))
    assert list(ds.shard(4, 1)) == [1, 5, 9]
    assert [b.tolist() for b in ds.shard(2, 0).batch(2)] == [[0, 2], [4, 6], [8]]


# ------------------------------------------------------------------ schedule / labels
def test_warmup_scheduler_matches_hf_torch_polynomial_schedule():
    """polus/schedulers.py:5-23 = HF `WarmUp` over Keras `PolynomialDecay(power=1, end_learning_rate=1e-7)`.  TensorFlow is
    not installable here, but transformers ships the torch twin of the same schedule
    (`get_polynomial_decay_schedule_with_warmup(lr_end=1e-7, power=1.0)`): an implementation that is neither the oracle's
    nor the product's.  Both must follow it step by step (the device evaluates the same closed form inside polus_adam).
    Its learning rates are stored in tests/golden/hf_polynomial_warmup.npz (generator: tests/golden/make_schedule_golden.py)."""
    from oracle import numpy_ref as R
    from polus_b200.schedulers import warmup_scheduler
    with np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "hf_polynomial_warmup.npz")) as z:
        cases = [(int(n), float(lr), z[f"lrs_{i}"]) for i, (n, lr) in enumerate(zip(z["n_steps"], z["lr"]))]
    assert [(n, lr) for n, lr, _ in cases] == [(200, 3e-4), (1000, 5e-5), (37, 1e-3)]
    for n_steps, lr, hf_lrs in cases:
        sched = warmup_scheduler(n_steps, lr)
        assert hf_lrs.shape == (n_steps + 1,)
        for step in range(n_steps + 1):
            want = float(hf_lrs[step])
            assert abs(sched(step) - want) <= 1e-12 * max(1.0, want / 1e-7), (n_steps, step, sched(step), want)
            assert abs(R.warmup_schedule_lr(step, n_steps, lr) - want) <= 1e-12 * max(1.0, want / 1e-7)


def test_warmup_scheduler_matches_oracle():
    from oracle import numpy_ref as R
    from polus_b200.schedulers import warmup_scheduler
    s = warmup_scheduler(200, 3e-4, warmup_percentage=0.1, end_lr=123.0)  # end_lr ignored, like the reference
    assert s.warmup_steps == 20 and s.decay_steps == 180 and s.end_learning_rate == 1e-7
    for step in (0, 1, 19, 20, 21, 100, 199, 200, 5000):
        assert abs(s(step) - R.warmup_schedule_lr(step, 200, 3e-4)) < 1e-15


def _ref_get_bio(spans, entities):
    """Loop-for-loop restatement of polus/ner/bio.py:13-114 (entity_fits_spans / update_tags / get_bio)."""
    tags = ["O"] * len(spans)
    for (es, ee, typ) in sorted(entities, key=lambda e: e[1] - e[0], reverse=True):
        start_found = end_found = False
        idx = []
        for i, sp in enumerate(spans):
            if not start_found:
                if es == sp[0]:
                    start_found = True
                elif es < sp[0]:
                    break
            if start_found and not end_found:
                idx.append(i)
                if ee == sp[1]:
                    end_found = True
                    break
                elif ee < sp[1]:
                    break
        if start_found and end_found and all(tags[i] == "O" for i in idx):
            tags[idx[0]] = f"B-{typ}"
            for i in idx[1:]:
                tags[i] = f"I-{typ}"
    return tags


def test_bio_labels_bit_exact_vs_reference_algorithm():
    from polus_b200.ner.bio import get_bio
    from polus_b200.ner.utils import TAG2INT
    assert TAG2INT == {"PAD": 0, "O": 1, "B-Chemical": 2, "I-Chemical": 3}
    rng = np.random.default_rng(0)
    for _ in range(200):
        n = int(rng.integers(1, 15))
        cuts = np.sort(rng.choice(np.arange(1, 80), size=2 * n, replace=False))
        spans = [(int(cuts[2 * i]), int(cuts[2 * i + 1])) for i in range(n)]
        ents = []
        for _ in range(int(rng.integers(0, 6))):
            a, b = sorted(rng.integers(0, n, 2))
            s, e = spans[a][0], spans[b][1]
            if rng.uniform() < 0.3:
                s += 1  # misaligned: must be discarded
            ents.append((int(s), int(e), "Chemical"))
        assert get_bio(spans, ents) == _ref_get_bio(spans, ents)
    assert get_bio([(0, 3), (4, 9), (10, 12)], [(4, 12, "Chemical"), (4, 9, "Chemical")]) == ["O", "B-Chemical", "I-Chemical"]


def test_bio_labels_bit_exact_vs_reference_fixture():
    """get_bio and TAG2INT against tests/golden/bio_ref.json, which tests/golden/make_bio_golden.py produced by running
    the reference's OWN polus/ner/bio.py + elements.py (TF-free, loaded with stubbed packages): label indices bit-exact
    with the reference itself, not with a restatement."""
    import json
    from polus_b200.ner.bio import get_bio
    from polus_b200.ner.utils import TAG2INT
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "bio_ref.json")) as f:
        doc = json.load(f)
    assert TAG2INT == doc["tag2int"]
    assert len(doc["cases"]) >= 400
    for case in doc["cases"]:
        spans = [tuple(sp) for sp in case["spans"]]
        ents = [tuple(e) for e in case["entities"]]
        assert get_bio(spans, ents) == case["tags"], case
        # and as label indices, for the Chemical-only cases the reference's TAG2INT covers
        if all(t in TAG2INT for t in case["tags"]):
            assert [TAG2INT[t] for t in get_bio(spans, ents)] == [doc["tag2int"][t] for t in case["tags"]]


# ------------------------------------------------------------------ callbacks + trainer loop (fake step, no device)
def test_training_loop_order_and_callbacks(monkeypatch):
    from polus_b200.callbacks import Callback, ConsoleLogCallback, EarlyStop, LossSmoothCallback, TimerCallback
    from polus_b200.training import BaseTrainer, ClassifierTrainer

    with pytest.raises(Exception):
        BaseTrainer(None, None, None)

    class M:
        name = "fake"
        trainable_weights = []

    events = []

    class Spy(Callback):
        def on_train_begin(self): events.append("tb")
        def on_epoch_begin(self, e): events.append(f"eb{e}")
        def on_train_batch_begin(self, e, s): events.append(f"bb{e}.{s}")
        def on_train_batch_end(self, e, s, l): events.append(f"be{e}.{s}")
        def on_epoch_end(self, e): events.append(f"ee{e}")
        def on_train_end(self): events.append("te")

    tr = ClassifierTrainer(M(), optimizer=object(), loss=None)
    losses = iter([4.0, 3.0, 2.0, 1.0, 0.5, 0.25])
    monkeypatch.setattr(tr, "train_step", lambda *d: next(losses))
    smooth = LossSmoothCallback(output=True)
    with pytest.raises(ValueError):
        tr.train(epochs=1)
    tr.train([(1, 2), (3, 4), (5, 6)], epochs=2, callbacks=[smooth, TimerCallback(), Spy(), ConsoleLogCallback(), EarlyStop()])
    assert events == ["tb", "eb0", "bb0.0", "be0.0", "bb0.1", "be0.1", "bb0.2", "be0.2", "bb0.3", "ee0",
                      "eb1", "bb1.0", "be1.0", "bb1.1", "be1.1", "bb1.2", "be1.2", "bb1.3", "ee1", "te"]
    assert tr.step_counter == 6
    # bias-corrected EMA, beta 0.97 (callbacks.py:176-182)
    mov, n = 0.0, 0
    for l in [4.0, 3.0, 2.0, 1.0, 0.5, 0.25]:
        n += 1
        mov = 0.97 * mov + 0.03 * l
    assert abs(smooth.smooth_loss - mov / (1 - 0.97 ** n)) < 1e-12


def test_profiler_env_appends_callback_and_stops(monkeypatch, tmp_path):
    from polus_b200 import callbacks
    from polus_b200.training import ClassifierTrainer

    class M:
        name = "fake"
        trainable_weights = []
    calls = []
    from polus_b200 import device
    monkeypatch.setattr(callbacks._lib, "call", lambda name, *a: calls.append((name, a)) or 0)
    monkeypatch.setattr(device, "stream", lambda: 0)
    monkeypatch.setenv("POLUS_PROFILER", "true")
    monkeypatch.setenv("POLUS_PROFILER_RANGE", "2:4")
    monkeypatch.chdir(tmp_path)
    tr = ClassifierTrainer(M(), optimizer=object(), loss=None)
    monkeypatch.setattr(tr, "train_step", lambda *d: 1.0)
    tr.train([(0, 0)] * 10, epochs=1, callbacks=[])
    assert tr.step_counter == 4 and tr.early_stop  # window [2,4) then stop, like the reference
    names = [n for n, _ in calls]
    assert names.count("polus_profiler_start") == 1 and names.count("polus_profiler_stop") == 1
    # one named range per step of the window (reference: tf.profiler.experimental.Trace('step', step_num=...), callbacks.py:452-461)
    pushes = [a[0] for n, a in calls if n == "polus_profiler_range_push"]
    assert pushes == [b"step 2", b"step 3"] and names.count("polus_profiler_range_pop") == 2
    assert names.index("polus_profiler_start") < names.index("polus_profiler_range_push")
    assert (tmp_path / "logs" / "tensorboard_logs" / "step_times.json").exists()


def test_gradient_bucket_plan():
    """Buckets are contiguous arena spans, ordered from the end of the arena (backward order)."""
    from polus_b200 import comm
    from polus_b200.tensor import Param

    class Chunk:
        index = 1   # creation order: plan_buckets' rank-invariant sort key
    ch = Chunk()
    ps, off = [], 0
    for n in [1000, 64, 5000, 64, 300000, 64, 128]:
        p = Param.__new__(Param)
        p.shape, p.chunk, p.offset = (n,), ch, off
        off += (n + 63) & ~63
        ps.append(p)
    buckets = comm.plan_buckets(ps, bucket_bytes=100000)
    spans = [(b[1], b[2]) for b in buckets]
    assert sum(n for _, n in spans) == off
    assert spans[0][0] + spans[0][1] == off                       # first bucket ends the arena
    for (o1, n1), (o2, n2) in zip(spans, spans[1:]):
        assert o2 + n2 == o1                                       # contiguous, descending
    # the 300000-element variable (>= bucket_bytes / 2) stands alone, cut into ~bucket_bytes / 2 pieces; nothing is merged
    # with it, so its neighbours are exchanged as soon as they are ready
    big = [b for b in buckets if b[3] == [ps[4]]]
    assert len(big) >= 2 and sum(b[2] for b in big) == 300032 and all(b[2] * 4 <= 100000 for b in big)
    assert all(n * 4 <= 100000 + 4 * 5056 for _, n in spans)
    order = []
    for b in buckets:
        for p in b[3]:
            if not order or order[-1] != id(p):
                order.append(id(p))
    assert order == [id(p) for p in reversed(ps)]


def test_mock_horovod_surface():
    from polus_b200.mock import horovod as hvd
    assert hvd.init() == "mock" and hvd.size() == 1 and hvd.local_rank() == 0
    t = object()
    assert hvd.DistributedGradientTape(t) is t
    assert hvd.broadcast_variables([1, 2], root_rank=0) is None
    assert hvd.allgather_object({"a": 1}) == [{"a": 1}]


def test_decode_bio_round_trip_and_error_counts():
    """§8f rank 1: BIO decoding (reference polus/ner/bio.py:115-188, with its loop-state bug fixed) inverts get_bio and
    counts the two error classes the reference logs."""
    from polus_b200.ner.bio import decode_bio, get_bio
    spans = [(0, 3), (4, 9), (10, 12), (13, 20), (21, 25), (26, 30)]
    ents = [(4, 12, "Chemical"), (21, 25, "Chemical")]
    tags = get_bio(spans, ents)
    assert tags == ["O", "B-Chemical", "I-Chemical", "O", "B-Chemical", "O"]
    es, counts = decode_bio(tags, spans)
    assert es == set(ents) and counts == {"tags": 6, "inside_tag_after_other_tag": 0, "inside_tag_with_different_entity_type": 0}
    # I after O opens an entity; I of another type closes + reopens; the trailing entity is flushed
    es, counts = decode_bio(["I-Chemical", "I-Gene", "O", "B-Chemical", "B-Chemical", "I-Chemical"], spans, allow_errors=True)
    assert es == {(0, 3, "Chemical"), (4, 9, "Gene"), (13, 20, "Chemical"), (21, 30, "Chemical")}
    assert counts["inside_tag_after_other_tag"] == 1 and counts["inside_tag_with_different_entity_type"] == 1
    with pytest.raises(AssertionError):
        decode_bio(["O", "I-Chemical"], spans[:2])


def test_entity_f1_strict_matching_and_window_filter():
    """Entity-level F1 (reference polus/ner/metrics.py:8-21 + ner/utils.py:231-308): strict span+type match, documents
    assembled from windows in arrival order, positions with is_prediction == 0 ignored."""
    from polus_b200.ner.metrics import EntityF1, eval_list_of_entity_sets, precision_recall_f1
    from polus_b200.ner.utils import TAG2INT as T
    O, B, I, P = T["O"], T["B-Chemical"], T["I-Chemical"], T["PAD"]
    spans = np.array([[[0, 2], [3, 5], [6, 8], [9, 11]], [[6, 8], [9, 11], [12, 14], [0, 0]]])
    batch = {"identifier": np.array(["doc1", "doc1"]), "spans": spans,
             "tags_int": np.array([[B, I, O, B], [O, B, I, P]]),
             "tags_int_pred": np.array([[B, I, O, B], [B, B, O, P]]),
             "is_prediction": np.array([[1, 1, 1, 1], [0, 0, 1, 0]])}  # second window: only its third token is new
    m = EntityF1()
    m.samples_from_batch(batch)
    r = m.evaluate_ner()
    # gold: (0,5), (9,14)   pred: (0,5), (9,11)   -> tp 1, fp 1, fn 1
    assert (r["tp"], r["fp"], r["fn"]) == (1, 1, 1) and r["f1"] == 0.5
    assert precision_recall_f1(0, 0, 0)[2] != precision_recall_f1(0, 0, 0)[2]  # nan
    assert precision_recall_f1(0, 0, 0, return_nan=False) == (0.0, 0.0, 0.0)
    assert eval_list_of_entity_sets([{(0, 1, "A")}], [{(0, 1, "A"), (2, 3, "A")}])["precision"] == 0.5
    # gold supplied as entity lists instead of gold tags
    m2 = EntityF1(gold={"doc1": [(0, 5, "Chemical"), (9, 14, "Chemical")]})
    del batch["tags_int"]
    m2.samples_from_batch([batch])
    assert m2.evaluate() == 0.5


# ------------------------------------------------------------------ cached loaders (reference tests/test_data.py:68-345)
def _count_gen(n, text="dummy"):
    def source_gen():
        for i in range(n):
            yield {"id": i, "text": text}
    return source_gen


def _walk(dl):
    ordered, n, sample = True, 0, None
    for sample in dl:
        ordered = ordered and sample["id"] == n
        n += 1
    return ordered, n, sample


def test_cached_dataloader_chunk_format_and_order(tmp_path):
    """Chunk files `<base>_NNNN.part` = pickled lists of <= chunk samples; `.index` = JSON with files / cache_chunk_size /
    n_samples (reference data.py:266-320): a reader that knows only that format recovers the samples."""
    import pickle
    from polus_b200.data import CachedDataLoader
    dl = CachedDataLoader(_count_gen(1000), cache_chunk_size=256, cache_folder=str(tmp_path))
    ordered, n, last = _walk(dl)
    assert ordered and n == 1000 and dl.get_n_samples() == 1000 and last == {"id": 999, "text": "dummy"}
    assert dl.cache_base_name == "_chunk256_source_gen"
    files = sorted(os.listdir(tmp_path))
    assert files == ["_chunk256_source_gen.index"] + [f"_chunk256_source_gen_{k:04}.part" for k in range(4)]
    with open(dl.cache_index_path) as f:
        index = json.load(f)
    assert set(index) == {"files", "cache_chunk_size", "n_samples"} and index["n_samples"] == 1000 and index["cache_chunk_size"] == 256
    sizes = []
    for path in index["files"]:
        with open(path, "rb") as f:
            sizes.append(len(pickle.load(f)))
    assert sizes == [256, 256, 256, 232]
    # a second loader over the same generator name finds the cache and never calls the generator
    def source_gen():
        raise AssertionError("the cache should have been used")
        yield
    again = CachedDataLoader(source_gen, cache_chunk_size=256, cache_folder=str(tmp_path))
    assert _walk(again)[:2] == (True, 1000)
    # through the dataset verbs the trainer consumes
    ids = [int(s["id"]) for s in dl.to_tfDataset()]
    assert ids == list(range(1000))
    dl.clean()
    assert os.listdir(tmp_path) == []


def test_cached_dataloader_reads_a_cache_written_in_the_reference_layout(tmp_path):
    """Files laid out by hand exactly as the reference writes them are opened with from_cached_index."""
    import pickle
    from polus_b200.data import CachedDataLoader
    files = []
    for k in range(3):
        path = str(tmp_path / f"x__chunk4_g_{k:04}.part")
        with open(path, "wb") as f:
            pickle.dump([{"id": 4 * k + i} for i in range(4 if k < 2 else 1)], f)
        files.append(path)
    index_path = str(tmp_path / "x__chunk4_g.index")
    with open(index_path, "w") as f:
        json.dump({"files": files, "cache_chunk_size": 4, "n_samples": 9}, f)
    dl = CachedDataLoader.from_cached_index(index_path)
    assert _walk(dl)[:2] == (True, 9) and dl.cache_chunk_size == 4 and dl.cache_index_path == index_path


def test_cached_dataloader_with_lookup_and_conversion(tmp_path):
    from polus_b200.data import CachedDataLoader, CachedDataLoaderwLookup
    data = {"a": 1, "b": 2, "c": 3}
    dl = CachedDataLoaderwLookup(_count_gen(1000), lookup_data=data, cache_chunk_size=256, cache_folder=str(tmp_path / "a"))
    assert _walk(dl)[:2] == (True, 1000) and dl.get_lookup_data()["c"] == 3
    files = os.listdir(tmp_path / "a")
    assert f"{dl.cache_base_name}.index" in files and f"{dl.cache_base_name}.lookup" in files
    assert all(os.path.basename(p) in files for p in dl.cache_index["files"])
    with pytest.raises(ValueError):
        CachedDataLoaderwLookup(_count_gen(3), cache_folder=str(tmp_path / "a"))
    # CachedDataLoader -> add_lookup_data -> CachedDataLoaderwLookup over the same chunks
    plain = CachedDataLoader(_count_gen(1000), cache_chunk_size=256, cache_folder=str(tmp_path / "b"))
    conv = plain.add_lookup_data(data)
    assert isinstance(conv, CachedDataLoaderwLookup) and _walk(conv)[:2] == (True, 1000) and conv.get_lookup_data() == data
    base = os.path.splitext(os.path.basename(conv.cache_index_path))[0]
    assert {f"{base}.index", f"{base}.lookup"} <= set(os.listdir(tmp_path / "b"))
    conv.clean()
    assert os.listdir(tmp_path / "b") == []


def test_cached_dataloader_pre_shuffle_merge_and_reopen(tmp_path):
    from polus_b200.data import CachedDataLoader, CachedDataLoaderwLookup
    import random
    random.seed(0)
    def new_gen():
        for s in _count_gen(1000)():
            s["new_entry"] = s["id"] * 2
            yield s
    dl = CachedDataLoader(new_gen, cache_chunk_size=16, cache_folder=str(tmp_path))
    assert _walk(dl)[:2] == (True, 1000)
    dl.pre_shuffle()
    ordered, n, _ = _walk(dl)
    assert not ordered and n == 1000
    seen = [s["id"] for s in dl]
    assert sorted(seen) == list(range(1000))
    # chunk-level shuffle: inside every chunk of 16 the samples stay consecutive
    assert all(seen[k - 1] == v - 1 for k, v in enumerate(seen) if v % 16 != 0)
    # merge of three caches with different lengths
    def named(n, text, name):
        g = _count_gen(n, text)
        g.__name__ = name
        return g
    parts = [CachedDataLoader(named(n, t, f"gen_{t}"), cache_chunk_size=64, cache_folder=str(tmp_path))
             for n, t in ((1000, "dummy"), (500, "dummy2"), (721, "dummy3"))]
    merged = CachedDataLoader.merge(*parts).pre_shuffle()
    ordered, n, _ = _walk(merged)
    assert not ordered and n == 2221 and merged.get_n_samples() == 2221 and merged.cache_chunk_size == 64
    assert {s["text"] for s in merged} == {"dummy", "dummy2", "dummy3"}
    # reopen from the index path alone
    again = CachedDataLoader.from_cached_index(parts[0].cache_index_path).pre_shuffle()
    ordered, n, last = _walk(again)
    assert not ordered and n == 1000 and last["text"] == "dummy"
    # merged lookups concatenate
    la = parts[1].add_lookup_data(["x", "y"])
    lb = parts[2].add_lookup_data(["z"])
    both = CachedDataLoaderwLookup.merge(la, lb)
    assert both.get_lookup_data() == ["x", "y", "z"] and both.get_n_samples() == 1221 and _walk(both)[1] == 1221
    # deep_copy: a second index over the same chunks
    parts[0].deep_copy(suffix="v2")
    assert parts[0].cache_index_path.endswith("_chunk64_gen_dummy_v2.index") and os.path.exists(parts[0].cache_index_path)


def test_cached_dataloader_cleans_up_when_the_generator_fails(tmp_path):
    from polus_b200.data import CachedDataLoader
    def bad_gen():
        for i in range(40):
            yield {"id": i}
        raise RuntimeError("source failed")
    with pytest.raises(RuntimeError):
        CachedDataLoader(bad_gen, cache_chunk_size=16, cache_folder=str(tmp_path))
    assert os.listdir(tmp_path) == []


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU port of the reference step, timed on host cores) prints ONE JSON line with the
    keys the driver reads; non-zero ranks of a torchrun launch exit 0 silently."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--ref-batch", "1"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "train_sequences_per_second" and d["unit"] == "sequences/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["n_gpus"] == 1 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "sequences/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    silent = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root, env=dict(os.environ, RANK="1", WORLD_SIZE="2"))
    assert silent.returncode == 0 and silent.stdout.strip() == ""


def test_bench_dump_outputs_writes_the_last_losses_as_float32(tmp_path):
    """`bench.py --dump-outputs DIR`: one float32 .npy of shape (1,) per timed region, named after the region."""
    import bench
    bench.dump_outputs(str(tmp_path / "out"), {"resident": 1.5, "e2e": 2.25})
    assert sorted(os.listdir(tmp_path / "out")) == ["loss_e2e.npy", "loss_resident.npy"]
    for name, value in (("loss_resident.npy", 1.5), ("loss_e2e.npy", 2.25)):
        a = np.load(tmp_path / "out" / name)
        assert a.dtype == np.float32 and a.tolist() == [value]


def test_bioc_sequence_decoder_flow_and_strict_evaluation():
    """polus/ner/utils.py: samples_from_batch (is_prediction filtering, windows of one document concatenated) -> decode
    (BIO error counters) -> strict entity-level evaluation; precision_recall_f1 / empty_results conventions."""
    import math
    from polus_b200.ner.utils import BioCSequenceDecoder, TAG2INT, empty_results, eval_list_of_entity_sets, precision_recall_f1
    assert precision_recall_f1(3, 1, 2) == (0.75, 0.6, 3 / 4.5)
    assert all(math.isnan(v) for v in precision_recall_f1(0, 0, 0)) and precision_recall_f1(0, 0, 0, return_nan=False) == (0.0, 0.0, 0.0)
    assert empty_results() == {"tp": 0, "fp": 0, "fn": 0, "precision": 0.0, "recall": 0.0, "f1": 0.0}
    assert empty_results(counts=False) == {"precision": 0.0, "recall": 0.0, "f1": 0.0}
    r = eval_list_of_entity_sets([{(0, 4, "Chemical"), (10, 15, "Chemical")}, set()], [{(0, 4, "Chemical"), (11, 15, "Chemical")}, {(1, 2, "Chemical")}])
    assert (r["tp"], r["fp"], r["fn"]) == (1, 2, 1) and r["f1"] == 1 / 2.5

    text = "aspirin and sodium chloride here"
    spans = [(0, 7), (8, 11), (12, 18), (19, 27), (28, 32)]
    gold = {"corpusA": {"train": {"doc1": {"text": text, "es": [(0, 7, "Chemical"), (12, 27, "Chemical")]},
                                  "doc2": {"text": "water", "es": [(0, 5, "Chemical")]}}}}
    dec = BioCSequenceDecoder(gold)
    O, B, I, PAD = TAG2INT["O"], TAG2INT["B-Chemical"], TAG2INT["I-Chemical"], TAG2INT["PAD"]
    pad = (0, 0)
    # doc1 arrives as two overlapping windows of 4 tokens: the overlap token is predicted by the first window only
    batch1 = {"corpus": np.array([b"corpusA", b"corpusA"]), "group": np.array([b"train", b"train"]),
              "identifier": np.array([b"doc1", b"doc1"]),
              "spans": np.array([[spans[0], spans[1], spans[2], pad], [spans[2], spans[3], spans[4], pad]]),
              "tags_int_pred": np.array([[B, O, B, PAD], [O, I, O, PAD]], np.int32),
              "is_prediction": np.array([[1, 1, 1, 0], [0, 1, 1, 0]], np.int32)}
    batch2 = {"corpus": np.array([b"corpusA"]), "group": np.array([b"train"]), "identifier": np.array([b"doc2"]),
              "spans": np.array([[(0, 5), pad, pad, pad]]), "tags_int_pred": np.array([[I, PAD, PAD, PAD]], np.int32),
              "is_prediction": np.array([[1, 0, 0, 0]], np.int32)}
    dec.samples_from_batch(batch1)
    dec.samples_from_batch([batch2])
    assert dec.documents_dict["corpusA"]["train"]["doc1"]["tags"] == ["B-Chemical", "O", "B-Chemical", "I-Chemical", "O"]
    counts = dec.decode()
    assert counts == {"tags": 6, "inside_tag_after_other_tag": 1, "inside_tag_with_different_entity_type": 0}
    assert dec.documents_dict["corpusA"]["train"]["doc1"]["es"] == {(0, 7, "Chemical"), (12, 27, "Chemical")}
    res = dec._evaluate_ner()
    assert (res["tp"], res["fp"], res["fn"]) == (3, 0, 0) and res["f1"] == 1.0 and dec.documents_dict == {}
    # one call from a giant batch, with a miss
    batch1["tags_int_pred"] = np.array([[B, O, O, PAD], [O, O, O, PAD]], np.int32)
    res = dec.evaluate_ner_from_sample([batch1, batch2])
    assert (res["tp"], res["fp"], res["fn"]) == (2, 0, 1)
    with pytest.raises(NotImplementedError):
        dec.get_collections()

    # corpus objects that iterate like the reference's Corpus / Collection / Document
    class Doc:
        def __init__(self, text, es):
            self._t, self._es = text, es
        def text(self):
            return self._t
        def get_entity_set(self):
            return self._es
    class Corpus:
        def __str__(self):
            return "corpusB"
        def __iter__(self):
            return iter([("test", [("d", Doc("water", {(0, 5, "Chemical")}))])])
    dec2 = BioCSequenceDecoder([Corpus()])
    assert dec2.documents == {"corpusB": {"test": {"d": {"text": "water", "es": {(0, 5, "Chemical")}}}}}


def test_bio_helpers_match_reference_semantics():
    """polus/ner/bio.py:5-114: longest entity first, exact fit over consecutive token spans, no overwriting."""
    from polus_b200.ner.bio import entity_fits_spans, get_bio, longer_entities_first, update_tags
    spans = [(0, 7), (8, 11), (12, 18), (19, 27), (28, 32)]
    assert entity_fits_spans((12, 27, "Chemical"), spans) == [2, 3]
    assert entity_fits_spans((0, 7, "Chemical"), spans) == [0]
    assert entity_fits_spans((12, 20, "Chemical"), spans) is False      # ends inside a token
    assert entity_fits_spans((13, 27, "Chemical"), spans) is False      # starts inside a token
    assert entity_fits_spans((40, 45, "Chemical"), spans) is False
    ents = [(12, 18, "Chemical"), (12, 27, "Chemical"), (0, 7, "Chemical")]
    assert longer_entities_first(ents)[0] == (12, 27, "Chemical")
    tags = ["O"] * 5
    update_tags(tags, spans, (12, 27, "Chemical"))
    update_tags(tags, spans, (12, 18, "Chemical"))                       # overlaps an annotated entity: discarded
    assert tags == ["O", "O", "B-Chemical", "I-Chemical", "O"]
    assert get_bio(spans, ents) == ["B-Chemical", "O", "B-Chemical", "I-Chemical", "O"]

    class E:  # reference-style entity objects
        def __init__(self, s, e, t):
            self.start, self.end, self.typ = s, e, t
    assert get_bio(spans, [E(19, 32, "Chemical")]) == ["O", "O", "O", "B-Chemical", "I-Chemical"]
    # randomised: same result as a direct statement of the rule
    rng = np.random.default_rng(0)
    for _ in range(200):
        cuts = np.sort(rng.choice(np.arange(1, 60), size=rng.integers(2, 12), replace=False))
        toks = [(int(a), int(b) - int(rng.integers(0, 2))) for a, b in zip(cuts[:-1], cuts[1:])]
        toks = [(a, max(b, a + 1)) for a, b in toks]
        ents = []
        for _ in range(rng.integers(0, 5)):
            i = int(rng.integers(0, len(toks)))
            j = int(rng.integers(i, len(toks)))
            s0, e0 = toks[i][0] + int(rng.integers(0, 2)) * int(rng.integers(0, 2)), toks[j][1]
            ents.append((s0, e0, "Chemical"))
        want = ["O"] * len(toks)
        for s0, e0, ty in sorted(ents, key=lambda e: e[1] - e[0], reverse=True):
            idx = [k for k, (a, b) in enumerate(toks) if a >= s0 and b <= e0]
            if idx and toks[idx[0]][0] == s0 and toks[idx[-1]][1] == e0 and all(want[k] == "O" for k in idx):
                want[idx[0]] = f"B-{ty}"
                for k in idx[1:]:
                    want[k] = f"I-{ty}"
        assert get_bio(toks, ents) == want


def test_hpo_prune_callback_without_and_with_backend():
    """polus/callbacks.py:366-405: a no-op (with a warning) when there is no HPO context; with a backend it reports the
    last validation score of the epoch and stops a pruned trial."""
    from types import SimpleNamespace
    from polus_b200.callbacks import HPOPruneCallback
    cb = HPOPruneCallback("val", "f1")
    cb.coordinator = SimpleNamespace(shared_dict={"validation": {"val": {"f1": [0.1, 0.2]}}}, trainer=SimpleNamespace(early_stop=False))
    cb.on_epoch_end(0)  # nothing happens
    seen = []
    backend = SimpleNamespace(report=lambda score, step: seen.append((score, step)), should_prune=lambda: len(seen) >= 2)
    cb = HPOPruneCallback("val", "f1", hpo_backend=backend)
    cb.coordinator = SimpleNamespace(shared_dict={"validation": {"val": {"f1": [0.1, 0.2]}}}, trainer=SimpleNamespace(early_stop=False))
    cb.on_epoch_end(0)
    assert seen == [(0.2, 0)] and cb.coordinator.trainer.early_stop is False
    try:
        cb.on_epoch_end(1)
        pruned = cb.coordinator.trainer.early_stop  # optuna absent: the trainer is told to stop
    except Exception as e:  # optuna present: TrialPruned
        pruned = type(e).__name__ == "TrialPruned"
    assert pruned and seen[-1] == (0.2, 1)


def test_polus_alias_package_resolves_to_the_same_modules():
    """`from polus.training import ClassifierTrainer` (a script written against the reference) gets polus_b200's class, and
    the module objects are shared (one parameter arena, one PolusContext), not re-imported copies."""
    import sys
    import polus
    import polus.callbacks
    from polus.ir.training import EfficientDenseRetrievalTrainer
    from polus.mock import horovod
    from polus.ner.models import baselineNER_MLP_Dropout_CRF
    from polus.training import BaseTrainer, ClassifierTrainer
    import polus_b200
    import polus_b200.training
    assert ClassifierTrainer is polus_b200.training.ClassifierTrainer and issubclass(ClassifierTrainer, BaseTrainer)
    assert sys.modules["polus.training"] is sys.modules["polus_b200.training"]
    assert sys.modules["polus.callbacks"] is sys.modules["polus_b200.callbacks"]
    assert polus.PolusContext is polus_b200.PolusContext and polus.__version__ == polus_b200.__version__
    assert horovod.size() == 1 and callable(baselineNER_MLP_Dropout_CRF) and EfficientDenseRetrievalTrainer.__name__ == "EfficientDenseRetrievalTrainer"
    import pytest
    with pytest.raises(ImportError):
        import polus.hpo  # noqa: F401  (out of scope: not provided, and the alias must not invent it)
