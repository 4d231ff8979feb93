"""Dataset-stack properties (same catalogue the reference pins, SURVEY.md §4.1; assertions re-written).
"Multi-node" is simulated in one process: N dataset objects with different (rank, worldsize)."""
import copy
import hashlib
import json
import os
import tarfile
import tempfile

import pyarrow as pa
import pytest
import torch

from fms_fsdp_b200.utils.dataset_utils import (ArrowHandler, BufferDataset, CheckpointDataset, PreloadBufferDataset,
                                               PreprocessDataset, SamplingDataset, ScalableShardDataset,
                                               StreamingDocDataset, _shard_inclusive, _shard_partition,
                                               _StatefulDataset, _WrapperDataset)

SCHEMA = pa.schema([pa.field("tokens", pa.uint32())])


def _write(path, docs):
    os.makedirs(os.path.dirname(path), exist_ok=True)
    with pa.ipc.new_file(path, SCHEMA) as w:
        for d in docs:
            w.write(pa.record_batch([d], schema=SCHEMA))


def make_corpus():
    """dataset_1: 100 docs x 100 tokens (doc i = range(100i, 100i+100)); dataset_2: 2 files x 50 docs x 50 tokens
    (one in a sub-folder); meta/combined_counts.csv.  Token values identify (doc, position)."""
    tmp = tempfile.mkdtemp()
    _write(f"{tmp}/dataset_1/fullshard.arrow", [list(range(i * 100, i * 100 + 100)) for i in range(100)])
    _write(f"{tmp}/dataset_2/quartershard_1.arrow", [list(range(i * 50, i * 50 + 50)) for i in range(50)])
    _write(f"{tmp}/dataset_2/subfolder/quartershard_2.arrow", [list(range(2500 + i * 50, 2500 + i * 50 + 50)) for i in range(50)])
    os.makedirs(f"{tmp}/meta")
    with open(f"{tmp}/meta/combined_counts.csv", "w") as f:
        f.write("dataset/filename,documents,tokens\n/dataset_1/fullshard.arrow,100,10000\n"
                "/dataset_2/quartershard_1.arrow,50,2500\n/dataset_2/subfolder/quartershard_2.arrow,50,2500\n")
    return tmp


@pytest.fixture(scope="module")
def corpus():
    return make_corpus()


def doc_reader(corpus, rank=0, world=1, ds="dataset_1", chunk=1000, **kw):
    return StreamingDocDataset(os.path.join(corpus, ds), rank, world, ArrowHandler(), -1, max_chunksize=chunk, **kw)


def scalable(corpus, rank=0, world=1, ds="dataset_1", chunk=1000, n=12, **kw):
    return ScalableShardDataset(doc_reader(corpus, rank, world, ds, chunk, **kw), -1, n_logical_shards=n)


def sampler(corpus, rank=0, world=1, chunk=1000, datasets=("dataset_1",), weights=None, scal=False, n=12):
    base = scalable(corpus, rank, world, "dataset_1", chunk, n) if scal else doc_reader(corpus, rank, world, "dataset_1", chunk)
    return SamplingDataset(corpus, base, -1, datasets=list(datasets), weights=weights)


BUILDERS = {
    "doc": lambda c, r=0, w=1, **k: doc_reader(c, r, w, **k),
    "scalable": lambda c, r=0, w=1, **k: scalable(c, r, w, **k),
    "sampler": lambda c, r=0, w=1, **k: sampler(c, r, w, **{x: y for x, y in k.items() if x == "chunk"}),
    "sampler_scalable": lambda c, r=0, w=1, **k: sampler(c, r, w, scal=True, **{x: y for x, y in k.items() if x == "chunk"}),
}


def take(it, n):
    return [next(it) for _ in range(n)]


def test_partition_helpers():
    items = list(range(10))
    assert [_shard_partition(items, r, 3) for r in range(3)] == [[0, 1, 2], [3, 4, 5], [6, 7, 8, 9]]
    assert _shard_inclusive(items, 1, 4) == [2, 3, 4] and _shard_inclusive(items, 0, 3) == [0, 1, 2, 3]
    assert issubclass(_WrapperDataset, _StatefulDataset)


@pytest.mark.parametrize("kind", list(BUILDERS))
def test_single_and_two_epochs(corpus, kind):
    d = BUILDERS[kind](corpus)
    it = iter(d)
    first = sorted(x[0] // 100 for x in take(it, 100))
    assert first == list(range(100))  # every doc exactly once per epoch
    second = sorted(x[0] // 100 for x in take(it, 100))
    assert second == list(range(100))
    if kind == "doc":
        assert d.docs_seen == 200 and d.tokens_seen == 20000 and d.epochs_seen == 1


@pytest.mark.parametrize("kind", list(BUILDERS))
def test_chunking(corpus, kind):
    it = iter(BUILDERS[kind](corpus, chunk=50))
    chunks = take(it, 300)  # 100-token doc + delimiter = 101 -> chunks of 50, 50, 1(delimiter only)
    lens = sorted(len(c) for c in chunks)
    assert lens == [1] * 100 + [50] * 200
    starts = sorted(c[0] for c in chunks if len(c) == 50)
    assert starts == list(range(0, 10000, 50))


def test_eos_bos_chunk_lengths(corpus):
    for chunk, expect in [(99, [99, 2]), (100, [100, 1]), (101, [101]), (102, [101])]:
        assert [len(c) for c in take(iter(doc_reader(corpus, chunk=chunk)), len(expect))] == expect
    for chunk, expect in [(100, [100, 2]), (101, [101, 1]), (102, [102]), (103, [102])]:
        out = take(iter(doc_reader(corpus, chunk=chunk, bos_token=-2)), len(expect))
        assert [len(c) for c in out] == expect and out[0][0] == -2 and out[-1][-1] == -1


@pytest.mark.parametrize("kind", list(BUILDERS))
def test_two_ranks_cover_disjointly(corpus, kind):
    its = [iter(BUILDERS[kind](corpus, r, 2)) for r in range(2)]
    seen = [sorted(x[0] // 100 for x in take(it, 50)) for it in its]
    assert not set(seen[0]) & set(seen[1]) and sorted(seen[0] + seen[1]) == list(range(100))


def test_multi_file_and_subfolder(corpus):
    it = iter(doc_reader(corpus, ds="dataset_2"))
    assert sorted(x[0] // 50 for x in take(it, 100)) == list(range(100))


@pytest.mark.parametrize("kind", list(BUILDERS))
def test_reload_mid_epoch_no_repeats(corpus, kind):
    ds = [BUILDERS[kind](corpus, r, 2, chunk=40) for r in range(2)]
    its = [iter(d) for d in ds]
    before = [take(it, 31) for it in its]
    states = [copy.deepcopy(d.state_dict()) for d in ds]
    fresh = [BUILDERS[kind](corpus, r, 2, chunk=40) for r in range(2)]
    for d in fresh:
        d.load_state_dict(copy.deepcopy(states))
    seen = {c[0] for b in before for c in b}
    n_rest = 3 * 100 - 62  # 3 chunks per doc (40, 40, 21)
    rest = [take(iter(d), n_rest // 2) for d in fresh]
    after = {c[0] for r in rest for c in r}
    assert not seen & after and len(seen | after) == 300
    cont = [take(it, 20) for it in its]           # the original keeps going: token-identical to the reload
    assert cont[0] == rest[0][:20] and cont[1] == rest[1][:20]


def test_sampler_rates(corpus):
    for weights, period in [([1, 1], [0, 1]), ([2, 1], None), ([2, 3], None)]:
        d = SamplingDataset(corpus, doc_reader(corpus), -1, datasets=["dataset_1", "dataset_2"], weights=weights)
        it = iter(d)
        toks = [0, 0]
        for _ in range(400):
            x = next(it)
            toks[0 if len(x) == 101 else 1] += len(x)
        share = toks[0] / sum(toks)
        assert abs(share - weights[0] / sum(weights)) < 0.02


def _pipelines(corpus):
    return {
        "doc": lambda r, w: doc_reader(corpus, r, w, chunk=17),
        "scalable": lambda r, w: scalable(corpus, r, w, chunk=17),
        "sampler": lambda r, w: SamplingDataset(corpus, scalable(corpus, r, w, chunk=17), -1, datasets=["dataset_1", "dataset_2"], weights=[3, 5]),
        "buffer": lambda r, w: BufferDataset(SamplingDataset(corpus, scalable(corpus, r, w, chunk=17), -1, datasets=["dataset_1", "dataset_2"], weights=[3, 5]), 73, True, bos_token=-5, eos_token=-6),
        "preload": lambda r, w: PreloadBufferDataset(BufferDataset(SamplingDataset(corpus, scalable(corpus, r, w, chunk=17), -1, datasets=["dataset_1", "dataset_2"], weights=[3, 5]), 73, True), 99),
    }


@pytest.mark.parametrize("name", ["doc", "scalable", "sampler", "buffer", "preload"])
@pytest.mark.parametrize("before,after", [(0, 50), (1, 100), (10, 150), (100, 200), (1000, 120)])
def test_reload_stress_token_identical(corpus, name, before, after):
    make = _pipelines(corpus)[name]
    ds = [make(r, 3) for r in range(3)]
    its = [iter(d) for d in ds]
    for it in its:
        take(it, before)
    states = [copy.deepcopy(d.state_dict()) for d in ds]
    expect = [take(it, after) for it in its]
    fresh = [make(r, 3) for r in range(3)]
    for d in fresh:
        d.load_state_dict(copy.deepcopy(states))
    got = [take(iter(d), after) for d in fresh]
    assert got == expect


@pytest.mark.parametrize("new_world", [1, 2, 3, 6, 12])
def test_scalable_rescale_partition(corpus, new_world):
    old = [scalable(corpus, r, 4) for r in range(4)]
    its = [iter(d) for d in old]
    seen = [x[0] // 100 for it in its for x in take(it, 9)]
    states = [copy.deepcopy(d.state_dict()) for d in old]
    new = [scalable(corpus, r, new_world) for r in range(new_world)]
    for d in new:
        d.load_state_dict(copy.deepcopy(states))
    per = [d.n_docs_remaining for d in new]
    assert sum(sum(p) for p in per) == 100 - len(seen)
    rest = []
    for d, p in zip(new, per):
        rest += [x[0] // 100 for x in take(iter(d), sum(p))]
    assert sorted(seen + rest) == list(range(100))  # disjoint and complete across the rescale


def test_scalable_sampler_rescale_completes_epoch(corpus):
    mk = lambda r, w: SamplingDataset(corpus, scalable(corpus, r, w), -1, datasets=["dataset_1"])  # noqa: E731
    old = [mk(r, 2) for r in range(2)]
    seen = [x[0] // 100 for d in old for x in take(iter(d), 20)]
    states = [copy.deepcopy(d.state_dict()) for d in old]
    new = [mk(r, 4) for r in range(4)]
    for d in new:
        d.load_state_dict(copy.deepcopy(states))
    rest = [x[0] // 100 for d in new for x in take(iter(d), sum(d.data[0].n_docs_remaining))]
    assert sorted(seen + rest) == list(range(100))


class _Counter(_StatefulDataset):
    def __init__(self, lens, rank=0, world=1):
        super().__init__(None, rank, world)
        self.lens, self.i, self.state_params = lens, 0, ["i"]

    def __iter__(self):
        while True:
            n = self.lens[self.i % len(self.lens)]
            yield list(range(self.i * 1000, self.i * 1000 + n))
            self.i += 1


def test_buffer_format_and_accounting():
    src = _Counter([5, 17, 3, 40, 8])
    lines = take(iter(BufferDataset(src, 16, True, bos_token=-1, eos_token=-2)), 50)
    assert all(len(l) == 16 and l[0] == -1 and l[-1] == -2 for l in lines)
    payload = [t for l in lines for t in l if t >= 0]
    expect = [t for i in range(len(payload)) for t in range(i * 1000, i * 1000 + [5, 17, 3, 40, 8][i % 5])][:len(payload)]
    assert payload == expect  # nothing lost, nothing duplicated, order preserved
    padded = take(iter(BufferDataset(_Counter([5, 6]), 16, False, pad_token=0, eos_token=-2)), 4)
    assert all(len(l) == 16 for l in padded) and padded[0][:5] == list(range(5))


def test_buffer_delimiter_overlap():
    class Src(_StatefulDataset):
        def __init__(self):
            super().__init__(None, 0, 1)

        def __iter__(self):
            while True:
                yield [-1, 7, 7, 7]
    lines = take(iter(BufferDataset(Src(), 8, True, bos_token=-1)), 3)
    assert lines[0] == [-1, 7, 7, 7, -1, 7, 7, 7]  # BOS not duplicated when already in slot 0


def test_preload_uniformity_and_no_loss():
    d = PreloadBufferDataset(_Counter([1]), 200)
    vals = [x[0] // 1000 for x in take(iter(d), 1000)]
    assert len(set(vals)) == 1000 and len({v for v in vals if v < 100}) >= 95


def test_checkpoint_dataset_autosave_and_resume(corpus):
    ck = tempfile.mkdtemp()
    def make():
        d = BufferDataset(scalable(corpus, 0, 1, chunk=17, n=3), 33, True)
        d = PreprocessDataset(d, torch.IntTensor)
        return CheckpointDataset(d, ck, 25, steps_per_batch=2, save_path=ck)
    a = iter(torch.utils.data.DataLoader(make(), num_workers=0, batch_size=2))
    first = [next(a) for _ in range(26)]  # the save fires when the worker resumes after the 25th batch
    assert os.listdir(os.path.join(ck, "checkpoints")) == ["step_25_ckp"]
    assert os.listdir(os.path.join(ck, "checkpoints", "step_25_ckp")) == ["loader_state_0.pth"]
    fresh = make()
    b = iter(torch.utils.data.DataLoader(fresh, num_workers=0, batch_size=2))
    got = [next(b)]                      # setup happens here: auto-loads step_25
    assert fresh.step == 25
    cont = [first[25]] + [next(a) for _ in range(20)]
    got += [next(b) for _ in range(20)]
    assert all(torch.equal(x, y) for x, y in zip(cont, got))


@pytest.mark.parametrize("world,workers", [(2, 0), (2, 2), (5, 2)])
def test_multiprocess_epoch(corpus, world, workers):
    n_logical = 20
    seen = []
    for r in range(world):
        d = PreprocessDataset(scalable(corpus, r, world, n=n_logical), lambda x: torch.tensor(x[0] // 100))
        dl = iter(torch.utils.data.DataLoader(d, num_workers=workers, batch_size=1))
        seen += [next(dl).item() for _ in range(100 // world)]
    assert sorted(seen) == list(range(100))


def test_dummy_loader_and_causal_lm():
    from fms_fsdp_b200.config import train_config
    from fms_fsdp_b200.utils.dataloader_utils import causal_lm, get_dummy_loader, parse_data_args
    cfg = train_config(); cfg.seq_length, cfg.vocab_size, cfg.batch_size = 8, 5, 2
    loader = get_dummy_loader(cfg, 0, 1)
    x, y = next(loader)
    # the reference stream: sample k = arange(k*seq, (k+1)*seq) % vocab (SteadyCounter advances by seq_len per sample)
    assert x.shape == (2, 8) and torch.equal(x, y) and x.dtype == torch.int32
    assert x[0].tolist() == [0, 1, 2, 3, 4, 0, 1, 2] and x[1].tolist() == [3, 4, 0, 1, 2, 3, 4, 0]
    assert next(loader)[0][0].tolist() == [(16 + j) % 5 for j in range(8)]
    i, t = causal_lm(torch.arange(6))
    assert i.tolist() == [0, 1, 2, 3, 4] and t.tolist() == [-100, 2, 3, 4, 5]
    assert parse_data_args("a,b", "1,2.5") == (["a", "b"], [1.0, 2.5])


# ------------------------------------------------------------------- interchange with the original fms-fsdp
# What the original's dataset_utils produced on this corpus, and the loader checkpoint it wrote, stored under
# tests/golden/reference (scripts/make_reference_golden.py regenerates them from a checkout of the original).
_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference")


def _golden(key):
    with open(os.path.join(_GOLDEN, "datasets.json")) as f:
        return json.load(f)[key]


@pytest.fixture(scope="module")
def reference_checkpoints(tmp_path_factory):
    """Loader checkpoints written by the original, one directory each."""
    out = tmp_path_factory.mktemp("reference_checkpoints")
    with tarfile.open(os.path.join(_GOLDEN, "loader_checkpoints.tar.xz")) as tar:
        tar.extractall(out, filter="data")
    return out


def _full_stack(D, corpus, rank, world, seq=33):
    d = D.StreamingDocDataset(corpus, rank, world, D.ArrowHandler(), -1, strip_tokens={-1}, min_length=3, seed=7)
    d = D.ScalableShardDataset(d, -1, n_logical_shards=8)
    d = D.SamplingDataset(corpus, d, -1, datasets=["dataset_1", "dataset_2"], weights=[3, 1], verbose=False)
    d = D.BufferDataset(d, seq, bos_token=None, eos_token=None, pack_hard=True)
    return D.PreloadBufferDataset(d, 50)


def _line_digests(it, n):
    """A 64-bit digest of each of the next ``n`` lines: equal lines, equal digests, at a fraction of the stored size."""
    return [hashlib.sha256(repr([int(x) for x in next(it)]).encode()).hexdigest()[:16] for _ in range(n)]


def _state_digest(obj):
    """Digest of a loader state (nested dicts, lists, scalars and tensors), independent of how it was pickled."""
    h = hashlib.sha256()

    def walk(o):
        if isinstance(o, dict):
            h.update(b"{")
            for k in sorted(o, key=repr):
                h.update(repr(k).encode())
                walk(o[k])
            h.update(b"}")
        elif isinstance(o, (list, tuple)):
            h.update(b"[")
            for x in o:
                walk(x)
            h.update(b"]")
        elif isinstance(o, torch.Tensor):
            h.update(f"{o.dtype}{tuple(o.shape)}".encode() + o.contiguous().numpy().tobytes())
        else:
            h.update(repr(o).encode())
    walk(obj)
    return h.hexdigest()


def _checkpoint_digests(path):
    return {f: _state_digest(torch.load(os.path.join(path, f), weights_only=False)) for f in sorted(os.listdir(path))}


def _write_checkpoint(D, corpus, path):
    """Two ranks of the full stack each take 40 lines, then save their loader states to ``path``."""
    stacks = [_full_stack(D, corpus, r, 2) for r in range(2)]
    its = [iter(s) for s in stacks]
    for it in its:
        take(it, 40)
    for s in stacks:
        s.save_to_path(path)


def _resume(D, corpus, world, path):
    """Line digests of the next 60 lines of each of ``world`` ranks resumed from the checkpoint at ``path``."""
    stacks = [_full_stack(D, corpus, r, world) for r in range(world)]
    for s in stacks:
        s.load_from_path(path)
    return [_line_digests(iter(s), 60) for s in stacks]


def test_token_stream_and_loader_checkpoints_interchange_with_the_reference(corpus, tmp_path, reference_checkpoints):
    """Same corpus, same pipeline as the original fms-fsdp: (1) the token streams are identical line by line; (2) a loader
    checkpoint written here is the one the original resumed at world 2, and resuming it here continues as the original
    did; one written by the original resumes here at world 4 -- a change of world size -- as it does in the original."""
    import fms_fsdp_b200.utils.dataset_utils as OURS
    assert _line_digests(iter(_full_stack(OURS, corpus, 0, 1)), 300) == _golden("stream")

    ck = str(tmp_path / "ours_to_ref")
    _write_checkpoint(OURS, corpus, ck)
    assert _checkpoint_digests(ck) == _golden("ours_to_ref checkpoint")
    assert _resume(OURS, corpus, 2, ck) == _golden("ours_to_ref")

    assert _resume(OURS, corpus, 4, str(reference_checkpoints / "ref_to_ours")) == _golden("ref_to_ours")


# ------------------------------------------------------------------------ parquet / auto handlers (raw text + tokenizer)
def make_text_corpus():
    """A local word-level tokenizer (saved so ``AutoTokenizer.from_pretrained(dir)`` works offline; it adds <s> ... </s> like
    the HF Llama tokenizers do) and a corpus with one parquet text shard and one pre-tokenised arrow shard."""
    import pyarrow.parquet as pq
    from tokenizers import Tokenizer, models, pre_tokenizers, processors
    from transformers import PreTrainedTokenizerFast
    tmp = tempfile.mkdtemp()
    words = [f"w{i}" for i in range(200)]
    vocab = {"<s>": 1, "</s>": 2, "[UNK]": 3, **{w: 10 + i for i, w in enumerate(words)}}
    tok = Tokenizer(models.WordLevel(vocab, unk_token="[UNK]"))
    tok.pre_tokenizer = pre_tokenizers.Whitespace()
    tok.post_processor = processors.TemplateProcessing(single="<s> $A </s>", special_tokens=[("<s>", 1), ("</s>", 2)])
    PreTrainedTokenizerFast(tokenizer_object=tok, unk_token="[UNK]", bos_token="<s>", eos_token="</s>").save_pretrained(f"{tmp}/tok")
    docs = [" ".join(words[(7 * d + j) % 200] for j in range(20 + d % 9)) for d in range(40)]
    os.makedirs(f"{tmp}/data/mix")
    pq.write_table(pa.table({"text": docs, "other": list(range(40))}), f"{tmp}/data/mix/part_0.parquet")
    _write(f"{tmp}/data/mix/part_1.arrow", [[300 + 50 * d + j for j in range(30)] for d in range(20)])
    return tmp, docs, vocab


@pytest.fixture(scope="module")
def text_corpus():
    return make_text_corpus()


def _text_reader(D, tmp):
    return D.StreamingDocDataset(f"{tmp}/data/mix", 0, 1, D.AutoHandler(f"{tmp}/tok", "text"), 0, strip_tokens={1, 2}, seed=3,
                                 max_chunksize=16)


def test_parquet_and_auto_handlers_tokenise_strip_and_match_the_reference(text_corpus):
    from fms_fsdp_b200.utils.dataset_utils import AutoHandler, ParquetHandler
    tmp, docs, vocab = text_corpus
    h = ParquetHandler(f"{tmp}/tok", "text")
    path = f"{tmp}/data/mix/part_0.parquet"
    assert h.is_legal(path) and not h.is_legal(f"{tmp}/data/mix/part_1.arrow") and h.length(path) == 40
    reader = h.open(path)
    want = [vocab[w] for w in docs[3].split()]
    assert h.get(reader, 3, set()) == [1] + want + [2]            # the tokenizer's own <s> ... </s>
    assert h.get(reader, 3, {1, 2}) == want                       # ... stripped when named in drop_tokens
    assert h.slice(want, 5, 4) == want[5:9]
    a = AutoHandler(f"{tmp}/tok", "text")
    assert a.is_legal(path) and a.is_legal(f"{tmp}/data/mix/part_1.arrow") and not a.is_legal(f"{tmp}/tok/tokenizer.json")
    assert a.length(path) == 40 and a.length(f"{tmp}/data/mix/part_1.arrow") == 20
    r = a.open(f"{tmp}/data/mix/part_1.arrow")
    assert a.slice(a.get(r, 2, set()), 0, 3) == [400, 401, 402]
    r = a.open(path)
    assert a.get(r, 0, {1, 2}) == [vocab[w] for w in docs[0].split()]

    # the whole reader on the mixed folder: same documents, same order as the original's classes
    import fms_fsdp_b200.utils.dataset_utils as OURS
    assert _line_digests(iter(_text_reader(OURS, tmp)), 200) == _golden("text_reader")


def test_get_data_loader_with_file_type_auto_runs_on_text_and_token_shards(text_corpus, tmp_path):
    from fms_fsdp_b200.config import train_config
    from fms_fsdp_b200.utils.dataloader_utils import get_data_loader
    tmp, docs, vocab = text_corpus
    cfg = train_config()
    cfg.data_path, cfg.datasets, cfg.weights = f"{tmp}/data", "mix", "1"
    cfg.file_type, cfg.tokenizer_path, cfg.col_name = "auto", f"{tmp}/tok", "text"
    cfg.seq_length, cfg.batch_size, cfg.num_workers, cfg.logical_shards = 24, 2, 0, 4
    cfg.bos_token, cfg.eos_token, cfg.strip_tokens = None, 0, "1,2"
    cfg.ckpt_save_path = cfg.ckpt_load_path = str(tmp_path)
    it = iter(get_data_loader(cfg, 0, 1))
    seen = set()
    for _ in range(30):
        x, y = next(it)
        assert x.shape == (2, 24) and torch.equal(x[:, 2:], y[:, 1:-1]) and bool((y[:, 0] == -100).all())
        seen.update(x.flatten().tolist())
    assert 1 not in seen and 2 not in seen and 0 in seen           # tokenizer BOS/EOS stripped, loader EOS delimits
    assert any(10 <= t < 210 for t in seen) and any(t >= 300 for t in seen)   # both the text and the token shard are read


PACKER_KW = [dict(pack_hard=False, pad_token=-5), dict(pack_hard=False, pad_token=-5, bos_token=-2, eos_token=-3),
             dict(pack_hard=True, bos_token=-2), dict(pack_hard=True, eos_token=-3, bos_token=-2)]


def _packer_stack(D, corpus, kw):
    d = D.StreamingDocDataset(corpus, 0, 1, D.ArrowHandler(), -1, seed=11, max_chunksize=40)
    d = D.SamplingDataset(corpus, d, -1, datasets=["dataset_1", "dataset_2"], weights=[1, 2], verbose=False)
    return D.BufferDataset(d, 37, **kw)


@pytest.mark.parametrize("kw", PACKER_KW)
def test_line_packer_modes_equal_the_reference(corpus, kw):
    """Every packing mode of ``BufferDataset`` (hard / soft packing, per-line BOS / EOS, padding) against the original
    class on the same sampled two-dataset stream."""
    import fms_fsdp_b200.utils.dataset_utils as OURS
    assert _line_digests(iter(_packer_stack(OURS, corpus, kw)), 250) == _golden(f"packer {kw!r}")


PARTITION_CASES = [(3, 1, None, 1, 6), (2, 0, -9, 3, 8), (4, 3, -9, 60, 12), (1, 0, None, 101, 5)]


def _partition_stack(D, corpus, world, rank, bos, min_len, nlog):
    d = D.StreamingDocDataset(os.path.join(corpus, "dataset_2") if min_len < 101 else corpus, rank, world, D.ArrowHandler(),
                              -1, bos_token=bos, min_length=min_len, seed=5, max_chunksize=33)
    return D.ScalableShardDataset(d, -1, n_logical_shards=nlog * world)


@pytest.mark.parametrize("world,rank,bos,min_len,nlog", PARTITION_CASES)
def test_reader_partitioning_options_equal_the_reference(corpus, world, rank, bos, min_len, nlog):
    """Document reader + logical shards under different partitionings, BOS insertion and minimum document lengths (which
    drop all of dataset_2's 50-token documents at 60 and everything at 101): chunk for chunk what the original yields."""
    # (50 tokens + delimiter + BOS = 52 < 60)
    import fms_fsdp_b200.utils.dataset_utils as OURS
    case = (world, rank, bos, min_len, nlog)
    if min_len >= 60:
        # nothing survives the length filter: the original spins forever in that case; here it is an error that says why
        with pytest.raises(RuntimeError, match="min_length"):
            next(iter(_partition_stack(OURS, corpus, *case)))
        return
    assert _line_digests(iter(_partition_stack(OURS, corpus, *case)), 150) == _golden(f"partition {case!r}")


RESCALE_CASES = [(True, 3, 2), (False, 4, 6), (True, 6, 4), (False, 2, 1)]


def _rescale_stack(D, corpus, rank, world):
    d = D.StreamingDocDataset(corpus, rank, world, D.ArrowHandler(), -1, strip_tokens={-1}, min_length=3, seed=7)
    d = D.ScalableShardDataset(d, -1, n_logical_shards=12)
    d = D.SamplingDataset(corpus, d, -1, datasets=["dataset_1", "dataset_2"], weights=[3, 1], verbose=False)
    d = D.BufferDataset(d, 33, bos_token=None, eos_token=None, pack_hard=True)
    return D.PreloadBufferDataset(d, 50)


def _rescale_write(D, corpus, world, path):
    olds = [_rescale_stack(D, corpus, r, world) for r in range(world)]
    for s in olds:
        take(iter(s), 30)
    for s in olds:
        s.save_to_path(path)


def _rescale_resume(D, corpus, world, path):
    out = []
    for r in range(world):
        s = _rescale_stack(D, corpus, r, world)
        s.load_from_path(path)
        out.append(_line_digests(iter(s), 40))
    return out


@pytest.mark.parametrize("writer_is_ours,old_world,new_world", RESCALE_CASES)
def test_rescaled_resume_equals_the_reference_for_more_world_size_pairs(corpus, tmp_path, reference_checkpoints, writer_is_ours,
                                                                        old_world, new_world):
    """Loader checkpoints written at ``old_world`` ranks by one implementation, resumed at ``new_world`` ranks by both: every
    new rank continues with the same lines in either implementation (shrinking, growing, non-divisible pairs).  A checkpoint
    written here must be the one the original resumed; one written by the original is stored."""
    import fms_fsdp_b200.utils.dataset_utils as OURS
    key = f"rescale {(writer_is_ours, old_world, new_world)!r}"
    if writer_is_ours:
        ck = str(tmp_path / "ck")
        _rescale_write(OURS, corpus, old_world, ck)
        assert _checkpoint_digests(ck) == _golden(key + " checkpoint")
    else:
        ck = str(reference_checkpoints / f"rescale_{old_world}_to_{new_world}")
    assert _rescale_resume(OURS, corpus, new_world, ck) == _golden(key)


def _worker_loader(D, corpus, path):
    d = D.StreamingDocDataset(corpus, 1, 2, D.ArrowHandler(), -1, min_length=3, seed=3)
    d = D.ScalableShardDataset(d, -1, n_logical_shards=8)
    d = D.SamplingDataset(corpus, d, -1, datasets=["dataset_1", "dataset_2"], weights=[1, 1], verbose=False)
    d = D.BufferDataset(d, 21, pack_hard=True)
    d = D.PreloadBufferDataset(d, 20)
    d = D.PreprocessDataset(d, torch.IntTensor)
    d = D.CheckpointDataset(d, path, 5, 2, path)
    return torch.utils.data.DataLoader(d, num_workers=2, batch_size=2)


def _worker_run(D, corpus, path):
    """Digests of 24 batches through two worker processes, and the auto-checkpoints they left under ``path``."""
    it = iter(_worker_loader(D, corpus, path))
    batches = [_state_digest(next(it))[:16] for _ in range(24)]
    del it
    steps = sorted(os.listdir(os.path.join(path, "checkpoints")))
    return {"batches": batches, "checkpoints": steps,
            "last_checkpoint_files": sorted(os.listdir(os.path.join(path, "checkpoints", steps[-1]))) if steps else []}


def test_multi_worker_dataloader_stream_equals_the_reference(corpus, tmp_path):
    """Through ``torch.utils.data.DataLoader(num_workers=2)``: each worker process derives its own partition from
    (rank, world, worker id); the batches are the original's, and so are the in-worker auto-checkpoints."""
    import fms_fsdp_b200.utils.dataset_utils as OURS
    mine = _worker_run(OURS, corpus, str(tmp_path / "ours"))
    assert mine["checkpoints"], mine
    assert mine == _golden("multi_worker")
