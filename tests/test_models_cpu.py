"""Host-side drop-in surface (models.py) on CPU: state_dict layout, known answer, freeze schedule,
config reader, C-ABI symbol table.  The cases of tests/reference_cases.py compare models.py with the
original end-to-end-SLU project: directly when SLU_REFERENCE names a checkout of it, else with the
outputs recorded in golden_reference_cpu.  Driving the original's own Trainer needs the checkout."""
import ctypes
import importlib
import os
import re
import sys
import types

import numpy as np
import pytest
import torch

import models
import reference_cases as RC
from util import ckpt_params, golden, load_test_wav, make_config, rel_err

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("SLU_REFERENCE", "")
has_ref = bool(REF) and os.path.isfile(os.path.join(REF, "models.py"))


def cpu_model(cfg=None):
    m = models.Model(cfg or make_config())
    m.cpu(); m.is_cuda = False
    return m


def load_ckpt(m):
    sd = m.state_dict()
    ck = ckpt_params()
    missing = set(sd) - set(ck)
    assert missing == {"pretrained_model.word_linear.weight", "pretrained_model.word_linear.bias"}
    for k, v in ck.items():
        assert sd[k].shape == v.shape and sd[k].dtype == v.dtype, k
    sd.update(ck)
    m.load_state_dict(sd, strict=True)


def test_state_dict_layout_and_known_answer():
    m = cpu_model().eval()
    load_ckpt(m)
    assert m.state_dict()["pretrained_model.phoneme_layers.0.filt_b1"].dtype == torch.float64
    g = golden("golden_testwav.npz")
    logits, pred = m.predict_intents(load_test_wav())
    assert rel_err(logits, g["logits"]) < 2e-5
    assert pred.tolist() == [[1, 2, 1]]
    # decode_intents with an index-named table: README.md:42 {activate, lights, kitchen} = (1, 2, 1)
    assert m.decode_intents(load_test_wav()) == [["action_1", "object_2", "location_1"]]
    assert rel_err(m.pretrained_model.compute_features(load_test_wav()), g["features"]) < 2e-5


def test_unfreeze_schedule_and_print(capsys):
    cfg = make_config("unfreeze_all_layers", pretraining_type=2)
    cfg.pretraining_type = 0          # no checkpoint on disk ...
    m = cpu_model(cfg)
    m.unfreezing_index = 1            # ... but exercise the pretraining_type=2 schedule
    m.freeze_all_layers()
    order = []
    names = lambda: [l.name for l in list(m.pretrained_model.phoneme_layers) + list(m.pretrained_model.word_layers)
                     if models.has_params(l) and not models.is_frozen(l)]
    for _ in range(8):
        m.unfreeze_one_layer()
        order.append(set(names()))
    seq = [sorted(order[0])] + [sorted(order[i] - order[i - 1]) for i in range(1, 8)]
    assert seq == [["word_rnn1"], ["word_rnn0"], ["phone_rnn1"], ["phone_rnn0"], ["conv2"], ["conv1"], ["sinc0"], []]
    m.print_frozen()
    assert "sinc0: unfrozen" in capsys.readouterr().out
    # unused ASR heads are never frozen (SURVEY.md 5.6)
    assert m.pretrained_model.word_linear.weight.requires_grad


def test_config_reader_matches_cfg_semantics():
    cfg = make_config("unfreeze_all_layers", pretraining_type=2)
    assert cfg.cnn_N_filt == [80, 60, 60] and cfg.cnn_len_filt == [401, 5, 5] and cfg.cnn_stride == [80, 1, 1]
    assert cfg.phone_downsample_factor == 640 and cfg.word_downsample_factor == 2560
    assert cfg.unfreezing_type == 2 and cfg.seq2seq is False and cfg.train_wording_path is None
    s2s = make_config("seq2seq")
    assert s2s.seq2seq and s2s.intent_decoder_dim == 256 and s2s.num_intent_decoder_layers == 2


def test_forward_loss_acc_matches_golden_on_cpu():
    from oracle import torch_ref as R
    g = golden("golden_synth_small.npz")
    m = cpu_model().eval()
    sd = m.state_dict()
    sd.update({k: v for k, v in R.synthetic_params(seed=int(g["pseed"])).items() if k in sd})
    m.load_state_dict(sd)
    x, y = R.synthetic_batch(int(g["B"]), int(g["T"]), seed=int(g["bseed"]))
    loss, acc = m(x, y)
    loss.backward()
    assert abs(loss.item() - float(g["loss"])) < 1e-5 * float(g["loss"])
    assert acc.item() == float(g["acc"])
    named = dict(m.named_parameters())
    for k in ("pretrained_model.phoneme_layers.0.filt_b1", "pretrained_model.phoneme_layers.0.filt_band",
              "pretrained_model.phoneme_layers.5.bias", "intent_layers.4.weight"):
        assert rel_err(named[k].grad.flatten(), g["g/" + k]) < 1e-4, k
        assert named[k].grad.dtype == named[k].dtype


def test_cabi_library_exports_declared_symbols():
    hdr = open(os.path.join(ROOT, "include", "slu_b200.h")).read()
    declared = set(re.findall(r"\bint\s+(slu_\w+)\s*\(", hdr))
    assert len(declared) >= 7
    lib_mod = importlib.import_module("end-to-end-slu_b200._lib")
    assert os.path.isfile(lib_mod.LIB_PATH), "build the library first: python __graft_entry__.py"
    lib = ctypes.CDLL(lib_mod.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    assert declared == set(lib_mod.SIGNATURES), declared ^ set(lib_mod.SIGNATURES)


def test_missing_library_fails_loudly(monkeypatch):
    lib_mod = importlib.import_module("end-to-end-slu_b200._lib")
    monkeypatch.setattr(lib_mod, "_lib", None)
    monkeypatch.setattr(lib_mod, "LIB_PATH", "/nonexistent/libslu_b200.so")
    with pytest.raises(RuntimeError, match="no fallback"):
        lib_mod.load()


# ---- comparison with the original project: live with SLU_REFERENCE, else its recorded outputs -------------
@pytest.fixture(scope="module")
def reference():
    if not has_ref:
        pytest.skip("needs the original end-to-end-SLU source tree (set SLU_REFERENCE)")
    saved = {k: sys.modules.get(k) for k in ("models", "data", "soundfile", "textgrid")}
    for m in ("soundfile", "textgrid"):
        sys.modules[m] = types.ModuleType(m)
    sys.path.insert(0, REF)
    del sys.modules["models"]
    sys.dont_write_bytecode = True
    ref_models = importlib.import_module("models")
    assert ref_models.__file__.startswith(REF)
    sys.path.remove(REF)
    sys.modules["ref_models"] = ref_models
    sys.modules["models"] = saved["models"]
    yield ref_models
    for m in ("soundfile", "textgrid"):
        sys.modules.pop(m, None)


@pytest.fixture(scope="module")
def expected():
    """case name -> the original's arrays for that case: computed live from SLU_REFERENCE, else read from the golden file."""
    if has_ref:
        ref = RC.import_reference(REF)
        return lambda case: RC.CASES[case](ref)
    return RC.golden


def check_state(got, exp, prefix):
    """Same state_dict keys in the same order and equal tensors (against the golden file: equal sums, sums of squares and
    sampled elements -- the sums up to the rounding of a float64 reduction)."""
    keys = [str(k) for k in got[prefix + "keys"]]
    assert keys == [str(k) for k in exp[prefix + "keys"]]
    for k in keys:
        name, t = prefix + "state/" + k, got[prefix + "state/" + k]
        if name in exp:
            assert torch.equal(t, exp[name]), k
            continue
        d = RC.digest({name: t})
        scale = 1e-12 * (float(d[name + "/sumsq"]) * t.numel()) ** 0.5
        assert abs(float(d[name + "/sum"]) - float(exp[name + "/sum"])) <= scale, k
        assert abs(float(d[name + "/sumsq"]) - float(exp[name + "/sumsq"])) <= 1e-12 * float(exp[name + "/sumsq"]), k
        assert np.array_equal(d[name + "/sample"], exp[name + "/sample"]), k


def test_same_seed_same_init_and_same_forward_as_reference(expected):
    P = "init_forward/"
    got, exp = RC.init_forward(models), expected("init_forward")
    check_state(got, exp, P)
    assert abs(float(got[P + "loss"]) - float(exp[P + "loss"])) < 1e-5 and float(got[P + "acc"]) == float(exp[P + "acc"])
    assert rel_err(got[P + "logits"], exp[P + "logits"]) < 2e-5
    assert np.array_equal(np.asarray(got[P + "pred"]), np.asarray(exp[P + "pred"]))


def test_unfreeze_matches_reference_for_all_types(expected):
    got, exp = RC.unfreeze(models), expected("unfreeze")
    for k in ("unfreeze/requires_grad", "unfreeze/index"):
        for c, (utype, start) in enumerate(RC.UNFREEZE_CASES):
            for step in range(9):
                assert np.array_equal(got[k][c, step], exp[k][c, step]), (k, utype, start, step)


def test_asr_forward_matches_reference(expected):
    got, exp = RC.asr_forward(models), expected("asr")
    for a, b in zip(np.asarray(got["asr/outputs"]), np.asarray(exp["asr/outputs"])):
        assert abs(float(a) - float(b)) < 1e-5
    assert rel_err(got["asr/phoneme_posteriors"], exp["asr/phoneme_posteriors"]) < 2e-5
    assert rel_err(got["asr/word_posteriors"], exp["asr/word_posteriors"]) < 2e-5


def test_seq2seq_surface_matches_reference(expected):
    """config 5 (repaired seq2seq cfg): same construction, teacher-forced loss and beam search as the reference, on CPU."""
    P = "seq2seq/"
    got, exp = RC.seq2seq(models), expected("seq2seq")
    check_state(got, exp, P)
    assert abs(float(got[P + "loss"]) - float(exp[P + "loss"])) < 1e-4 * abs(float(exp[P + "loss"]))
    # beam search (shortened: the reference runs a fixed 200 steps unless y_lengths is given)
    assert rel_err(got[P + "beam_scores"], exp[P + "beam_scores"]) < 1e-4
    assert np.array_equal(np.asarray(got[P + "beam_ids"]), np.asarray(exp[P + "beam_ids"]))
    assert str(got[P + "best"]) == str(exp[P + "best"])


def test_packed_gru_parameters_keep_identity_values_and_checkpoints():
    """ops.packed_params re-homes the 8 tensors of a bidirectional GRU into one buffer in kernel order (host logic only):
    Parameter objects, values, optimizer updates, load_state_dict and nn.GRU's own CPU forward must be unaffected."""
    import importlib
    ops = importlib.import_module("end-to-end-slu_b200").ops
    g = torch.nn.GRU(60, 128, batch_first=True, bidirectional=True)
    sd = {k: v.clone() for k, v in g.state_dict().items()}
    ids = [id(p) for p in g.parameters()]
    x = torch.randn(2, 5, 60)
    y0 = g(x)[0].detach().clone()
    v = ops.packed_params(g)
    assert [id(p) for p in g.parameters()] == ids
    assert all(torch.equal(t, sd[k]) for k, t in g.state_dict().items())
    assert torch.equal(v[0], torch.cat([g.weight_ih_l0, g.weight_ih_l0_reverse]))
    assert torch.equal(v[1], torch.cat([g.bias_ih_l0, g.bias_ih_l0_reverse]))
    assert torch.equal(v[2], torch.stack([g.weight_hh_l0, g.weight_hh_l0_reverse]))
    assert torch.equal(v[3], torch.stack([g.bias_hh_l0, g.bias_hh_l0_reverse]))
    assert torch.equal(g(x)[0], y0)
    assert ops.packed_params(g) is v                                   # still aliased: nothing to do
    opt = torch.optim.Adam(g.parameters(), lr=0.1)
    g(x)[0].sum().backward()
    opt.step()
    assert ops.packed_params(g) is v and torch.equal(v[0], torch.cat([g.weight_ih_l0, g.weight_ih_l0_reverse]))
    g.load_state_dict(sd)
    assert torch.equal(v[0][:384], sd["weight_ih_l0"])
    g.double(); g.float()                                              # Module._apply re-homes the parameters
    v2 = ops.packed_params(g)
    assert v2 is not v and torch.equal(v2[0][:384], sd["weight_ih_l0"]) and torch.equal(g(x)[0], y0)


def test_premask_shapes_and_draw_order(monkeypatch):
    """engine._premask generates the keep-masks of several GRU stacks ahead of time; shapes follow the downsampling chain and the
    draw order is the layer order (host logic; a supplied `_drop_mask` -- as the golden dropout test uses -- is called in line)."""
    import importlib
    eng = importlib.import_module("end-to-end-slu_b200").engine
    calls = []

    def fake(shape, p, training, device):
        calls.append((tuple(shape), p, training))
        return torch.zeros(shape)
    monkeypatch.setattr(eng, "_drop_mask", fake)
    stacks = [[(None, 0.5, 2), (None, 0.5, 2)], [(None, 0.25, 2), (None, 0.5, 1)]]
    (m0, m1), join = eng._premask(stacks, 3, 401, True, torch.device("cpu"))
    assert join is None
    assert [c[0] for c in calls] == [(3, 401, 256), (3, 201, 256), (3, 101, 256), (3, 51, 256)]
    assert [c[1] for c in calls] == [0.5, 0.5, 0.25, 0.5]
    assert [tuple(m.shape) for m in m0] == [(3, 401, 256), (3, 201, 256)] and [tuple(m.shape) for m in m1] == [(3, 101, 256), (3, 51, 256)]


def test_prefetcher_iteration_protocol_without_a_device(monkeypatch):
    """loader.DevicePrefetcher's iteration logic (order, early close, loader exceptions surfacing in the consumer) for the in-line
    and the helper-thread variant, with the device staging stubbed out (host logic only)."""
    import importlib
    ld = importlib.import_module("end-to-end-slu_b200").loader
    monkeypatch.setattr(ld, "_copy_stream", lambda device: None)
    monkeypatch.setattr(torch.cuda, "set_device", lambda d: None)
    monkeypatch.setattr(ld.DevicePrefetcher, "_stage", lambda self, batch, stream: (batch, "ready"))
    monkeypatch.setattr(ld.DevicePrefetcher, "_hand_over", lambda self, staged: staged[0])
    for background in (False, True):
        mk = lambda it: ld.DevicePrefetcher(it, device="cuda:0", background=background)
        assert list(mk([(i, i * i) for i in range(5)])) == [(i, i * i) for i in range(5)]
        assert list(mk([])) == []

        def bad():
            yield (1, 1)
            raise ValueError("boom")
        try:
            list(mk(bad()))
            raised = False
        except ValueError:
            raised = True
        assert raised
        it = iter(mk([(i,) for i in range(100)]))
        assert next(it) == (0,) and next(it) == (1,)
        it.close()                                         # abandoning the epoch must not hang (helper thread joins)


def test_reference_trainer_drives_this_model_unchanged(reference, tmp_path, capsys):
    """SURVEY 8(a9)/(b): the UNMODIFIED reference `training.Trainer` (imported from the reference tree, resolving `from models
    import ...` to this repo's models.py) trains this Model for an epoch of synthetic batches on the CPU; the same Trainer code
    over the reference's own Model from the same seed must land on the same losses and the same updated parameters."""
    import importlib.util
    saved_data = sys.modules.get("data")
    sys.path.insert(0, REF)
    try:
        sys.modules.pop("data", None)
        sys.modules.pop("training", None)
        for m in ("soundfile", "textgrid"):
            sys.modules.setdefault(m, types.ModuleType(m))
        training = importlib.import_module("training")            # reference/training.py: `from models import ...` -> OUR models
    finally:
        sys.path.remove(REF)
    assert training.__file__.startswith(REF) and training.Model is models.Model
    # the same Trainer source bound to the reference's own classes (isinstance(model, PretrainedModel) picks lr / folder)
    spec = importlib.util.spec_from_file_location("training_ref", os.path.join(REF, "training.py"))
    training_ref = importlib.util.module_from_spec(spec)
    sys.modules["models"] = reference
    try:
        spec.loader.exec_module(training_ref)
    finally:
        sys.modules["models"] = models
    assert training_ref.Model is reference.Model

    class Loader(list):
        pass

    class FakeSLU:                      # Trainer.train only needs `.loader`; it is not an ASRDataset -> SLU branch
        def __init__(self, batches):
            self.loader = Loader(batches)
    g = torch.Generator().manual_seed(5)
    batches = [(0.1 * torch.randn(3, 8000, generator=g), torch.stack([torch.randint(0, v, (3,), generator=g) for v in (6, 14, 4)], 1))
               for _ in range(3)]
    out = {}
    for name, mod, trainer_mod in (("new", models, training), ("ref", reference, training_ref)):
        cfg = make_config("unfreeze_all_layers")
        cfg.folder = str(tmp_path / name)
        os.makedirs(os.path.join(cfg.folder, "training"))
        torch.manual_seed(77)
        m = mod.Model(cfg)
        m.cpu(); m.is_cuda = False
        for layer in list(m.pretrained_model.phoneme_layers) + list(m.pretrained_model.word_layers):
            for q in layer.parameters():
                q.requires_grad = True            # fully unfrozen, dropout active: one generator seed drives both runs
        trainer = trainer_mod.Trainer(model=m, config=cfg)
        torch.manual_seed(99)
        acc, loss = trainer.train(FakeSLU(batches), print_interval=10 ** 9)
        out[name] = (acc, loss, {k: v.detach().clone() for k, v in m.state_dict().items()})
        assert os.path.isfile(os.path.join(cfg.folder, "training", "log.csv"))
    capsys.readouterr()
    (a_n, l_n, sd_n), (a_r, l_r, sd_r) = out["new"], out["ref"]
    assert abs(l_n - l_r) < 1e-4 * abs(l_r) and a_n == a_r
    for k in sd_r:
        assert rel_err(sd_n[k], sd_r[k]) < 1e-4, k
    if saved_data is not None:
        sys.modules["data"] = saved_data


def test_seq2seq_cpu_path_matches_the_reference_golden():
    """config 5 without the reference tree (GPU box): same seed -> same default init (checksum), then the teacher-forced loss,
    log-likelihoods and the best beam hypothesis of the reference's Model (tests/golden/make_golden.py section 6)."""
    g = golden("golden_seq2seq.npz")
    cfg = make_config("seq2seq")
    cfg.Sy_intent = ["<sos>"] + list("abcdefghij {}:'\",") + ["<eos>"]
    torch.manual_seed(int(g["seed"]))
    m = cpu_model(cfg).eval()
    psum = sum(v.detach().double().abs().sum().item() for v in m.state_dict().values())
    assert abs(psum - float(g["param_abs_sum"])) < 1e-9 * psum
    from oracle import torch_ref as R
    x, _ = R.synthetic_batch(int(g["B"]), int(g["T"]), seed=int(g["bseed"]))
    y = torch.nn.functional.one_hot(torch.from_numpy(g["idx"].astype(np.int64)), len(cfg.Sy_intent)).float()
    with torch.no_grad():
        loss, _ = m(x, y)
        enc = m.encoder(m.pretrained_model.compute_features(x))
        scores, beam = m.decoder.infer(enc, cfg.Sy_intent, B=4, y_lengths=[6])
    assert abs(loss.item() - float(g["loss"])) < 1e-5 * float(g["loss"])
    assert rel_err(enc, g["enc"]) < 2e-5 and rel_err(scores, g["beam_scores"]) < 1e-5
    assert np.array_equal(beam.argmax(-1).numpy(), g["beam_ids"])


def test_sharded_bucket_batch_sampler_shards_and_buckets():
    """SURVEY 8(f) rank 4: per-rank disjoint shards of one global batch, full coverage, same permutation on every rank, less
    padding than the reference's plain shuffle, usable as a DataLoader batch_sampler with the reference's pad-collate contract."""
    loader = importlib.import_module("end-to-end-slu_b200.loader")
    rs = np.random.RandomState(0)
    lengths = (16000 * (1.0 + 3.0 * rs.beta(2, 5, size=1003))).astype(int).tolist()      # 1-4 s, skewed like FSC
    world, bs = 4, 8
    samplers = [loader.ShardedBucketBatchSampler(lengths, bs, rank=r, world=world, seed=7, bucket_batches=10) for r in range(world)]
    per_rank = [list(s) for s in samplers]
    assert len({len(b) for b in per_rank}) == 1 and len(per_rank[0]) == len(samplers[0]) == -(-1003 // (bs * world))
    seen = []
    for step in range(len(per_rank[0])):
        shard = [per_rank[r][step] for r in range(world)]
        assert all(len(b) == bs for b in shard)
        flat = [i for b in shard for i in b]
        assert len(set(flat)) == len(flat)                           # ranks are disjoint within a step
        means = [np.mean([lengths[i] for i in b]) for b in shard]
        assert max(means) - min(means) < 0.1 * np.mean(means)       # same length profile on every rank
        seen += flat
    assert set(seen) == set(range(1003))                            # every utterance once per epoch (+ wrap-around fill)
    assert len(seen) - 1003 == (-1003) % (bs * world)
    plain = list(loader.ShardedBucketBatchSampler(None, bs, rank=0, world=world, seed=7, n_items=1003))   # the reference's plain shuffle
    plain_pad = 1.0 - sum(sum(lengths[i] for i in b) for b in plain) / sum(max(lengths[i] for i in b) * len(b) for b in plain)
    assert samplers[0].padding_fraction() < 0.35 * plain_pad
    e0 = list(samplers[1]); samplers[1].set_epoch(1); e1 = list(samplers[1]); samplers[1].set_epoch(0)
    assert e0 == list(samplers[1]) and e0 != e1                      # deterministic per epoch, reshuffled across epochs
    drop = loader.ShardedBucketBatchSampler(lengths, bs, rank=1, world=world, seed=7, drop_last=True)
    assert len(list(drop)) == len(drop) == 1003 // (bs * world)

    class Wavs(torch.utils.data.Dataset):                            # contract of data.py:373-376: (x [T_i], y [3])
        def __len__(self):
            return 1003

        def __getitem__(self, i):
            return torch.full((lengths[i] // 100,), float(i)), torch.tensor([i % 6, i % 14, i % 4])

    def collate(batch):                                              # pad-and-stack like CollateWavsSLU (data.py:344-391)
        T = max(len(x) for x, _ in batch)
        return torch.stack([torch.nn.functional.pad(x, (0, T - len(x))) for x, _ in batch]), torch.stack([y for _, y in batch])
    dl = torch.utils.data.DataLoader(Wavs(), batch_sampler=samplers[2], collate_fn=collate)
    x, y = next(iter(dl))
    assert x.shape[0] == bs and y.shape == (bs, 3)
