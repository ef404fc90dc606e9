"""The four CPU cases in which tests/test_models_cpu.py compares models.py with the original end-to-end-SLU project: seeded
init + forward, the freeze / unfreeze schedule, the ASR forward and the seq2seq surface.  Each case runs the same code on any
`models` module -- this repository's, or the original's (import_reference) -- and returns named arrays.  The tests compare
models.py with the original directly when SLU_REFERENCE names a checkout of it, and with golden_reference_cpu.npz otherwise.

    python tests/reference_cases.py [ORIGINAL_CHECKOUT]

rewrites golden_reference_cpu.npz from the original's models.py when a checkout is given, else from this repository's models.py;
the file's `source` entry says which.  Parameter tensors are stored as digests (float64 sum, sum of squares and 64 seeded
elements per tensor) to keep the file small."""
import importlib
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from util import make_config  # noqa: E402

GOLDEN_FILE = os.path.join(HERE, "golden", "golden_reference_cpu.npz")
UNFREEZE_CASES = ((1, 1), (2, 1), (2, 3), (0, 1))            # (unfreezing_type, starting unfreezing_index)
S2S_LABELS = ["<sos>"] + list("abcdefghij {}:'\",") + ["<eos>"]


def import_reference(path):
    """The original project's models module, imported unmodified from `path` (soundfile / textgrid, unused on these paths, are
    stubbed); this repository's `models` stays what `import models` resolves to."""
    saved = sys.modules.get("models")
    for m in ("soundfile", "textgrid"):
        sys.modules.setdefault(m, types.ModuleType(m))
    sys.path.insert(0, path)
    sys.modules.pop("models", None)
    sys.dont_write_bytecode = True
    try:
        ref_models = importlib.import_module("models")
    finally:
        sys.path.remove(path)
        if saved is not None:
            sys.modules["models"] = saved
        else:
            sys.modules.pop("models", None)
    assert ref_models.__file__.startswith(path)
    sys.modules["ref_models"] = ref_models
    return ref_models


def _cpu(model):
    model.cpu()
    model.is_cuda = False
    return model


def _state(prefix, model):
    return {prefix + "state/" + k: v.detach().clone() for k, v in model.state_dict().items()} | \
           {prefix + "keys": np.array(list(model.state_dict()))}


def init_forward(m):
    """Default config, torch.manual_seed(1234): the initial state dict, then loss / acc / intent logits on a random batch."""
    cfg = make_config()
    torch.manual_seed(1234)
    model = _cpu(m.Model(cfg))
    x = 0.1 * torch.randn(2, 9000)
    y = torch.tensor([[1, 2, 3], [0, 13, 0]])
    model.eval()
    loss, acc = model(x, y)
    logits, pred = model.predict_intents(x)
    return _state("init_forward/", model) | {"init_forward/loss": loss.detach(), "init_forward/acc": acc.detach(),
                                              "init_forward/logits": logits.detach(), "init_forward/pred": pred}


def unfreeze(m):
    """requires_grad of every parameter and unfreezing_index after each of 9 unfreeze_one_layer calls, per UNFREEZE_CASES."""
    flags, index = [], []
    for utype, start in UNFREEZE_CASES:
        model = m.Model(make_config(unfreezing_type=utype))
        model.unfreezing_index = start
        model.freeze_all_layers()
        for _ in range(9):
            model.unfreeze_one_layer()
            flags.append([p.requires_grad for p in model.parameters()])
            index.append(model.unfreezing_index)
    return {"unfreeze/requires_grad": np.array(flags, dtype=np.uint8).reshape(len(UNFREEZE_CASES), 9, -1),
            "unfreeze/index": np.array(index).reshape(len(UNFREEZE_CASES), 9)}


def asr_forward(m):
    """PretrainedModel (pretraining_type 2), torch.manual_seed(7): the four outputs of forward and both posteriors."""
    torch.manual_seed(7)
    model = m.PretrainedModel(make_config(pretraining_type=2)).cpu().eval()
    x = 0.1 * torch.randn(2, 5120)
    yp = torch.randint(-1, 42, (2, 8))
    yw = torch.randint(-1, 10000, (2, 2))
    out = model(x, yp, yw)
    post_p, post_w = model.compute_posteriors(x)
    return {"asr/outputs": torch.stack([o.detach().reshape(()) for o in out]), "asr/phoneme_posteriors": post_p.detach(),
            "asr/word_posteriors": post_w.detach()}


def seq2seq(m):
    """seq2seq config, torch.manual_seed(11): the initial state dict, the teacher-forced loss and a 4-beam search of 6 steps."""
    cfg = make_config("seq2seq")
    cfg.Sy_intent = list(S2S_LABELS)
    torch.manual_seed(11)
    model = _cpu(m.Model(cfg))
    S, U = len(cfg.Sy_intent), 7
    x = 0.1 * torch.randn(3, 6000)
    idx = torch.randint(1, S - 1, (3, U))
    idx[:, 0] = 0
    idx[:, -1] = S - 1
    y = torch.nn.functional.one_hot(idx, S).float()
    model.eval()
    loss, _ = model(x, y)
    enc = model.encoder(model.pretrained_model.compute_features(x))
    scores, beam = model.decoder.infer(enc, cfg.Sy_intent, B=4, y_lengths=[6])
    return _state("seq2seq/", model) | {"seq2seq/loss": loss.detach(), "seq2seq/beam_scores": scores.detach(),
                                         "seq2seq/beam_ids": beam.argmax(-1),
                                         "seq2seq/best": np.array(model.one_hot_to_string(beam[0, 0], cfg.Sy_intent))}


CASES = {"init_forward": init_forward, "unfreeze": unfreeze, "asr": asr_forward, "seq2seq": seq2seq}


def digest(out):
    """Parameter tensors -> float64 sum, sum of squares and 64 elements at seeded positions; everything else as numpy."""
    res = {}
    for k, v in out.items():
        if "/state/" in k:
            flat = v.reshape(-1)
            pos = np.random.RandomState(0).randint(0, flat.numel(), size=min(64, flat.numel()))
            d = flat.double()
            res[k + "/sum"] = np.float64(d.sum().item())
            res[k + "/sumsq"] = np.float64((d * d).sum().item())
            res[k + "/sample"] = flat[torch.from_numpy(pos)].numpy()
        else:
            res[k] = v.numpy() if torch.is_tensor(v) else np.asarray(v)
    return res


def golden(case):
    with np.load(GOLDEN_FILE) as z:
        return {k: z[k] for k in z.files if k.startswith(case + "/")}


if __name__ == "__main__":
    root = os.path.dirname(HERE)
    sys.path.insert(0, root)
    if len(sys.argv) > 1:
        mod, source = import_reference(os.path.abspath(sys.argv[1])), "original end-to-end-SLU models.py"
    else:
        import models as mod
        source = "this repository's models.py"
    arrays = {"source": np.array(source)}
    for fn in CASES.values():
        arrays.update(digest(fn(mod)))
    np.savez_compressed(GOLDEN_FILE, **arrays)
    print(GOLDEN_FILE, len(arrays), "arrays from", source, os.path.getsize(GOLDEN_FILE), "bytes")
