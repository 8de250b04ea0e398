"""Differential tests against the original BERT-PyTorch code (CPU): the unmodified original modules (with the
torch-native shims of baseline/shims standing in for apex / dllogger / ...) were run on fixed inputs, their results are
stored in tests/golden/reference_parity.pkl.gz, and this repository runs on the same inputs and is compared:

* model zoo: the original's state dict loads strictly into our models; logits agree to float precision
* tokenizers (BasicTokenizer / WordpieceTokenizer), SQuAD featurisation and n-best post-processing
* LR schedulers coupled to the optimizer step, BertAdam updates, distributed sampler chunking

The golden file is rewritten from a checkout of the original project with

    python tests/test_reference_parity.py PATH_TO_ORIGINAL_CHECKOUT

To keep it small, model weights on the original side are drawn from a seed and the tensor's name (``det_fill``) and are
regenerated here instead of stored, trained weights and gradients are kept as a fixed sample per tensor, and random
inputs the original drew from a seed are drawn again here."""
import gzip
import hashlib
import json
import os
import pickle
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_parity.pkl.gz")
WORK = "<work>"                  # stands for the per-run scratch directory in the stored paths

# shared by the original-side script (prepended to REF_SCRIPT) and this module
FILL_SRC = r'''
def draw(name, shape, seed):
    """Weights of tensor ``name``: a function of the seed, the name and the shape only (LayerNorm scales around 1)."""
    import zlib
    import numpy as np
    a = np.random.default_rng([seed, zlib.crc32(name.encode())]).standard_normal(tuple(shape)).astype(np.float32) * 0.05
    return a + np.float32(1.0) if name.endswith("LayerNorm.weight") else a


def det_fill(state, seed):
    """Overwrite a state dict in place with ``draw``; tensors sharing storage (tied weights) keep the first name's."""
    import torch
    seen = set()
    with torch.no_grad():
        for k, v in state.items():
            if v.data_ptr() not in seen:
                seen.add(v.data_ptr())
                v.copy_(torch.from_numpy(draw(k, v.shape, seed)))
'''
exec(FILL_SRC)
FILL_SEED, TRAIN_SEED = 0, 77              # the seeds REF_SCRIPT passes to det_fill


def _sample_idx(n, k=128):
    """Fixed flat positions at which trained weights / gradients of an n-element tensor are kept."""
    return np.arange(n) if n <= k else np.sort(np.random.default_rng(n).choice(n, k, replace=False))


def _sample(a):
    return np.asarray(a).ravel()[_sample_idx(np.asarray(a).size)]


def _digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]

MODEL_CFG = dict(vocab_size=120, hidden_size=32, num_hidden_layers=2, num_attention_heads=4, intermediate_size=64,
                 hidden_act="gelu", hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1, max_position_embeddings=64,
                 type_vocab_size=2, initializer_range=0.02, next_sentence=True)
VOCAB = ["[PAD]", "[UNK]", "[CLS]", "[SEP]", "[MASK]", "the", "capital", "of", "france", "is", "paris", ".", "river",
         "seine", "flows", "through", "what", "?", "who", "wrote", "hamlet", "a", "play", "was", "written", "by",
         "william", "shakespeare", "##s", "##ing", "un", "##aff", "##able", ",", "-", "'", "1603", "in", "and", "it"]
TEXTS = ["The capital of France is Paris.", "  Hello,\tWORLD!! unaffable-playing  ", "naïve café — 東京 is big",
         "Who wrote Hamlet? William Shakespeare's play, in 1603.", "", "x" * 120]


def _fuzz_texts(n=250, seed=13):
    """Random strings over Latin / accented / CJK / punctuation / control / whitespace code points."""
    import random
    rnd = random.Random(seed)
    pools = ["abcdefghijklmnopqrstuvwxyz", "ABCDEFGHIJKLMNOPQRSTUVWXYZ", "0123456789", " \t\n\r\u00a0\u2003", ".,;:!?'\"()[]{}-_/\\@#$%^&*+=<>|~`",
             "\u00e9\u00e8\u00fc\u00f1\u00e7\u00df\u00f8\u0142\u0159\u015f", "\u4e2d\u6587\u6f22\u5b57\u6771\u4eac", "\u3042\u3044\u30a2\u30a4", "\uac00\ub098",
             "\u0430\u0431\u0432\u0433\u0414\u0416", "\u03b1\u03b2\u03b3\u0394", "\u0627\u0644\u0639", "\u0000\u0007\ufffd\u200b\u200d\u00ad", "\u2014\u2013\u2018\u2019\u201c\u201d\u2026\u20ac",
             "\u0301\u0308\u0327", "\U0001f600\U0001f680"]
    out = []
    for _ in range(n):
        k = rnd.randint(1, 40)
        out.append("".join(rnd.choice(rnd.choice(pools)) for _ in range(k)))
    return out


TEXTS = TEXTS + _fuzz_texts()
SQUAD = {"version": "1.1", "data": [{"title": "t", "paragraphs": [
    {"context": "The capital of France is Paris. The river Seine flows through Paris and it is a river.",
     "qas": [{"id": "q1", "question": "What is the capital of France?", "answers": [{"text": "Paris", "answer_start": 25}]},
             {"id": "q2", "question": "What river flows through Paris?", "answers": [{"text": "Seine", "answer_start": 42}]}]},
    {"context": "Hamlet is a play. The play was written by William Shakespeare in 1603.",
     "qas": [{"id": "q3", "question": "Who wrote Hamlet?", "answers": [{"text": "William Shakespeare", "answer_start": 42}]}]}]}]}

NER_LABELS = ["O", "B-PER", "I-PER", "B-LOC"]
NER_TEXT = ("-DOCSTART- -X- -X- O\n\nWilliam NNP B-NP B-PER\nShakespeare NNP I-NP I-PER\nwrote VBD B-VP O\nHamlet NNP B-NP O\n"
            "in IN B-PP O\nParis NNP B-NP B-LOC\n.\t.\tO\tO\n\nThe DT B-NP O\nriver NN I-NP O\nSeine NNP I-NP B-LOC\nflows VBZ B-VP O\n"
            "through IN B-PP O\nParis NNP B-NP B-LOC\nand CC O O\nit PRP B-NP O\nis VBZ B-VP O\na DT B-NP O\nriver NN I-NP O\n. . O O\n")



def _random_squad(n_par=12, seed=17):
    """Long random paragraphs over the toy vocabulary (several sliding windows each) with exact answer offsets."""
    import random
    rnd = random.Random(seed)
    words = [w for w in VOCAB if w.isalpha()] + ["Paris,", "(1603)", "river-bank", "Seine's", "unaffable."]
    pars = []
    for p_i in range(n_par):
        ctx_words = [rnd.choice(words) for _ in range(rnd.randint(30, 90))]
        ctx = " ".join(ctx_words)
        qas = []
        for q_i in range(rnd.randint(1, 3)):
            i = rnd.randrange(len(ctx_words)); j = min(len(ctx_words) - 1, i + rnd.randint(0, 3))
            start = len(" ".join(ctx_words[:i])) + (1 if i else 0)
            text = " ".join(ctx_words[i:j + 1])
            assert ctx[start:start + len(text)] == text
            qas.append({"id": f"r{p_i}_{q_i}", "question": " ".join(rnd.choice(words) for _ in range(rnd.randint(3, 15))) + "?",
                        "answers": [{"text": text, "answer_start": start}]})
        pars.append({"context": ctx, "qas": qas})
    return pars


SQUAD["data"][0]["paragraphs"] += _random_squad()

REF_SCRIPT = r'''
import collections, json, os, pickle, sys, types
import numpy as np, torch
sys.path.insert(0, ".")
work, = sys.argv[1:]
spec = pickle.load(open(work + "/spec.pkl", "rb"))
out = {}
import src.modeling as M, src.tokenization as T, src.schedulers as S, src.optimization as O, src.dataset as D
import run_squad as RS

# ---- models
torch.manual_seed(0)
cfg = M.BertConfig.from_dict(spec["cfg"])
ids, seg, mask = (torch.tensor(a) for a in spec["inputs"])
models = {}
for name, ctor in (("pretraining", lambda: M.BertForPreTraining(cfg)), ("qa", lambda: M.BertForQuestionAnswering(cfg)),
                   ("token", lambda: M.BertForTokenClassification(cfg, 5)), ("seq", lambda: M.BertForSequenceClassification(cfg, 3)),
                   ("mlm", lambda: M.BertForMaskedLM(cfg))):
    m = ctor().eval()
    det_fill(m.state_dict(), 0)
    with torch.no_grad():
        y = m(ids, seg, mask)
    y = [t.numpy() for t in (y if isinstance(y, (tuple, list)) else [y])]
    models[name] = ({k: v.numpy() for k, v in m.state_dict().items()}, y)
out["models"] = models

# ---- tokenizers
vocab = T.load_vocab(work + "/vocab.txt")
basic = T.BasicTokenizer(do_lower_case=True)
wp = T.WordpieceTokenizer(vocab=vocab)
out["basic"] = [basic.tokenize(t) for t in spec["texts"]]
out["wordpiece"] = [[p for w in basic.tokenize(t) for p in wp.tokenize(w)] for t in spec["texts"]]
out["basic_cased"] = [T.BasicTokenizer(do_lower_case=False).tokenize(t) for t in spec["texts"]]
bt = T.BertTokenizer(work + "/vocab.txt", do_lower_case=True)
out["bert_tokenizer"] = [(bt.tokenize(t), bt.convert_tokens_to_ids(bt.tokenize(t))) for t in spec["texts"][:40]]
out["ids_to_tokens"] = bt.convert_ids_to_tokens([0, 5, 10, 28, 3])

# ---- SQuAD featurisation + post-processing
tok = T.get_wordpiece_tokenizer(work + "/vocab.txt", uppercase=False)
ex = RS.read_squad_examples(work + "/squad.json", True, False)
feats = RS.convert_examples_to_features(ex, tok, 48, 16, 12, True)
out["features"] = [dict(unique_id=f.unique_id, example_index=f.example_index, doc_span_index=f.doc_span_index,
                        tokens=list(f.tokens), token_to_orig_map=dict(f.token_to_orig_map),
                        token_is_max_context=dict(f.token_is_max_context), input_ids=list(f.input_ids),
                        input_mask=list(f.input_mask), segment_ids=list(f.segment_ids),
                        start_position=f.start_position, end_position=f.end_position) for f in feats]
ex_eval = RS.read_squad_examples(work + "/squad.json", False, False)
feats_eval = RS.convert_examples_to_features(ex_eval, tok, 48, 16, 12, False)
rng = np.random.default_rng(0)
results = []
logits = {}
for f in feats_eval:
    s, e = rng.normal(size=48).tolist(), rng.normal(size=48).tolist()
    logits[f.unique_id] = (s, e)
    results.append(RS.RawResult(f.unique_id, s, e))
args = types.SimpleNamespace(version_2_with_negative=False, n_best_size=5, max_answer_length=10, do_lower_case=True,
                             null_score_diff_threshold=0.0, verbose_logging=False)
answers, nbest = RS.get_answers(ex_eval, feats_eval, results, args)
out["logits"] = logits
out["answers"] = dict(answers)
out["nbest"] = {k: [dict(d) for d in v] for k, v in nbest.items()}

# ---- schedulers coupled to the optimizer's step counter (src/schedulers.py:97-105,126-134)
def lr_curve(cls, **kw):
    p = torch.nn.Parameter(torch.zeros(1))
    opt = torch.optim.SGD([p], lr=1.0)
    sch = cls(opt, **kw)
    lrs = []
    for step in range(1, 41):
        opt.param_groups[0]["step"] = step
        sch.step()
        lrs.append(opt.param_groups[0]["lr"])
    return lrs
out["poly"] = lr_curve(S.PolyWarmUpScheduler, warmup=0.25, total_steps=40)
out["linear"] = lr_curve(S.LinearWarmUpScheduler, warmup=0.25, total_steps=40)

# ---- BertAdam (src/optimization.py:64-174)
torch.manual_seed(3)
w = torch.nn.Parameter(torch.randn(7, 5))
opt = O.BertAdam([w], lr=1e-2, warmup=0.1, t_total=20, weight_decay=0.01, max_grad_norm=1.0)
traj = []
for i in range(6):
    w.grad = torch.randn(7, 5, generator=torch.Generator().manual_seed(10 + i)) * (3.0 if i == 2 else 1.0)
    opt.step()
    traj.append(w.detach().clone().numpy())
out["bertadam"] = traj

# ---- sampler chunking (src/dataset.py:341-428)
class _DS(torch.utils.data.Dataset):
    def __len__(self): return 23
    def __getitem__(self, i): return i
    def set_epoch(self, epoch): pass
chunks = {}
for world in (1, 2, 4):
    for rank in range(world):
        sm = D.DistributedSampler(_DS(), num_replicas=world, rank=rank)
        sm.set_epoch(1)
        chunks[(world, rank)] = list(iter(sm))
out["sampler"] = chunks
sm = D.DistributedSampler(_DS(), num_replicas=2, rank=1)
sm.set_epoch(3)
it = iter(sm); first = [next(it) for _ in range(4)]
out["sampler_state"] = (first, sm.state_dict())

# ---- more task models
extra = {}
ids4 = torch.stack([ids, ids.flip(1)], dim=1)            # [B, 2 choices, S]
seg4, mask4 = torch.stack([seg, seg], dim=1), torch.stack([mask, mask], dim=1)
for name, ctor, inp in (("nsp", lambda: M.BertForNextSentencePrediction(cfg), (ids, seg, mask)),
                        ("choice", lambda: M.BertForMultipleChoice(cfg, 2), (ids4, seg4, mask4)),
                        ("encoder", lambda: M.BertModel(cfg), (ids, seg, mask))):
    torch.manual_seed(5)
    m = ctor().eval()
    det_fill(m.state_dict(), 0)
    with torch.no_grad():
        y = m(*inp)
    flat = []
    for t in (y if isinstance(y, (tuple, list)) else [y]):
        flat += [u.numpy() for u in (t if isinstance(t, (tuple, list)) else [t]) if torch.is_tensor(u)]
    extra[name] = ({k: v.numpy() for k, v in m.state_dict().items()}, flat, type(y[0]).__name__ if isinstance(y, tuple) else "")
out["models2"] = extra

# ---- pre-training criterion (run_pretraining.py:58-72) incl. ignored labels and the no-NSP form
import run_pretraining as RP
g = torch.Generator().manual_seed(11)
scores = torch.randn(3, 24, cfg.vocab_size, generator=g)
labels = torch.full((3, 24), -1, dtype=torch.long); labels[:, 3] = 7; labels[1, 9] = 50
nsp_s, nsp_l = torch.randn(3, 2, generator=g), torch.tensor([0, 1, 1])
crit = RP.BertPretrainingCriterion(cfg.vocab_size)
out["criterion"] = (scores.numpy(), labels.numpy(), nsp_s.numpy(), nsp_l.numpy(),
                    float(crit(scores, labels, nsp_s, nsp_l)), float(crit(scores, labels)))

# ---- dataset helpers (src/dataset.py:224-275): deterministic parts
ds = D.ShardedPretrainingDataset.__new__(D.ShardedPretrainingDataset)
row = np.zeros(16, dtype=np.int64); row[:11] = np.arange(20, 31)
out["segments"] = [(ds._get_segment_ids(row, np.array(sp)).tolist(), ds._get_input_mask(row, np.array(sp)).tolist())
                   for sp in ([0, 10], [0, 4, 10], [0, 1, 2])]
pos = np.array([2, 5, 9, 0, 0]); lab = np.array([21, 22, 23, 0, 0])
out["premasked"] = ds._get_masked_labels(row, pos, lab).tolist()

# ---- NER: CoNLL parsing, word-piece label replication, truncation, macro-F1
from src.ner_dataset import NERDataset
import run_ner as RN
nds = NERDataset(work + "/ner.txt", tok, spec["ner_labels"], 12)
out["ner"] = [[t.tolist() for t in nds[i]] for i in range(len(nds))]
rngm = np.random.default_rng(4)
preds = rngm.normal(size=(3, 12, len(spec["ner_labels"]) + 1))
lbl = rngm.integers(-1, len(spec["ner_labels"]) + 1, size=(3, 12)); lbl[lbl < 0] = -100
idx_to_label = {i: l for i, l in enumerate(spec["ner_labels"], start=1)}
idx_to_label[0] = "O"
out["ner_f1"] = (preds, lbl, float(RN.compute_metrics(preds, lbl, idx_to_label)))

# ---- small helpers
import src.utils as U, src.file_utils as F
out["format_step"] = [U.format_step(x) for x in ("PARAMETER", (1,), (1, 20), (2, 30, 4), ())]
out["url_to_filename"] = [F.url_to_filename("https://example.org/a/b.bin"), F.url_to_filename("s3://bucket/key", etag='"abc"')]

# ---- CLI: defaults, JSON overlay and CLI precedence of run_pretraining.py / run_ner.py
import sys as _sys
def parse(mod, argv):
    old = _sys.argv
    _sys.argv = ["prog"] + argv
    try:
        return {k: v for k, v in vars(mod.parse_arguments()).items()}
    finally:
        _sys.argv = old
out["cli_pretrain"] = [parse(RP, a) for a in spec["pretrain_argvs"]]
out["cli_ner"] = parse(RN, spec["ner_argv"])

# ---- fresh initialisation under a fixed seed (structure + init rules), config JSON round trip
torch.manual_seed(123)
fresh = M.BertForPreTraining(cfg)
out["fresh"] = {k: (tuple(v.shape), float(v.float().mean()), float(v.float().std()) if v.numel() > 1 else 0.0)
                for k, v in fresh.state_dict().items()}
out["fresh_exact"] = {k: v.numpy() for k, v in fresh.state_dict().items()}
out["config_json"] = json.loads(cfg.to_json_string())

# ---- encoder sample layout (utils/encode_data.py:12-35)
try:
    import importlib.util
    sp_ = importlib.util.spec_from_file_location("ref_encode_data", spec["ref_utils"] + "/encode_data.py")
    E = importlib.util.module_from_spec(sp_); sp_.loader.exec_module(E)
    ts = [E.TrainingSample(["a", "b", "c"]), E.TrainingSample(["a", "b"], ["c", "d", "e"], True), E.TrainingSample([], [])]
    out["samples"] = [(t.sequence, t.special_token_positions, t.is_random_next) for t in ts]
except Exception as e:
    out["samples"] = repr(e)

# ---- SQuAD v2 (impossible questions, null scores) and the small post-processing helpers
ex2 = RS.read_squad_examples(work + "/squad2.json", True, True)
out["v2_examples"] = [(e.qas_id, e.is_impossible, e.start_position, e.end_position, e.orig_answer_text) for e in ex2]
f2 = RS.convert_examples_to_features(ex2, tok, 48, 16, 12, True)
out["v2_features"] = [(f.unique_id, f.start_position, f.end_position, f.is_impossible) for f in f2]
ex2e = RS.read_squad_examples(work + "/squad2.json", False, True)
f2e = RS.convert_examples_to_features(ex2e, tok, 48, 16, 12, False)
rng2 = np.random.default_rng(7)
lg2, res2 = {}, []
for f in f2e:
    a, b = rng2.normal(size=48).tolist(), rng2.normal(size=48).tolist()
    lg2[f.unique_id] = (a, b); res2.append(RS.RawResult(f.unique_id, a, b))
args2 = types.SimpleNamespace(version_2_with_negative=True, n_best_size=4, max_answer_length=8, do_lower_case=True,
                              null_score_diff_threshold=-1.0, verbose_logging=False)
ans2, nb2 = RS.get_answers(ex2e, f2e, res2, args2)
out["v2_logits"], out["v2_answers"], out["v2_nbest"] = lg2, dict(ans2), {k: [dict(d) for d in v] for k, v in nb2.items()}
out["final_text"] = [RS.get_final_text(a, b, True, False) for a, b in spec["final_text_pairs"]]
out["best_indices"] = RS._get_best_indices([0.1, 3.0, -1.0, 3.0, 2.5, 0.0], 3)
out["softmax"] = RS._compute_softmax([1.0, 2.0, -3.0, 0.5])

# ---- the sharded dataset over real shard files (deterministic outputs only; masking is random)
np.random.seed(0)
dsr = D.ShardedPretrainingDataset(sorted(spec["shards"]), 4, 5, 0.2, vocab_size=100)
rows = []
for i in range(len(dsr)):
    ids_, seg_, msk_, lab_, nsl_ = dsr[i]
    ids_, lab_ = np.asarray(ids_), np.asarray(lab_)
    rows.append((np.asarray(seg_).tolist(), np.asarray(msk_).tolist(), int(np.asarray(nsl_)),
                 int((lab_ >= 0).sum()), ids_.shape[0]))
out["dataset_rows"] = rows
out["dataset_len"] = len(dsr)

# ---- a few optimisation steps end to end (model backward through autograd + criterion + BertAdam), dropout off
cfg0 = M.BertConfig.from_dict(dict(spec["cfg"], hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0))
torch.manual_seed(77)
net = M.BertForPreTraining(cfg0).train()
det_fill(net.state_dict(), 77)
out["train_init"] = {k: v.numpy().copy() for k, v in net.state_dict().items()}
opt2 = O.BertAdam([p for p in net.parameters()], lr=5e-3, warmup=0.2, t_total=10, weight_decay=0.01, max_grad_norm=1.0)
crit2 = RP.BertPretrainingCriterion(cfg0.vocab_size)
lab2 = torch.full_like(ids, -1); lab2[:, 2] = 9; lab2[:, 7] = 30; lab2[0, 11] = 5
nsl2 = torch.tensor([1, 0, 1])
losses = []
for step in range(4):
    sc, rel = net(torch.roll(ids, step, 1), seg, mask)
    loss = crit2(sc, lab2, rel, nsl2)
    loss.backward()
    opt2.step(); opt2.zero_grad()
    losses.append(float(loss))
out["train_losses"] = losses
out["train_final"] = {k: v.numpy().copy() for k, v in net.state_dict().items()}

# ---- dynamic masking statistics (src/dataset.py:277-296)
dm = D.ShardedPretrainingDataset.__new__(D.ShardedPretrainingDataset)
dm.max_pred_per_seq, dm.masked_lm_prob, dm.original_token_prob, dm.random_token_prob = 20, 0.2, 0.1, 0.1
dm.vocab_size, dm.mask_token_index = 1000, 4
np.random.seed(123)
base = np.zeros(64, dtype=np.int64); base[:50] = np.arange(100, 150); spx = np.array([0, 20, 49])
n_lab = n_mask = n_keep = n_rand = bad = 0
for _ in range(3000):
    ids_m, lab_m = dm._mask_input(base.copy(), spx)
    sel = lab_m >= 0
    n_lab += int(sel.sum()); bad += int(sel[[0, 20, 49]].sum()) + int(sel[50:].sum())
    n_mask += int((ids_m[sel] == 4).sum()); n_keep += int((ids_m[sel] == base[sel]).sum())
    n_rand += int(((ids_m[sel] != 4) & (ids_m[sel] != base[sel])).sum())
out["mask_stats"] = (n_lab / 3000.0, n_mask / n_lab, n_keep / n_lab, n_rand / n_lab, bad)

# ---- task models called WITH labels return their loss (src/modeling.py:998-1271)
lab_tok = torch.randint(0, 5, ids.shape, generator=torch.Generator().manual_seed(2))
mlm_lab = torch.full_like(ids, -1); mlm_lab[:, 4] = 17; mlm_lab[2, 1] = 8
with_labels = {}
for name, ctor, kwargs in (("mlm", lambda: M.BertForMaskedLM(cfg), dict(masked_lm_labels=mlm_lab)),
                           ("nsp", lambda: M.BertForNextSentencePrediction(cfg), dict(next_sentence_label=torch.tensor([0, 1, 0]))),
                           ("token", lambda: M.BertForTokenClassification(cfg, 5), dict(labels=lab_tok)),
                           ("choice", lambda: M.BertForMultipleChoice(cfg, 2), dict(labels=torch.tensor([1, 0, 1])))):
    torch.manual_seed(9)
    m = ctor().eval()
    det_fill(m.state_dict(), 0)
    inp = (ids4, seg4, mask4) if name == "choice" else (ids, seg, mask)
    with torch.no_grad():
        y = m(*inp, **kwargs)
    with_labels[name] = ({k: v.numpy() for k, v in m.state_dict().items()}, float(y if torch.is_tensor(y) else y[0]))
out["with_labels"] = with_labels

# ---- from_pretrained: directory with bert_config.json + pytorch_model.bin in the OLD naming (gamma / beta), loaded
#      (a) into the full pre-training model, (b) into a bare encoder (bert. prefix stripped), (c) a task model with extra args
import os as _os
pt_dir = work + "/pretrained"
_os.makedirs(pt_dir, exist_ok=True)
torch.manual_seed(21)
src_model = M.BertForPreTraining(cfg)
det_fill(src_model.state_dict(), 0)
old_sd = collections.OrderedDict((k.replace("LayerNorm.weight", "LayerNorm.gamma").replace("LayerNorm.bias", "LayerNorm.beta"), v)
                                 for k, v in src_model.state_dict().items())
torch.save(old_sd, pt_dir + "/pytorch_model.bin")
open(pt_dir + "/bert_config.json", "w").write(cfg.to_json_string())
fp = {}
for name, loader in (("pretraining", lambda: M.BertForPreTraining.from_pretrained(pt_dir)),
                     ("encoder", lambda: M.BertModel.from_pretrained(pt_dir)),
                     ("token", lambda: M.BertForTokenClassification.from_pretrained(pt_dir, num_labels=5))):
    torch.manual_seed(33)                           # the heads that are not in the archive are freshly initialised
    m = loader().eval()
    with torch.no_grad():
        y = m(ids, seg, mask)
    flat = []
    for t in (y if isinstance(y, (tuple, list)) else [y]):
        flat += [u.numpy() for u in (t if isinstance(t, (tuple, list)) else [t]) if torch.is_tensor(u)]
    fp[name] = flat
out["from_pretrained"] = fp

# ---- the runtime's micro-step (run_pretraining.py:420-460) with accumulation: loss / divisor, gradients add up
torch.manual_seed(77)
net3 = M.BertForPreTraining(cfg0).train()
net3.load_state_dict({k: torch.from_numpy(v) for k, v in out["train_init"].items()})
crit3 = RP.BertPretrainingCriterion(cfg0.vocab_size)
micro_losses = []
for mstep in range(3):
    batch = (torch.roll(ids, mstep, 1), seg, mask, lab2, nsl2)
    micro_losses.append(float(RP.forward_backward_pass(net3, crit3, None, batch, 3, sync_grads=True)))
out["micro_losses"] = micro_losses
out["micro_grads"] = {k: p.grad.numpy().copy() for k, p in net3.named_parameters() if p.grad is not None}

# ---- optimizer set-up and the resume surgery of run_pretraining.prepare_optimizers (phase 1 -> phase 2)
import copy as _copy
net4 = M.BertForPreTraining(cfg0)
a1 = types.SimpleNamespace(lr_decay="poly", learning_rate=6e-3, warmup_proportion=0.25, max_steps=8, fp16=False, kfac=False,
                           resume_step=0, previous_phase_end_step=0)
opt4, _, sch4, _ = RP.prepare_optimizers(a1, net4, None, 0)
names = dict((id(p), n) for n, p in net4.named_parameters())
out["opt_groups"] = [(g["weight_decay"], sorted(names[id(p)] for p in g["params"])) for g in opt4.param_groups]
for _ in range(4):
    for p_ in net4.parameters(): p_.grad = torch.ones_like(p_) * 0.01
    sch4[0].step(); opt4.step()
ck4 = {"optimizer": _copy.deepcopy(opt4.state_dict())}
a2 = types.SimpleNamespace(lr_decay="poly", learning_rate=4e-3, warmup_proportion=0.5, max_steps=10, fp16=False, kfac=False,
                           resume_step=4, previous_phase_end_step=4)
opt5, _, sch5, _ = RP.prepare_optimizers(a2, net4, ck4, 0)
out["resumed_group"] = {k: v for k, v in opt5.param_groups[0].items() if k != "params"}
out["resumed_base_lrs"] = list(sch5[0].base_lrs)
out["resumed_state_steps"] = sorted({int(st["step"]) for st in opt5.state_dict()["state"].values()})

# ---- legacy pre-masked shards (NVIDIA format, src/dataset.py:183-192): no randomness -> every field is comparable;
#      plus a missing and a corrupt file in the list (skipped with a warning)
import warnings as _w
with _w.catch_warnings():
    _w.simplefilter("ignore")
    dleg = D.ShardedPretrainingDataset(sorted(spec["legacy_shards"]) + [work + "/does_not_exist.hdf5", work + "/vocab.txt"],
                                       4, 5, 0.2, vocab_size=100)
out["legacy_len"] = len(dleg)
out["legacy_rows"] = [[np.asarray(a).tolist() for a in dleg[i]] for i in range(len(dleg))]

# ---- run_ner.get_data: vocabulary / tokenizer resolved from the model config, loaders over the CoNLL files
json.dump(dict(spec["cfg"], vocab_file=work + "/vocab.txt", tokenizer="wordpiece"), open(work + "/ner_model.json", "w"))
nargs = types.SimpleNamespace(cuda=False, batch_size=2, vocab_file=None, tokenizer=None, model_config_file=work + "/ner_model.json",
                              uppercase=False, train_file=work + "/ner.txt", val_file=work + "/ner.txt", test_file=None,
                              labels=spec["ner_labels"], max_seq_len=12)
tl, vl, tel = RN.get_data(nargs)
out["ner_get_data"] = (len(tl), len(vl), tel is None, nargs.vocab_file, nargs.tokenizer,
                       [[t.tolist() for t in b] for b in vl])

# ---- run_pretraining.prepare_dataset: recursive shard discovery, tokenizer from the model config, sampler resume
json.dump(dict(spec["cfg"], vocab_size=100, vocab_file=work + "/vocab.txt", tokenizer="wordpiece", lowercase=True),
          open(work + "/pt_model.json", "w"))
pargs = types.SimpleNamespace(input_dir=os.path.dirname(spec["shards"][0]), model_config_file=work + "/pt_model.json",
                              max_predictions_per_seq=5, masked_token_fraction=0.2, local_batch_size=4, seed=42)
ld, sm_ = RP.prepare_dataset(pargs, {"sampler": {"epoch": 0, "seed": 0, "num_replicas": 1, "total_size": 21, "index": 9}})
out["prepare_dataset"] = (len(ld.dataset), len(sm_), sm_.index, len(ld), ld.dataset.mask_token_index)

# ---- activation table and the Linear+activation module (src/modeling.py:118-185)
xa = torch.randn(5, 7, generator=torch.Generator().manual_seed(1)) * 3
ba = torch.randn(7, generator=torch.Generator().manual_seed(2))
acts = {}
for name, fn in M.ACT2FN.items():
    try:
        acts[name] = (fn(ba, xa) if name.startswith("bias_") else fn(xa)).numpy()
    except Exception as e:
        acts[name] = repr(e)
out["acts"] = (xa.numpy(), ba.numpy(), acts)
torch.manual_seed(4)
la = M.LinearActivation(7, 6, act="gelu")
lt = M.LinearActivation(7, 6, act="tanh")
out["linear_act"] = ({k: v.numpy() for k, v in la.state_dict().items()}, la(xa).detach().numpy(),
                     {k: v.numpy() for k, v in lt.state_dict().items()}, lt(xa).detach().numpy())
pickle.dump(out, open(work + "/ref.pkl", "wb"))
'''


def _write_inputs(work, ref_utils=""):
    """Every input file both sides read, written under ``work`` (a pathlib.Path); returns the spec of the run."""
    rng = np.random.default_rng(1)
    ids = rng.integers(5, MODEL_CFG["vocab_size"], size=(3, 24))
    seg = np.zeros_like(ids); seg[:, 12:] = 1
    mask = np.ones_like(ids); mask[1, 18:] = 0; mask[2, 9:] = 0
    (work / "train.json").write_text(json.dumps({"learning_rate": 1e-3, "max_steps": 77, "kfac_damping": 0.5, "lr_decay": "linear",
                                                  "unknown_key": 1, "global_batch_size": 1024}))
    argvs = [[], ["--config_file", str(work / "train.json")],
             # (no store_true flag here: the reference's auxiliary parser registers every option as taking a value, so
             #  `--fp16` on its command line is an argparse error -- booleans can only come from the JSON file there)
             ["--config_file", str(work / "train.json"), "--learning_rate", "0.5", "--steps", "12", "--input_dir", "/x"]]
    v2 = {"version": "v2.0", "data": [{"title": "t", "paragraphs": [
        {"context": "Hamlet is a play. The play was written by William Shakespeare in 1603.",
         "qas": [{"id": "i1", "question": "Who wrote the river?", "is_impossible": True, "answers": []},
                 {"id": "a1", "question": "Who wrote Hamlet?", "is_impossible": False,
                  "answers": [{"text": "William Shakespeare", "answer_start": 42}]}]}]}]}
    (work / "squad2.json").write_text(json.dumps(v2))
    from bert_pytorch_b200.data import synthetic
    shards = synthetic.write_shards(str(work / "shards"), 3, 7, 16, 100, True, seed=3)
    import random as _r
    rr = _r.Random(3)
    fuzz_pairs = []
    for t in _fuzz_texts(120, seed=29):
        words = t.split()
        if not words:
            continue
        i = rr.randrange(len(words)); j = rr.randrange(i, min(len(words), i + 3))
        fuzz_pairs.append((" ".join(w.lower().strip(".,!?") for w in words[i:j + 1]), " ".join(words[max(0, i - 1):j + 2])))
    from bert_pytorch_b200.data import hdf5 as _h5
    legacy = []
    lr_ = np.random.default_rng(21)
    for k in range(2):
        n = 5 + k
        lids = lr_.integers(5, 100, size=(n, 16)).astype(np.int32)
        lens = lr_.integers(6, 16, size=n)
        lmask = (np.arange(16)[None, :] < lens[:, None]).astype(np.int32)
        lids *= lmask
        lseg = ((np.arange(16)[None, :] >= (lens // 2)[:, None]) & (lmask == 1)).astype(np.int32)
        lpos = np.zeros((n, 4), dtype=np.int32); lmid = np.zeros((n, 4), dtype=np.int32)
        for r_ in range(n):
            cnt = int(lr_.integers(1, 4))
            lpos[r_, :cnt] = np.sort(lr_.choice(np.arange(1, lens[r_]), size=cnt, replace=False))
            lmid[r_, :cnt] = lr_.integers(5, 100, size=cnt)
        path = str(work / f"legacy_{k}.hdf5")
        with _h5.File(path, "w") as f:
            for name, arr in (("input_ids", lids), ("segment_ids", lseg), ("input_mask", lmask), ("masked_lm_positions", lpos),
                              ("masked_lm_ids", lmid), ("next_sentence_labels", lr_.integers(0, 2, size=n).astype(np.int8))):
                f.create_dataset(name, data=arr, dtype=arr.dtype.str[1:], compression="gzip")
        legacy.append(path)
    pairs = fuzz_pairs + [("paris", "Paris."), ("william shakespeare", "William   Shakespeare's"), ("1603", "(1603)."), ("seine", "the Seine,"),
             ("x y", "completely different")]
    spec = dict(shards=shards, legacy_shards=legacy, final_text_pairs=pairs, cfg=MODEL_CFG, inputs=[ids.tolist(), seg.tolist(), mask.tolist()], texts=TEXTS, ner_labels=NER_LABELS,
                pretrain_argvs=argvs, ner_argv=["--train_file", "t.txt", "--labels", "O", "B-X", "--model_config_file", "m.json", "--model_checkpoint", "c.pt"],
                ref_utils=ref_utils)
    (work / "ner.txt").write_text(NER_TEXT)
    pickle.dump(spec, open(work / "spec.pkl", "wb"))
    (work / "vocab.txt").write_text("\n".join(VOCAB) + "\n")
    (work / "squad.json").write_text(json.dumps(SQUAD))
    return spec


def _swap(obj, a, b):
    """``obj`` with the substring a of every string (dict keys included) replaced by b."""
    if isinstance(obj, str):
        return obj.replace(a, b)
    if isinstance(obj, dict):
        return {_swap(k, a, b): _swap(v, a, b) for k, v in obj.items()}
    if isinstance(obj, (list, tuple)):
        return type(obj)(_swap(v, a, b) for v in obj)
    return obj


def _squad_logits(order, seed):
    """The random start / end logits the original run drew for its features, in its feature order."""
    rng = np.random.default_rng(seed)
    return {uid: (rng.normal(size=48).tolist(), rng.normal(size=48).tolist()) for uid in order}


def _criterion_inputs():
    g = torch.Generator().manual_seed(11)
    scores = torch.randn(3, 24, MODEL_CFG["vocab_size"], generator=g)
    labels = torch.full((3, 24), -1, dtype=torch.long); labels[:, 3] = 7; labels[1, 9] = 50
    nsp_s, nsp_l = torch.randn(3, 2, generator=g), torch.tensor([0, 1, 1])
    return scores.numpy(), labels.numpy(), nsp_s.numpy(), nsp_l.numpy()


def _ner_f1_inputs():
    rngm = np.random.default_rng(4)
    preds = rngm.normal(size=(3, 12, len(NER_LABELS) + 1))
    lbl = rngm.integers(-1, len(NER_LABELS) + 1, size=(3, 12)); lbl[lbl < 0] = -100
    return preds, lbl


def _layout(sd, seed):
    """A state dict filled by ``det_fill(.., seed)`` -> its keys, shapes and ties (alias -> first name of the storage)."""
    keys, ties, vals = [(k, tuple(v.shape)) for k, v in sd.items()], {}, {}
    for k, shape in keys:
        want = draw(k, shape, seed)
        if not np.array_equal(sd[k], want):
            ties[k] = next(j for j in vals if j not in ties and np.array_equal(sd[k], vals[j]))
        vals[k] = want
    return keys, ties, seed


def _state(layout):
    keys, ties, seed = layout
    sd = {k: draw(k, shape, seed) for k, shape in keys}
    return {k: sd[ties.get(k, k)] for k, _ in keys}


def _compact(out, work):
    """The original run's results -> what the golden file keeps (see the module docstring)."""
    out = _swap(out, work, WORK)
    out["models"] = {n: (_layout(sd, FILL_SEED), y) for n, (sd, y) in out["models"].items()}
    out["models2"] = {n: (_layout(sd, FILL_SEED), y, t) for n, (sd, y, t) in out["models2"].items()}
    out["with_labels"] = {n: (_layout(sd, FILL_SEED), loss) for n, (sd, loss) in out["with_labels"].items()}
    out["train_init"] = _layout(out["train_init"], TRAIN_SEED)
    out["train_final"] = {k: _sample(v) for k, v in out["train_final"].items()}
    out["micro_grads"] = {k: (_sample(v), float(np.abs(v).max())) for k, v in out["micro_grads"].items()}
    out["fresh_exact"] = {k: _digest(v) for k, v in out["fresh_exact"].items()}
    for key, seed in (("logits", 0), ("v2_logits", 7)):
        assert out[key] == _squad_logits(list(out[key]), seed), key
        out[key] = list(out[key])
    for a, b in zip(out["criterion"][:4], _criterion_inputs()):
        assert np.array_equal(a, b)
    out["criterion"] = out["criterion"][4:]
    for a, b in zip(out["ner_f1"][:2], _ner_f1_inputs()):
        assert np.array_equal(a, b)
    out["ner_f1"] = out["ner_f1"][2]
    seen = {}                                  # identical outputs (same weights, same inputs) are stored once

    def dedup(o):
        if isinstance(o, np.ndarray):
            return seen.setdefault((o.dtype.str, o.shape, o.tobytes()), o)
        if isinstance(o, dict):
            return {k: dedup(v) for k, v in o.items()}
        if isinstance(o, (list, tuple)):
            return type(o)(dedup(v) for v in o)
        return o
    return dedup(out)


def _expand(golden, work):
    """Inverse of ``_compact`` for the scratch directory ``work``: the results in the form the tests read."""
    out = _swap(golden, WORK, work)
    out["models"] = {n: (_state(lay), y) for n, (lay, y) in out["models"].items()}
    out["models2"] = {n: (_state(lay), y, t) for n, (lay, y, t) in out["models2"].items()}
    out["with_labels"] = {n: (_state(lay), loss) for n, (lay, loss) in out["with_labels"].items()}
    out["train_init"] = _state(out["train_init"])
    out["logits"], out["v2_logits"] = _squad_logits(out["logits"], 0), _squad_logits(out["v2_logits"], 7)
    out["criterion"] = _criterion_inputs() + tuple(out["criterion"])
    out["ner_f1"] = _ner_f1_inputs() + (out["ner_f1"],)
    return out


@pytest.fixture(scope="module")
def golden():
    with gzip.open(GOLDEN, "rb") as f:
        return pickle.load(f)


@pytest.fixture(scope="module")
def ref(tmp_path_factory, golden):
    work = tmp_path_factory.mktemp("refparity")
    spec = _write_inputs(work)
    out = _expand(golden["script"], str(work))
    out["work"], out["spec"] = str(work), spec
    # the files the original-side script wrote for the tests below: the from_pretrained archive in the old gamma / beta
    # naming (the same det_fill weights as the pre-training model of the zoo) and two model configs
    (work / "pretrained").mkdir()
    old = {k.replace("LayerNorm.weight", "LayerNorm.gamma").replace("LayerNorm.bias", "LayerNorm.beta"): torch.from_numpy(v)
           for k, v in out["models"]["pretraining"][0].items()}
    torch.save(old, work / "pretrained" / "pytorch_model.bin")
    (work / "pretrained" / "bert_config.json").write_text(json.dumps(out["config_json"], indent=2, sort_keys=True) + "\n")
    vocab = str(work / "vocab.txt")
    json.dump(dict(MODEL_CFG, vocab_file=vocab, tokenizer="wordpiece"), open(work / "ner_model.json", "w"))
    json.dump(dict(MODEL_CFG, vocab_size=100, vocab_file=vocab, tokenizer="wordpiece", lowercase=True),
              open(work / "pt_model.json", "w"))
    return out


def test_reference_state_dicts_load_and_logits_agree(ref):
    from bert_pytorch_b200 import BertConfig, models as M
    cfg = BertConfig.from_dict(MODEL_CFG)
    ids, seg, mask = (torch.tensor(a) for a in ref["spec"]["inputs"])
    ctors = {"pretraining": lambda: M.BertForPreTraining(cfg), "qa": lambda: M.BertForQuestionAnswering(cfg),
             "token": lambda: M.BertForTokenClassification(cfg, 5), "seq": lambda: M.BertForSequenceClassification(cfg, 3),
             "mlm": lambda: M.BertForMaskedLM(cfg)}
    for name, (sd, outs) in ref["models"].items():
        m = ctors[name]().eval()
        ours = set(m.state_dict())
        assert ours == set(sd), (name, sorted(ours ^ set(sd))[:6])          # the checkpoint contract, both directions
        m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()}, strict=True)
        with torch.no_grad():
            y = m(ids, seg, mask)
        y = list(y) if isinstance(y, (tuple, list)) else [y]
        assert len(y) == len(outs), name
        for a, b in zip(y, outs):
            assert a.shape == b.shape and np.allclose(a.numpy(), b, atol=2e-5, rtol=1e-4), (name, np.abs(a.numpy() - b).max())


def test_tokenizers_agree(ref):
    from bert_pytorch_b200.data import tokenization as T
    vocab = T.load_vocab(os.path.join(ref["work"], "vocab.txt"))
    basic, wp = T.BasicTokenizer(do_lower_case=True), T.WordpieceTokenizer(vocab=vocab)
    assert [basic.tokenize(t) for t in TEXTS] == ref["basic"]
    assert [[p for w in basic.tokenize(t) for p in wp.tokenize(w)] for t in TEXTS] == ref["wordpiece"]
    assert [T.BasicTokenizer(do_lower_case=False).tokenize(t) for t in TEXTS] == ref["basic_cased"]
    bt = T.BertTokenizer(os.path.join(ref["work"], "vocab.txt"), do_lower_case=True)
    assert [(bt.tokenize(t), bt.convert_tokens_to_ids(bt.tokenize(t))) for t in TEXTS[:40]] == ref["bert_tokenizer"]
    assert bt.convert_ids_to_tokens([0, 5, 10, 28, 3]) == ref["ids_to_tokens"]


def test_squad_features_and_answers_agree(ref):
    from bert_pytorch_b200.data import squad as SQ
    from bert_pytorch_b200.data.tokenization import get_wordpiece_tokenizer
    work = ref["work"]
    tok = get_wordpiece_tokenizer(os.path.join(work, "vocab.txt"), uppercase=False)
    ex = SQ.read_squad_examples(os.path.join(work, "squad.json"), True, False)
    # the reference's answer-span refinement never fires (it compares against a string with [CLS] / [SEP]):
    # improve_answer_span=False reproduces its targets exactly, the default tightens "paris ." to "paris"
    feats = SQ.convert_examples_to_features(ex, tok, 48, 16, 12, True, improve_answer_span=False)
    tight = SQ.convert_examples_to_features(ex, tok, 48, 16, 12, True)
    assert tight[0].tokens[tight[0].start_position:tight[0].end_position + 1] == ["paris"]
    assert feats[0].tokens[feats[0].start_position:feats[0].end_position + 1] == ["paris", "."]
    assert len(feats) == len(ref["features"])
    for f, r in zip(feats, ref["features"]):
        for k, v in r.items():
            mine = getattr(f, k)
            mine = dict(mine) if isinstance(v, dict) else (list(mine) if isinstance(v, list) else mine)
            assert mine == v, (r["unique_id"], k)
    ex_eval = SQ.read_squad_examples(os.path.join(work, "squad.json"), False, False)
    feats_eval = SQ.convert_examples_to_features(ex_eval, tok, 48, 16, 12, False)
    results = [SQ.RawResult(f.unique_id, *ref["logits"][f.unique_id]) for f in feats_eval]
    answers, nbest = SQ.get_answers(ex_eval, feats_eval, results, n_best_size=5, max_answer_length=10, do_lower_case=True)
    assert dict(answers) == ref["answers"]
    for qid, lst in ref["nbest"].items():
        mine = nbest[qid]
        assert [d["text"] for d in mine] == [d["text"] for d in lst], qid
        for a, b in zip(mine, lst):
            assert abs(a["probability"] - b["probability"]) < 1e-9 and abs(a["start_logit"] - b["start_logit"]) < 1e-12


def test_schedulers_bertadam_and_sampler_agree(ref):
    from bert_pytorch_b200.data.dataset import DistributedSampler
    from bert_pytorch_b200.optim import BertAdam, LinearWarmUpScheduler, PolyWarmUpScheduler

    def lr_curve(cls, **kw):
        p = torch.nn.Parameter(torch.zeros(1))
        opt = torch.optim.SGD([p], lr=1.0)
        sch = cls(opt, **kw)
        lrs = []
        for step in range(1, 41):
            opt.param_groups[0]["step"] = step
            sch.step()
            lrs.append(opt.param_groups[0]["lr"])
        return lrs
    poly = lr_curve(PolyWarmUpScheduler, warmup=0.25, total_steps=40)
    # identical while progress <= 1; one step past the end the reference returns a complex number
    # ((1 - 41/40) ** 0.5), this repo clamps the decay at zero
    assert np.allclose(poly[:39], np.real(ref["poly"][:39]), rtol=1e-12, atol=1e-15)
    assert isinstance(ref["poly"][39], complex) and poly[39] == 0.0
    assert np.allclose(lr_curve(LinearWarmUpScheduler, warmup=0.25, total_steps=40), ref["linear"], rtol=1e-12, atol=1e-15)

    torch.manual_seed(3)
    w = torch.nn.Parameter(torch.randn(7, 5))
    opt = BertAdam([w], lr=1e-2, warmup=0.1, t_total=20, weight_decay=0.01, max_grad_norm=1.0)
    for i, want in enumerate(ref["bertadam"]):
        w.grad = torch.randn(7, 5, generator=torch.Generator().manual_seed(10 + i)) * (3.0 if i == 2 else 1.0)
        opt.step()
        assert np.allclose(w.detach().numpy(), want, atol=1e-6, rtol=1e-5), i

    class _DS(torch.utils.data.Dataset):
        files = ["x"]
        def __len__(self): return 23
        def __getitem__(self, i): return i
        def set_epoch(self, epoch): pass
    for (world, rank), want in ref["sampler"].items():
        sm = DistributedSampler(_DS(), world, rank=rank)
        sm.set_epoch(1)
        assert list(iter(sm)) == want, (world, rank)


def test_more_models_criterion_dataset_helpers_ner_and_small_helpers_agree(ref):
    from bert_pytorch_b200 import BertConfig, models as M
    from bert_pytorch_b200.data import dataset as D
    from bert_pytorch_b200.data.ner import NERDataset
    from bert_pytorch_b200.data.tokenization import get_wordpiece_tokenizer
    from bert_pytorch_b200.finetune_ner import compute_metrics
    from bert_pytorch_b200.utils.dist import format_step
    from bert_pytorch_b200.utils.file_utils import url_to_filename
    cfg = BertConfig.from_dict(MODEL_CFG)
    ids, seg, mask = (torch.tensor(a) for a in ref["spec"]["inputs"])
    ids4 = torch.stack([ids, ids.flip(1)], dim=1)
    seg4, mask4 = torch.stack([seg, seg], dim=1), torch.stack([mask, mask], dim=1)
    ctors = {"nsp": (lambda: M.BertForNextSentencePrediction(cfg), (ids, seg, mask)),
             "choice": (lambda: M.BertForMultipleChoice(cfg, 2), (ids4, seg4, mask4)),
             "encoder": (lambda: M.BertModel(cfg), (ids, seg, mask))}
    for name, (sd, outs, first_type) in ref["models2"].items():
        ctor, inp = ctors[name]
        m = ctor().eval()
        assert set(m.state_dict()) == set(sd), (name, sorted(set(m.state_dict()) ^ set(sd))[:6])
        m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()}, strict=True)
        with torch.no_grad():
            y = m(*inp)
        if isinstance(y, tuple):
            assert type(y[0]).__name__ == first_type, (name, type(y[0]).__name__, first_type)   # e.g. BertModel -> (list, tensor)
        flat = []
        for t in (y if isinstance(y, (tuple, list)) else [y]):
            flat += [u for u in (t if isinstance(t, (tuple, list)) else [t]) if torch.is_tensor(u)]
        assert len(flat) == len(outs), name
        for a, b in zip(flat, outs):
            assert a.shape == b.shape and np.allclose(a.numpy(), b, atol=2e-5, rtol=1e-4), (name, np.abs(a.numpy() - b).max())

    scores, labels, nsp_s, nsp_l, with_nsp, without = ref["criterion"]
    crit = M.BertPretrainingCriterion(cfg.vocab_size)
    t = torch.from_numpy
    assert abs(float(crit(t(scores), t(labels), t(nsp_s), t(nsp_l))) - with_nsp) < 1e-5
    assert abs(float(crit(t(scores), t(labels))) - without) < 1e-5

    row = np.zeros((1, 16), dtype=np.int32); row[0, :11] = np.arange(20, 31)
    for sp, (want_seg, want_mask) in zip(([0, 10], [0, 4, 10], [0, 1, 2]), ref["segments"]):
        sg, im = D.segment_ids_and_input_mask(row, np.array([sp], dtype=np.int32))
        assert sg[0].tolist() == want_seg and im[0].tolist() == want_mask, sp
    lab = D.labels_from_premasked(row, np.array([[2, 5, 9, 0, 0]]), np.array([[21, 22, 23, 0, 0]]))
    assert lab[0].tolist() == ref["premasked"]

    tok = get_wordpiece_tokenizer(os.path.join(ref["work"], "vocab.txt"), uppercase=False)
    nds = NERDataset(os.path.join(ref["work"], "ner.txt"), tok, NER_LABELS, 12)
    assert len(nds) == len(ref["ner"])
    for i, want in enumerate(ref["ner"]):
        assert [x.tolist() for x in nds[i]] == want, i
    preds, lbl, f1 = ref["ner_f1"]
    idx_to_label = {i: l for i, l in enumerate(NER_LABELS, start=1)}
    idx_to_label[0] = "O"
    assert abs(compute_metrics(preds, lbl, idx_to_label) - f1) < 1e-9

    assert [format_step(x) for x in ("PARAMETER", (1,), (1, 20), (2, 30, 4), ())] == ref["format_step"]
    assert [url_to_filename("https://example.org/a/b.bin"), url_to_filename("s3://bucket/key", etag='"abc"')] == ref["url_to_filename"]

    first, state = ref["sampler_state"]
    class _DS(torch.utils.data.Dataset):
        files = ["x"]
        def __len__(self): return 23
        def __getitem__(self, i): return i
        def set_epoch(self, epoch): pass
    sm = D.DistributedSampler(_DS(), 2, rank=1)
    sm.set_epoch(3)
    it = iter(sm)
    assert [next(it) for _ in range(4)] == first
    # the reference's set_epoch() only forwards to the dataset, so its state dict always says epoch 0; this
    # sampler records the epoch it was given -- everything else is identical
    assert state["epoch"] == 0 and sm.state_dict() == dict(state, epoch=3)
    sm2 = D.DistributedSampler(_DS(), 2, rank=1)
    sm2.load_state_dict(state)
    assert sm2.index == state["index"] and sm2.epoch == state["epoch"]


def test_cli_defaults_overlay_and_initialisation_agree(ref, monkeypatch):
    from bert_pytorch_b200 import BertConfig, finetune_ner, models as M, pretrain
    from bert_pytorch_b200.data.encode import TrainingSample
    monkeypatch.delenv("LOCAL_RANK", raising=False)
    for argv, want in zip(ref["spec"]["pretrain_argvs"], ref["cli_pretrain"]):
        mine = vars(pretrain.parse_arguments(argv))
        for k, v in want.items():                                   # every reference flag: same name, same resolved value
            assert k in mine, k
            assert mine[k] == v, (argv, k, mine[k], v)
    mine = vars(finetune_ner.parse_arguments(ref["spec"]["ner_argv"]))
    for k, v in ref["cli_ner"].items():
        assert k in mine and mine[k] == v, (k, mine.get(k), v)

    # same seed -> the same freshly initialised weights, tensor by tensor (module order, init rules, kaiming vs normal)
    cfg = BertConfig.from_dict(MODEL_CFG)
    torch.manual_seed(123)
    fresh = M.BertForPreTraining(cfg).state_dict()
    assert list(fresh) == list(ref["fresh"])                          # same registration order
    exact = 0
    for k, (shape, mean, std) in ref["fresh"].items():
        v = fresh[k]
        assert tuple(v.shape) == shape, k
        if _digest(v.numpy()) == ref["fresh_exact"][k]:
            exact += 1
            continue
        assert abs(float(v.float().mean()) - mean) < 0.02 and abs((float(v.float().std()) if v.numel() > 1 else 0.0) - std) < 0.02 + 0.25 * std, k
    assert exact >= len(fresh) // 2, (exact, len(fresh))              # LayerNorm / bias tensors at least are bit-identical

    mine_json = json.loads(cfg.to_json_string())
    for k, v in ref["config_json"].items():
        assert mine_json.get(k) == v, k

    if isinstance(ref["samples"], list):
        ts = [TrainingSample([1, 2, 3]), TrainingSample([1, 2], [3, 4, 5], True), TrainingSample([], [])]
        for t, (seq, special, rnd) in zip(ts, ref["samples"]):
            ids, sp = t.layout(101, 102)
            assert sp == special and len(ids) == len(seq) and t.is_random_next == rnd
            assert [i for i, tok in enumerate(seq) if tok in ("[CLS]", "[SEP]")] == sp


def test_squad_v2_helpers_and_sharded_dataset_agree(ref):
    from bert_pytorch_b200.data import dataset as D, squad as SQ
    from bert_pytorch_b200.data.tokenization import get_wordpiece_tokenizer
    work = ref["work"]
    tok = get_wordpiece_tokenizer(os.path.join(work, "vocab.txt"), uppercase=False)
    ex2 = SQ.read_squad_examples(os.path.join(work, "squad2.json"), True, True)
    assert [(e.qas_id, e.is_impossible, e.start_position, e.end_position, e.orig_answer_text) for e in ex2] == ref["v2_examples"]
    f2 = SQ.convert_examples_to_features(ex2, tok, 48, 16, 12, True, improve_answer_span=False)
    assert [(f.unique_id, f.start_position, f.end_position, f.is_impossible) for f in f2] == ref["v2_features"]
    ex2e = SQ.read_squad_examples(os.path.join(work, "squad2.json"), False, True)
    f2e = SQ.convert_examples_to_features(ex2e, tok, 48, 16, 12, False)
    res2 = [SQ.RawResult(f.unique_id, *ref["v2_logits"][f.unique_id]) for f in f2e]
    ans, nb = SQ.get_answers(ex2e, f2e, res2, n_best_size=4, max_answer_length=8, do_lower_case=True,
                             version_2_with_negative=True, null_score_diff_threshold=-1.0)
    # the reference indexes its null scores with the LAST example for every question (quirk Q20): only the last
    # question of the file is comparable; the first one must simply be well formed here
    last = ex2e[-1].qas_id
    assert ans[last] == ref["v2_answers"][last]
    assert [d["text"] for d in nb[last]] == [d["text"] for d in ref["v2_nbest"][last]]
    for a, b in zip(nb[last], ref["v2_nbest"][last]):
        assert abs(a["probability"] - b["probability"]) < 1e-9
    assert set(ans) == set(ref["v2_answers"]) and all(len(v) >= 1 for v in nb.values())

    assert [SQ.get_final_text(a, b, True, False) for a, b in ref["spec"]["final_text_pairs"]] == ref["final_text"]
    assert SQ._get_best_indices([0.1, 3.0, -1.0, 3.0, 2.5, 0.0], 3) == ref["best_indices"]
    assert np.allclose(SQ._compute_softmax([1.0, 2.0, -3.0, 0.5]), ref["softmax"], rtol=1e-12)

    ds = D.ShardedPretrainingDataset(sorted(ref["spec"]["shards"]), 4, 5, 0.2, vocab_size=100, seed=0)
    assert len(ds) == ref["dataset_len"]
    for i, (seg, msk, nsl, n_masked, width) in enumerate(ref["dataset_rows"]):
        ids_, seg_, msk_, lab_, nsl_ = ds[i]
        assert np.asarray(seg_).tolist() == seg and np.asarray(msk_).tolist() == msk and int(np.asarray(nsl_)) == nsl, i
        assert np.asarray(ids_).shape[0] == width
        assert 1 <= int((np.asarray(lab_) >= 0).sum()) <= 5 and 1 <= n_masked <= 5     # masking itself is random on both sides


def test_training_steps_agree(ref):
    """Four optimisation steps of BertForPreTraining + criterion + BertAdam from the reference's initial weights:
    the same loss trajectory and the same final weights (autograd backward of every module, tied decoder, optimizer)."""
    from bert_pytorch_b200 import BertConfig, models as M
    from bert_pytorch_b200.optim import BertAdam
    cfg0 = BertConfig.from_dict(dict(MODEL_CFG, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0))
    ids, seg, mask = (torch.tensor(a) for a in ref["spec"]["inputs"])
    net = M.BertForPreTraining(cfg0).train()
    net.load_state_dict({k: torch.from_numpy(v) for k, v in ref["train_init"].items()}, strict=True)
    opt = BertAdam([p for p in net.parameters()], lr=5e-3, warmup=0.2, t_total=10, weight_decay=0.01, max_grad_norm=1.0)
    crit = M.BertPretrainingCriterion(cfg0.vocab_size)
    lab = torch.full_like(ids, -1); lab[:, 2] = 9; lab[:, 7] = 30; lab[0, 11] = 5
    nsl = torch.tensor([1, 0, 1])
    for step, want in enumerate(ref["train_losses"]):
        sc, rel = net(torch.roll(ids, step, 1), seg, mask)
        loss = crit(sc, lab, rel, nsl)
        loss.backward()
        opt.step(); opt.zero_grad()
        assert abs(float(loss) - want) < 2e-5 * max(1.0, abs(want)), (step, float(loss), want)
    worst = max(float(np.abs(_sample(v.numpy()) - ref["train_final"][k]).max()) for k, v in net.state_dict().items())
    assert worst < 5e-5, worst


def _squad_cli_args(work, tmp_path):
    """run_squad.py command line (without --output_dir) over a checkpoint with ``det_fill`` weights."""
    from bert_pytorch_b200 import BertConfig, models as M
    cfg = dict(MODEL_CFG, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0,
               vocab_file=os.path.join(work, "vocab.txt"), tokenizer="wordpiece", lowercase=True)
    model_json = str(tmp_path / "model.json")
    json.dump(cfg, open(model_json, "w"))
    sd = M.BertForPreTraining(BertConfig.from_dict(cfg)).state_dict()
    det_fill(sd, 5)
    ckpt = str(tmp_path / "ckpt_10.pt")
    torch.save({"model": sd}, ckpt)
    return ["--no_cuda", "--bert_model", "bert-large-uncased", "--init_checkpoint", ckpt, "--config_file", model_json,
            "--vocab_file", cfg["vocab_file"], "--do_predict", "--predict_file", os.path.join(work, "squad.json"),
            "--predict_batch_size", "4", "--max_seq_length", "48", "--doc_stride", "16", "--max_query_length", "12",
            "--do_lower_case", "--seed", "42"]


def _original_run_squad(ref_dir, work, tmp_path):
    env = dict(os.environ, PYTHONPATH=os.path.join(ROOT, "baseline", "shims"), CUDA_VISIBLE_DEVICES="")
    out = tmp_path / "ref_out"
    subprocess.run([sys.executable, "run_squad.py", *_squad_cli_args(work, tmp_path), "--output_dir", str(out)], cwd=ref_dir,
                   env=env, check=True, capture_output=True, text=True, timeout=600)
    return json.load(open(out / "predictions.json")), json.load(open(out / "nbest_predictions.json"))


def test_run_squad_predict_cli_end_to_end(ref, golden, tmp_path):
    """Both run_squad.py command lines (the original's and this repo's), same checkpoint, prediction only on the CPU:
    identical predictions.json and n-best lists (CLI -> checkpoint load -> features -> forward -> post-processing)."""
    from bert_pytorch_b200 import finetune_squad
    finetune_squad.main([*_squad_cli_args(ref["work"], tmp_path), "--output_dir", str(tmp_path / "my_out")])
    a, na = golden["run_squad"]
    b = json.load(open(tmp_path / "my_out" / "predictions.json"))
    assert a == b and {"q1", "q2", "q3"} <= set(a) and len(a) >= 15
    nb = json.load(open(tmp_path / "my_out" / "nbest_predictions.json"))
    for k in na:
        # logits come out of two implementations of the forward pass (agreement ~1e-6): candidates whose scores are
        # (nearly) tied may swap places deep in the list, so compare the head exactly and the tail as a set
        ta, tb = [x["text"] for x in na[k]], [x["text"] for x in nb[k]]
        assert ta[:3] == tb[:3] and len(ta) == len(tb), k
        assert len(set(ta[:15]) & set(tb[:15])) >= min(13, len(set(ta[:15]))), k
        assert max(abs(x["probability"] - y["probability"]) for x, y in zip(na[k][:3], nb[k][:3])) < 1e-3   # normalised over a list whose tail may differ


def _load_original_util(ref_dir, script):
    """A module of the original's utils/ directory (the h5py stand-in of baseline/shims on the path for its import)."""
    import importlib.util
    sys.path.insert(0, os.path.join(ROOT, "baseline", "shims"))
    try:
        spec = importlib.util.spec_from_file_location("original_" + script[:-3], os.path.join(ref_dir, "utils", script))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        sys.path.pop(0)
    return mod


SHARD_TEXT = "".join(f"Article {i} sentence one.\nArticle {i} sentence two is a little longer than one.\n\n" for i in range(40))
SHARD_SIZES = (5, "123", "2K", "1.5M", "3b")


def _original_shard(ref_dir, tmp_path):
    RSH = _load_original_util(ref_dir, "shard.py")
    src = tmp_path / "in.txt"
    src.write_text(SHARD_TEXT)
    files = {}
    for limit in (None, 3):
        a = tmp_path / f"ref_{limit}"
        a.mkdir()
        RSH.shard(str(src), str(a / "shard_{index}.txt"), 700, limit)
        files[limit] = {f: (a / f).read_text() for f in sorted(os.listdir(a))}
    return files, [RSH.parse_value_as_int(v) for v in SHARD_SIZES]


def test_text_sharder_agrees(golden, tmp_path):
    """utils/shard.py: same shard files for the same input (split at the first article boundary past the byte budget,
    1-based names, optional shard limit) and the same size parser."""
    from bert_pytorch_b200.data import corpus
    files, sizes = golden["shard"]
    src = tmp_path / "in.txt"
    src.write_text(SHARD_TEXT)
    for limit in (None, 3):
        b = tmp_path / f"mine_{limit}"
        b.mkdir()
        corpus.shard_text(str(src), str(b / "shard_{index}.txt"), 700, limit)
        fa, fb = sorted(files[limit]), sorted(os.listdir(b))
        assert fa == fb and len(fa) >= 3, (fa, fb)
        for f in fa:
            assert files[limit][f] == (b / f).read_text(), (limit, f)
    assert [corpus.parse_value_as_int(v) for v in SHARD_SIZES] == sizes


SAMPLE_TEXT = "".join("".join(f"Article {i} sentence {j}.\n" for j in range(1 + i % 4)) + "\n" for i in range(60))


def _original_sample_and_shard(ref_dir, tmp_path):
    src, a = tmp_path / "in.txt", tmp_path / "ref"
    src.write_text(SAMPLE_TEXT)
    code = ("import random, runpy, sys; random.seed(11); sys.argv = ['sample_and_shard.py', '-i', sys.argv[1], '-o', sys.argv[2], "
            "'-b', '400', '-n', '50']; runpy.run_path(%r, run_name='__main__')"
            % os.path.join(ref_dir, "utils", "sample_and_shard.py"))
    subprocess.run([sys.executable, "-c", code, str(src), str(a)], check=True, capture_output=True, text=True, timeout=300)
    return {f: (a / f).read_text() for f in sorted(os.listdir(a))}


def test_sample_and_shard_agrees(golden, tmp_path):
    """utils/sample_and_shard.py under the same `random` seed: the same articles in the same shard files."""
    import random
    from bert_pytorch_b200.data import corpus
    src, b = tmp_path / "in.txt", tmp_path / "mine"
    src.write_text(SAMPLE_TEXT)
    corpus.sample_and_shard([str(src)], str(b / "shard_{index}.txt"), 400, 50, random.Random(11))
    want = golden["sample_and_shard"]
    fa, fb = sorted(want), sorted(os.listdir(b))
    assert fa == fb and len(fa) >= 2, (fa, fb)
    for f in fa:
        assert want[f] == (b / f).read_text(), f


def _packing_docs():
    import random
    gen = random.Random(5)
    return [[[gen.randrange(10, 500) for _ in range(gen.randint(1, 30))] for _ in range(gen.randint(1, 12))] for _ in range(9)]


def _original_packing(ref_dir):
    import random
    E = _load_original_util(ref_dir, "encode_data.py")
    docs_ref = [[[f"t{t}" for t in sent] for sent in d] for d in _packing_docs()]
    out = {}
    for next_seq_prob in (0.5, 0.0):
        for seed in range(6):
            random.seed(seed)
            want = []
            for i in range(len(docs_ref)):
                want.extend(E.create_samples_from_document(i, docs_ref, 48, next_seq_prob, 0.3))
            random.shuffle(want)
            out[next_seq_prob, seed] = [(w.seq_tokens, w.next_seq_tokens, w.is_random_next, w.special_token_positions,
                                         len(w.sequence)) for w in want]
    return out


@pytest.mark.parametrize("next_seq_prob", [0.5, 0.0])
def test_sample_packing_agrees_draw_for_draw(golden, next_seq_prob):
    """utils/encode_data.py:create_samples_from_document under the same `random` seed: the packer makes the same random
    decisions in the same order (target lengths, A/B cut, random-next documents, re-use of displaced sentences, final
    shuffle), so the samples are identical."""
    import random
    from bert_pytorch_b200.data.encode import SamplePacker
    docs = _packing_docs()
    for seed in range(6):
        want = golden["packing"][next_seq_prob, seed]
        got = SamplePacker(48, next_seq_prob, 0.3, random.Random(seed)).pack_file(docs)
        assert len(got) == len(want), seed
        for g, (seq_tokens, next_seq_tokens, is_random_next, special_positions, n) in zip(got, want):
            assert [f"t{t}" for t in g.seq_ids] == seq_tokens, seed
            assert (None if g.next_seq_ids is None else [f"t{t}" for t in g.next_seq_ids]) == next_seq_tokens, seed
            assert g.is_random_next == is_random_next
            ids, special = g.layout(1, 2)
            assert special == special_positions and len(ids) == n <= 48


def test_dynamic_masking_statistics_agree(ref):
    """Same sampling law as src/dataset.py:_mask_input (draws WITH replacement, 80/10/10 applied in draw order): labelled
    positions per sample and the [MASK] / kept / random split agree with the reference within sampling noise."""
    from bert_pytorch_b200.data.dataset import mask_batch
    base = np.zeros((1, 64), dtype=np.int32); base[0, :50] = np.arange(100, 150)
    sp = np.array([[0, 20, 49]], dtype=np.int32)
    rng = np.random.default_rng(9)
    rows = np.repeat(base, 3000, axis=0)
    ids_m, lab = mask_batch(rows, np.repeat(sp, 3000, axis=0), mask_token_index=4, max_pred_per_seq=20, masked_lm_prob=0.2,
                            vocab_size=1000, rng=rng)
    sel = lab >= 0
    assert not sel[:, [0, 20, 49]].any() and not sel[:, 50:].any()
    n_lab = sel.sum()
    mine = (n_lab / 3000.0, (ids_m[sel] == 4).sum() / n_lab, (ids_m[sel] == rows[sel]).sum() / n_lab,
            ((ids_m[sel] != 4) & (ids_m[sel] != rows[sel])).sum() / n_lab)
    per_sample, p_mask, p_keep, p_rand, bad = ref["mask_stats"]
    assert bad == 0
    assert abs(mine[0] - per_sample) < 0.15, (mine[0], per_sample)          # ~8.3 unique positions out of 9 draws
    for a, b in zip(mine[1:], (p_mask, p_keep, p_rand)):
        assert abs(a - b) < 0.012, (mine, ref["mask_stats"])


def test_task_models_with_labels_return_the_same_loss(ref):
    from bert_pytorch_b200 import BertConfig, models as M
    cfg = BertConfig.from_dict(MODEL_CFG)
    ids, seg, mask = (torch.tensor(a) for a in ref["spec"]["inputs"])
    ids4 = torch.stack([ids, ids.flip(1)], dim=1)
    seg4, mask4 = torch.stack([seg, seg], dim=1), torch.stack([mask, mask], dim=1)
    lab_tok = torch.randint(0, 5, ids.shape, generator=torch.Generator().manual_seed(2))
    mlm_lab = torch.full_like(ids, -1); mlm_lab[:, 4] = 17; mlm_lab[2, 1] = 8
    cases = {"mlm": (lambda: M.BertForMaskedLM(cfg), dict(masked_lm_labels=mlm_lab)),
             "nsp": (lambda: M.BertForNextSentencePrediction(cfg), dict(next_sentence_label=torch.tensor([0, 1, 0]))),
             "token": (lambda: M.BertForTokenClassification(cfg, 5), dict(labels=lab_tok)),
             "choice": (lambda: M.BertForMultipleChoice(cfg, 2), dict(labels=torch.tensor([1, 0, 1])))}
    for name, (sd, want) in ref["with_labels"].items():
        ctor, kwargs = cases[name]
        m = ctor().eval()
        m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()}, strict=True)
        inp = (ids4, seg4, mask4) if name == "choice" else (ids, seg, mask)
        with torch.no_grad():
            y = m(*inp, **kwargs)
        got = float(y if torch.is_tensor(y) else y[0])
        assert abs(got - want) < 2e-5 * max(1.0, abs(want)), (name, got, want)


def test_from_pretrained_agrees(ref):
    """A reference-written archive directory in the old gamma / beta naming loads through ``from_pretrained`` into the full
    model, a bare encoder (``bert.`` prefix) and a task model with constructor arguments -- same outputs."""
    from bert_pytorch_b200 import models as M
    pt_dir = os.path.join(ref["work"], "pretrained")
    ids, seg, mask = (torch.tensor(a) for a in ref["spec"]["inputs"])
    loaders = {"pretraining": lambda: M.BertForPreTraining.from_pretrained(pt_dir),
               "encoder": lambda: M.BertModel.from_pretrained(pt_dir),
               "token": lambda: M.BertForTokenClassification.from_pretrained(pt_dir, num_labels=5)}
    for name, want in ref["from_pretrained"].items():
        torch.manual_seed(33)
        m = loaders[name]().eval()
        with torch.no_grad():
            y = m(ids, seg, mask)
        flat = []
        for t in (y if isinstance(y, (tuple, list)) else [y]):
            flat += [u for u in (t if isinstance(t, (tuple, list)) else [t]) if torch.is_tensor(u)]
        assert len(flat) == len(want), name
        for a, b in zip(flat, want):
            if name == "token":                     # the classifier is freshly initialised on both sides: shapes only
                assert a.shape == b.shape
            else:
                assert np.allclose(a.numpy(), b, atol=2e-5, rtol=1e-4), (name, np.abs(a.numpy() - b).max())


class _Tok:                                                # "t17" -> 17, specials like a real vocabulary
    def token_to_id(self, t):
        return {"[CLS]": 101, "[SEP]": 102}.get(t) or int(t[1:])


WRITER_SAMPLES = [([5, 6, 7], [8, 9], True), ([10], [11, 12, 13, 14], False), ([20, 21, 22, 23, 24], [25], False)]


def _original_shard_writer(ref_dir, tmp_path):
    from bert_pytorch_b200.data import hdf5
    E = _load_original_util(ref_dir, "encode_data.py")
    out = {}
    for nsp in (True, False):
        ref_samples = [E.TrainingSample([f"t{x}" for x in a], [f"t{x}" for x in b] if nsp else None, r and nsp)
                       for a, b, r in WRITER_SAMPLES]
        fa = str(tmp_path / f"ref_{nsp}.hdf5")
        E.write_samples_to_hdf5(fa, list(ref_samples), _Tok(), 16)
        with hdf5.File(fa, "r") as A:
            out[nsp] = {k: A[k][:] for k in A.keys()}
    return out


def test_shard_writer_agrees(golden, tmp_path):
    """utils/encode_data.py:write_samples_to_hdf5 (the original, writing through the h5py stand-in = this repo's HDF5
    writer) and data/encode.py write the same three datasets for the same samples (the original pops from the end of the
    list, so its rows come out reversed)."""
    from bert_pytorch_b200.data import encode, hdf5
    for nsp in (True, False):
        mine = [encode.TrainingSample(list(a), list(b) if nsp else None, r and nsp) for a, b, r in WRITER_SAMPLES]
        fb = str(tmp_path / f"mine_{nsp}.hdf5")
        encode.write_samples_to_hdf5(fb, mine, 16, 101, 102)
        A = golden["shard_writer"][nsp]
        with hdf5.File(fb, "r") as B:
            assert sorted(A.keys()) == sorted(B.keys()) == ["input_ids", "next_sentence_labels", "special_token_positions"]
            for k in A.keys():
                a, b = A[k], B[k][:]
                assert a.dtype == b.dtype and a.shape == b.shape, (k, a.dtype, b.dtype, a.shape, b.shape)
                assert np.array_equal(a[::-1], b), k


def test_runtime_micro_step_accumulation_agrees(ref):
    """pretrain.forward_backward_pass vs run_pretraining.forward_backward_pass: three accumulated micro-steps with
    divisor 3 return the same (already divided) losses and leave the same summed gradients."""
    from bert_pytorch_b200 import BertConfig, models as M, pretrain
    from bert_pytorch_b200.models.arena import ParamArena
    from bert_pytorch_b200.parallel import DataParallel
    from bert_pytorch_b200.parallel.comm import SingleComm
    cfg0 = BertConfig.from_dict(dict(MODEL_CFG, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0))
    ids, seg, mask = (torch.tensor(a) for a in ref["spec"]["inputs"])
    net = M.BertForPreTraining(cfg0).train()
    net.load_state_dict({k: torch.from_numpy(v) for k, v in ref["train_init"].items()}, strict=True)
    arena = ParamArena(net)
    ddp = DataParallel(net, comm=SingleComm(), arena=arena)
    crit = M.BertPretrainingCriterion(cfg0.vocab_size)
    lab = torch.full_like(ids, -1); lab[:, 2] = 9; lab[:, 7] = 30; lab[0, 11] = 5
    nsl = torch.tensor([1, 0, 1])
    for mstep, want in enumerate(ref["micro_losses"]):
        batch = (torch.roll(ids, mstep, 1), seg, mask, lab, nsl)
        loss = pretrain.forward_backward_pass(ddp, crit, None, batch, 3, sync_grads=(mstep == 2), compute_dtype=torch.float32)
        assert abs(float(loss) - want) < 2e-5 * max(1.0, abs(want)), (mstep, float(loss), want)
    for k, p in net.named_parameters():
        if k in ref["micro_grads"]:
            g, g_max = ref["micro_grads"][k]
            assert np.allclose(_sample(p.grad.numpy()), g, atol=2e-6 + 1e-4 * g_max), k


def test_optimizer_groups_and_resume_surgery(ref):
    """pretrain.prepare_optimizers vs run_pretraining.prepare_optimizers: the same decay / no-decay parameter groups, and
    on a phase-1 -> phase-2 resume the same surgery (step counters reset, t_total / warmup / lr overwritten).  One
    deliberate difference: the reference leaves the scheduler's ``initial_lr`` of the checkpoint in place, so its
    phase 2 decays from the PHASE-1 learning rate although ``lr`` was overwritten; here phase 2 starts from its own."""
    import copy
    import types
    from bert_pytorch_b200 import BertConfig, models as M, pretrain
    from bert_pytorch_b200.models.arena import ParamArena
    from bert_pytorch_b200.parallel import DataParallel
    from bert_pytorch_b200.parallel.comm import SingleComm
    cfg0 = BertConfig.from_dict(dict(MODEL_CFG, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0))
    net = M.BertForPreTraining(cfg0)
    ddp = DataParallel(net, comm=SingleComm(), arena=ParamArena(net))
    base = dict(lr_decay="poly", fp16=False, kfac=False, device_obj=torch.device("cpu"))
    a1 = types.SimpleNamespace(learning_rate=6e-3, warmup_proportion=0.25, max_steps=8, resume_step=0, previous_phase_end_step=0, **base)
    opt, _, sch, _ = pretrain.prepare_optimizers(a1, ddp, None, 0)
    names = dict((id(p), n) for n, p in net.named_parameters())
    mine = [(g["weight_decay"], sorted(names[id(p)] for p in g["params"])) for g in opt.param_groups]
    assert mine == ref["opt_groups"]
    for _ in range(4):
        for p in net.parameters():
            p.grad.fill_(0.01) if p.grad is not None else None
        sch[0].step(); opt.step()
    ck = {"optimizer": copy.deepcopy(opt.state_dict())}
    a2 = types.SimpleNamespace(learning_rate=4e-3, warmup_proportion=0.5, max_steps=10, resume_step=4, previous_phase_end_step=4, **base)
    net2 = M.BertForPreTraining(cfg0)
    ddp2 = DataParallel(net2, comm=SingleComm(), arena=ParamArena(net2))
    opt2, _, sch2, _ = pretrain.prepare_optimizers(a2, ddp2, ck, 0)
    g, want = opt2.param_groups[0], ref["resumed_group"]
    for k in ("step", "t_total", "warmup", "weight_decay", "betas", "eps", "bias_correction", "grad_averaging", "max_grad_norm"):
        assert g[k] == want[k] or tuple(g[k]) == tuple(want[k]), (k, g[k], want[k])
    assert sorted({int(st["step"]) for st in opt2.state_dict()["state"].values()}) == ref["resumed_state_steps"] == [0]
    assert ref["resumed_base_lrs"] == [6e-3, 6e-3] and want["initial_lr"] == 6e-3      # the reference keeps phase 1's base LR
    assert list(sch2[0].base_lrs) == [4e-3, 4e-3]                                       # this repo uses the configured one


def test_legacy_premasked_shards_agree(ref):
    """Shards in the NVIDIA pre-masked layout (no dynamic masking, nothing random): all five outputs of every sample are
    identical, and a missing / unreadable file in the list is skipped by both."""
    import warnings
    from bert_pytorch_b200.data.dataset import ShardedPretrainingDataset
    work = ref["work"]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ds = ShardedPretrainingDataset(sorted(ref["spec"]["legacy_shards"]) + [os.path.join(work, "does_not_exist.hdf5"),
                                                                                os.path.join(work, "vocab.txt")],
                                       4, 5, 0.2, vocab_size=100)
    assert len(ds) == ref["legacy_len"] == 11
    for i, want in enumerate(ref["legacy_rows"]):
        got = [np.asarray(a).tolist() for a in ds[i]]
        assert got == want, i


def test_ner_get_data_agrees(ref):
    import types
    from bert_pytorch_b200 import finetune_ner
    work = ref["work"]
    args = types.SimpleNamespace(cuda=False, batch_size=2, vocab_file=None, tokenizer=None,
                                 model_config_file=os.path.join(work, "ner_model.json"), uppercase=False,
                                 train_file=os.path.join(work, "ner.txt"), val_file=os.path.join(work, "ner.txt"), test_file=None,
                                 labels=NER_LABELS, max_seq_len=12)
    tl, vl, tel = finetune_ner.get_data(args)
    n_train, n_val, no_test, vocab_file, tok_kind, val_batches = ref["ner_get_data"]
    assert (len(tl), len(vl), tel is None) == (n_train, n_val, no_test)
    assert args.vocab_file == vocab_file and args.tokenizer == tok_kind
    assert [[t.tolist() for t in b] for b in vl] == val_batches


def test_prepare_dataset_agrees(ref):
    import types
    from bert_pytorch_b200 import pretrain
    work = ref["work"]
    args = types.SimpleNamespace(input_dir=os.path.dirname(ref["spec"]["shards"][0]), model_config_file=os.path.join(work, "pt_model.json"),
                                 max_predictions_per_seq=5, masked_token_fraction=0.2, local_batch_size=4, seed=42, loader_depth=2,
                                 device_obj=torch.device("cpu"))
    loader, sampler = pretrain.prepare_dataset(args, {"sampler": {"epoch": 0, "seed": 0, "num_replicas": 1, "total_size": 21, "index": 9}})
    n_data, n_sampler, index, n_batches, mask_id = ref["prepare_dataset"]
    assert (len(loader.dataset), len(sampler), sampler.index) == (n_data, n_sampler, index)
    assert loader.dataset.mask_token_index == mask_id
    # the reference's DataLoader reports the batches of a full epoch; this loader reports what is left after the resume point
    assert n_batches == -(-n_data // 4) and len(loader) == -(-(n_data - index) // 4)
    loader.close()


def test_activation_table_and_linear_activation_agree(ref):
    from bert_pytorch_b200 import models as M
    xa, ba, acts = ref["acts"]
    x, b = torch.from_numpy(xa), torch.from_numpy(ba)
    assert set(acts) <= set(M.ACT2FN), sorted(set(acts) - set(M.ACT2FN))
    for name, want in acts.items():
        if isinstance(want, str):
            continue
        got = (M.ACT2FN[name](b, x) if name.startswith("bias_") else M.ACT2FN[name](x)).numpy()
        assert np.allclose(got, want, atol=1e-6, rtol=1e-5), name
    sd_g, y_g, sd_t, y_t = ref["linear_act"]
    for act, sd, want in (("gelu", sd_g, y_g), ("tanh", sd_t, y_t)):
        m = M.LinearActivation(7, 6, act=act)
        m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()}, strict=True)
        assert np.allclose(m(x).detach().numpy(), want, atol=1e-6, rtol=1e-5), act


def _original_run_squad_flags(ref_dir):
    """run_squad.py builds its parser inside main(): flag -> default / action / type name of its add_argument calls
    (AST, nothing is executed)."""
    import ast
    tree = ast.parse(open(os.path.join(ref_dir, "run_squad.py")).read())
    ref = {}
    for node in ast.walk(tree):
        if isinstance(node, ast.Call) and isinstance(node.func, ast.Attribute) and node.func.attr == "add_argument":
            names = [a.value for a in node.args if isinstance(a, ast.Constant) and isinstance(a.value, str)]
            if not names:
                continue
            kw = {}
            for k in node.keywords:
                if k.arg in ("default", "action"):
                    try:
                        kw[k.arg] = ast.literal_eval(k.value)
                    except ValueError:
                        kw[k.arg] = None                         # computed default (LOCAL_RANK from the environment)
                elif k.arg == "type" and isinstance(k.value, ast.Name):
                    kw["type"] = k.value.id
            ref[names[-1].lstrip("-").replace("-", "_")] = kw
    return ref


def test_run_squad_flags_and_defaults_agree(golden):
    """Every flag of the original run_squad.py exists in this repo's parser with the same default, type and store_true
    behaviour."""
    from bert_pytorch_b200 import finetune_squad
    ref = golden["run_squad_flags"]
    assert len(ref) >= 40
    mine = {a.dest: a for a in finetune_squad.build_parser()._actions}
    assert not [k for k in ref if k not in mine]
    for k, kw in ref.items():
        a = mine[k]
        if kw.get("default", None) is not None:
            assert a.default == kw["default"], (k, a.default, kw["default"])
        if kw.get("action") == "store_true":
            assert a.nargs == 0 and a.const is True and a.default is False, k
        if kw.get("type") in ("int", "float", "str") and a.type is not None:
            assert a.type.__name__ == kw["type"], k


def _argparse_table(path):
    """flag -> (default, type name, action) of every add_argument call in a source file (AST, nothing is executed)."""
    import ast
    table = {}
    for node in ast.walk(ast.parse(open(path).read())):
        if isinstance(node, ast.Call) and isinstance(node.func, ast.Attribute) and node.func.attr == "add_argument":
            names = [a.value for a in node.args if isinstance(a, ast.Constant) and isinstance(a.value, str)]
            if not names:
                continue
            kw = {"default": None, "type": None, "action": None}
            for k in node.keywords:
                if k.arg in ("default", "action"):
                    try:
                        kw[k.arg] = ast.literal_eval(k.value)
                    except ValueError:
                        kw[k.arg] = "<computed>"
                elif k.arg == "type" and isinstance(k.value, ast.Name):
                    kw["type"] = k.value.id
            table[names[-1].lstrip("-").replace("-", "_")] = kw
    return table


DATA_TOOLS = ["encode_data.py", "format.py", "download.py", "build_vocab.py", "shard.py", "sample_and_shard.py"]


@pytest.mark.parametrize("script", DATA_TOOLS)
def test_data_tool_flags_and_defaults_agree(golden, script):
    ref, mine = golden["data_tool_flags"][script], _argparse_table(os.path.join(ROOT, "utils", script))
    assert ref, script
    for flag, kw in ref.items():
        assert flag in mine, (script, flag)
        m = mine[flag]
        if kw["default"] not in (None, "<computed>"):
            assert m["default"] == kw["default"], (script, flag, m["default"], kw["default"])
        if kw["action"] == "store_true":
            assert m["action"] == "store_true", (script, flag)
        if kw["type"] in ("int", "float", "str") and m["type"] is not None:
            assert m["type"] == kw["type"], (script, flag)


def _regenerate(ref_dir):
    """Run the original code at ``ref_dir`` on this module's inputs and rewrite the golden file."""
    import pathlib
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        tmp = pathlib.Path(d)
        work = tmp / "work"
        work.mkdir()
        spec = _write_inputs(work, os.path.join(ref_dir, "utils"))
        (work / "ref_script.py").write_text(FILL_SRC + REF_SCRIPT)
        env = dict(os.environ, PYTHONPATH=os.path.join(ROOT, "baseline", "shims"), CUDA_VISIBLE_DEVICES="")
        subprocess.run([sys.executable, str(work / "ref_script.py"), str(work)], cwd=ref_dir, env=env, check=True, timeout=600)
        out = pickle.load(open(work / "ref.pkl", "rb"))
        assert not isinstance(out["samples"], str), out["samples"]
        golden = {"script": _compact(out, str(work))}
        for name, make in (("run_squad", lambda t: _original_run_squad(ref_dir, str(work), t)),
                           ("shard", lambda t: _original_shard(ref_dir, t)),
                           ("sample_and_shard", lambda t: _original_sample_and_shard(ref_dir, t)),
                           ("packing", lambda t: _original_packing(ref_dir)),
                           ("shard_writer", lambda t: _original_shard_writer(ref_dir, t)),
                           ("run_squad_flags", lambda t: _original_run_squad_flags(ref_dir)),
                           ("data_tool_flags", lambda t: {s: _argparse_table(os.path.join(ref_dir, "utils", s)) for s in DATA_TOOLS})):
            (tmp / name).mkdir()
            golden[name] = make(tmp / name)
    os.makedirs(os.path.dirname(GOLDEN), exist_ok=True)
    with gzip.GzipFile(GOLDEN, "wb", mtime=0) as f:
        pickle.dump(golden, f, protocol=4)


if __name__ == "__main__":
    sys.path.insert(0, ROOT)
    _regenerate(os.path.abspath(sys.argv[1]))
