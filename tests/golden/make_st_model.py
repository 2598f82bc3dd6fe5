"""Generate the sentence-transformers model-directory fixtures by running the REFERENCE's own module classes.

    python tests/golden/make_st_model.py     # needs /root/reference and `transformers`; writes st_tiny*/ + st_tiny.npz

What is executed: HuggingFace ``GPTNeoModel`` (tiny, seeded) saved with ``save_pretrained`` exactly like
``models/Transformer.py:158-163``; the reference's ``models/WeightedMeanPooling.py``, ``models/Pooling.py``,
``models/Dense.py``, ``models/Asym.py`` and ``models/Normalize.py`` — loaded by file path as members of a stub
``sentence_transformers`` package (the real package import needs nltk / hub helpers that are absent offline) — are
instantiated, given random parameters, SAVED with their own ``save`` methods (so the directory layout and file
contents are the reference's) and RUN on the HF hidden states to produce the expected sentence embeddings.
``modules.json`` is written in the format of ``SentenceTransformer.save`` (SentenceTransformer.py:416-429).

Two model directories:
  st_tiny/       Transformer -> WeightedMeanPooling (learnt position weights) -> Dense(Tanh) -> Normalize
  st_tiny_asym/  Transformer (files shared: modules.json path "../st_tiny") -> Pooling(weightedmean)
                 -> Asym{QRY: [Dense(Identity)], DOCPOS: [Dense(Tanh)]}
and st_tiny.npz with the token batch and the embeddings the reference modules produce for it.
The GPU box has no /root/reference, so the fixtures are committed; tests only read them.
"""
import importlib.util
import json
import os
import shutil
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REF_ST = "/root/reference/biencoder/nli_msmarco/sentence-transformers/sentence_transformers"


def reference_models():
    """The reference's models/*.py as a stub package `sentence_transformers.models` (+ the two util helpers Dense/Asym
    import, restated: they are 5-line importlib helpers, util.py:430-455)."""
    pkg = types.ModuleType("sentence_transformers")
    pkg.__path__ = []
    util = types.ModuleType("sentence_transformers.util")

    def fullname(o):
        module = o.__class__.__module__
        return o.__class__.__name__ if module is None or module == str.__class__.__module__ else module + "." + o.__class__.__name__

    def import_from_string(dotted_path):
        module_path, class_name = dotted_path.rsplit(".", 1)
        return getattr(importlib.import_module(module_path), class_name)

    util.fullname, util.import_from_string = fullname, import_from_string
    models = types.ModuleType("sentence_transformers.models")
    models.__path__ = []
    sys.modules.update({"sentence_transformers": pkg, "sentence_transformers.util": util,
                        "sentence_transformers.models": models})
    out = {}
    for name in ("Pooling", "WeightedMeanPooling", "Dense", "Normalize", "Asym"):
        spec = importlib.util.spec_from_file_location(f"sentence_transformers.models.{name}",
                                                      os.path.join(REF_ST, "models", f"{name}.py"))
        mod = importlib.util.module_from_spec(spec)
        sys.modules[spec.name] = mod
        spec.loader.exec_module(mod)
        out[name] = getattr(mod, name)
        setattr(models, name, out[name])
    return out


def tiny_hf():
    from transformers import GPTNeoConfig, GPTNeoModel

    torch.manual_seed(0)
    cfg = GPTNeoConfig(vocab_size=300, max_position_embeddings=64, hidden_size=128, num_layers=2, num_heads=2,
                       intermediate_size=256, window_size=8, attention_types=[[["global", "local"], 1]],
                       embed_dropout=0.0, attention_dropout=0.0, resid_dropout=0.0, activation_function="gelu_new")
    model = GPTNeoModel(cfg).float().eval()
    with torch.no_grad():  # default init is sigma=0.02: scale up so LayerNorm/attention see non-trivial activations
        for n, p in model.named_parameters():
            if p.dim() == 2 and "wte" not in n and "wpe" not in n:
                p.mul_(4.0)
            if "ln_" in n and n.endswith("bias"):
                p.normal_(0, 0.1)
        # the kernel stores linear weights in bf16: make the fixture weights exactly representable
        for p in model.parameters():
            if p.dim() == 2:
                p.copy_(p.to(torch.bfloat16).float())
    return model


def write_modules_json(path, entries):
    with open(os.path.join(path, "modules.json"), "w") as f:
        json.dump([{"idx": i, "name": str(i), "path": p, "type": t} for i, (p, t) in enumerate(entries)], f, indent=2)


def save_transformer(model, path, max_seq_length):
    model.save_pretrained(path)  # Transformer.save: auto_model.save_pretrained + tokenizer + sentence_bert_config.json
    # the 2-D weights are bf16-exact (tiny_hf): stored as bf16 they keep every value in half the bytes (file < 1 MB)
    from safetensors.torch import load_file, save_file

    st = os.path.join(path, "model.safetensors")
    save_file({k: v.to(torch.bfloat16) if v.dim() == 2 else v for k, v in load_file(st).items()}, st,
              metadata={"format": "pt"})
    with open(os.path.join(path, "sentence_bert_config.json"), "w") as f:
        json.dump({"max_seq_length": max_seq_length, "do_lower_case": False}, f, indent=2)


def main():
    M = reference_models()
    hf = tiny_hf()
    d = hf.config.hidden_size
    g = torch.Generator().manual_seed(7)
    B, S = 6, 24
    lens = torch.tensor([1, S, 5, 17, 24, 9])
    ids = torch.randint(0, 299, (B, S), generator=g)
    mask = (torch.arange(S).unsqueeze(0) < lens.unsqueeze(1)).long()
    ids = torch.where(mask.bool(), ids, torch.full_like(ids, 299))
    with torch.no_grad():
        tok = hf(input_ids=ids, attention_mask=mask).last_hidden_state

    # ---- st_tiny: learnt weighted mean -> Dense(Tanh) -> Normalize ------------------------------------------------
    p1 = os.path.join(HERE, "st_tiny")
    shutil.rmtree(p1, ignore_errors=True)
    os.makedirs(p1)
    save_transformer(hf, p1, max_seq_length=32)
    wmp = M["WeightedMeanPooling"](d, num_positions=40)
    with torch.no_grad():
        wmp.position_weights.copy_(torch.rand(41, generator=g) * 2 + 0.1)
    dense = M["Dense"](d, 48, activation_function=torch.nn.Tanh())
    with torch.no_grad():
        dense.linear.weight.normal_(0, 0.3, generator=g)
        dense.linear.bias.normal_(0, 0.1, generator=g)
    norm = M["Normalize"]()
    for sub, mod in (("1_WeightedMeanPooling", wmp), ("2_Dense", dense), ("3_Normalize", norm)):
        os.makedirs(os.path.join(p1, sub))
        mod.save(os.path.join(p1, sub))
    write_modules_json(p1, [("", "sentence_transformers.models.Transformer"),
                            ("1_WeightedMeanPooling", "sentence_transformers.models.WeightedMeanPooling"),
                            ("2_Dense", "sentence_transformers.models.Dense"),
                            ("3_Normalize", "sentence_transformers.models.Normalize")])
    with torch.no_grad():
        f = wmp({"token_embeddings": tok, "attention_mask": mask})
        pooled_learnt = f["sentence_embedding"].clone()
        f = dense(f)
        dense_out = f["sentence_embedding"].clone()
        full = norm(f)["sentence_embedding"].clone()

    # ---- st_tiny_asym: fixed weighted mean -> Asym{QRY, DOCPOS} -----------------------------------------------------
    p2 = os.path.join(HERE, "st_tiny_asym")
    shutil.rmtree(p2, ignore_errors=True)
    os.makedirs(p2)
    # the Transformer module is shared with st_tiny: modules.json paths are relative to the model directory
    # (SentenceTransformer.py:933 joins them), so "../st_tiny" loads the same files
    pool = M["Pooling"](d, pooling_mode="weightedmean")
    dq = M["Dense"](d, 32, bias=False, activation_function=torch.nn.Identity())
    dd = M["Dense"](d, 32, activation_function=torch.nn.Tanh())
    with torch.no_grad():
        dq.linear.weight.normal_(0, 0.3, generator=g)
        dd.linear.weight.normal_(0, 0.3, generator=g)
        dd.linear.bias.normal_(0, 0.1, generator=g)
    asym = M["Asym"]({"QRY": [dq], "DOCPOS": [dd]})
    for sub, mod in (("1_Pooling", pool), ("2_Asym", asym)):
        os.makedirs(os.path.join(p2, sub))
        mod.save(os.path.join(p2, sub))
    write_modules_json(p2, [("../st_tiny", "sentence_transformers.models.Transformer"),
                            ("1_Pooling", "sentence_transformers.models.Pooling"),
                            ("2_Asym", "sentence_transformers.models.Asym")])
    with torch.no_grad():
        base = pool({"token_embeddings": tok, "attention_mask": mask})["sentence_embedding"].clone()
        q_out = asym({"sentence_embedding": base.clone(), "text_keys": ["QRY"] * B})["sentence_embedding"].clone()
        d_out = asym({"sentence_embedding": base.clone(), "text_keys": ["DOCPOS"] * B})["sentence_embedding"].clone()

    np.savez_compressed(os.path.join(HERE, "st_tiny.npz"), ids=ids.numpy(), mask=mask.numpy(),
                        token_embeddings=tok.numpy(), position_weights=wmp.position_weights.detach().numpy(),
                        pooled_learnt=pooled_learnt.numpy(), dense_out=dense_out.numpy(), full=full.numpy(),
                        pooled_fixed=base.numpy(), asym_qry=q_out.numpy(), asym_doc=d_out.numpy(),
                        dense_w=dense.linear.weight.detach().numpy(), dense_b=dense.linear.bias.detach().numpy())
    for p in (p1, p2):
        size = sum(os.path.getsize(os.path.join(r, f)) for r, _, fs in os.walk(p) for f in fs)
        print(p, f"{size / 1024:.0f} KiB")


if __name__ == "__main__":
    main()
