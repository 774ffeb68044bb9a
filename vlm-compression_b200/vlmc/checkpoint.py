"""Pruned-checkpoint wire format and side files of the reference's prune-and-save flow (SURVEY 8f-3).

Mirrors evaluate_old.py:
  remaining_proportion        <- :331-334   sum((param != 0).float().sum()) / original size, one K17 launch per 64 tensors
  save_pruned_model           <- :336-378   the four artefacts a pruning job leaves, same folders and file names:
                                             pruned_checkpoint/V+L/<method>/<job_id>.pth   model.state_dict()
                                             sparsity_dict/<job_id>.yaml                    per-layer sparsities (if a dict)
                                             training_statistics/<job_id>.yaml              {memory (GB), time (s)}
                                             importance_scores/<job_id>.pth                 {param name: importance_score}
  load_pruned_language_model  <- :246-265   t5_model / opt_model / llm_model: keys filtered by prefix, prefix stripped
  load_pruned_vision_model    <- :268-290   "visual." / "visual_encoder." prefix, missing keys keep the current weights
The format is the reference's (dense tensors with explicit zeros): checkpoints written here load in evaluate_old.py and
the other way round.  torch.save / torch.load / yaml are plumbing; the only arithmetic is the non-zero count (K17).

save_compressed_checkpoint / load_compressed_checkpoint write and read a model whose 2:4 linears are compressed
(vlmc.sparse24): {"format": COMPRESSED_FORMAT, "state_dict": ..., "sparse24": {linear name: in_features}}, the linears'
entries being `values` / `meta` / `bias` instead of `weight` / `bias`.
"""
import os
import time

import torch
import torch.nn as nn
import yaml

from vlmc import native
from vlmc.sparse24 import Sparse24Linear

LANGUAGE_PREFIXES = ("t5_model", "opt_model", "llm_model")      # evaluate_old.py:246,253,260 (checked in this order)
VISION_PREFIXES = ("visual.", "visual_encoder.")                 # evaluate_old.py:271
COMPRESSED_FORMAT = "vlmc-sparse24-v1"


def remaining_proportion(model, orig_total_size=None):
    """Percentage of non-zero parameters (evaluate_old.py:331-334): returns (percent, non-zero count, total)."""
    params = [p.data for p in model.parameters()]
    total = sum(p.numel() for p in params) if orig_total_size is None else int(orig_total_size)
    nz = int(native.count_nonzero(params).sum().item())
    return nz / total * 100.0, nz, total


def save_pruned_model(model, job_id, pruning_method, sparsity_dict=None, start_time=None, root="."):
    """evaluate_old.py:336-378.  Returns the paths written, keyed like the folders."""
    out = {}
    folder = os.path.join(root, "pruned_checkpoint/V+L", pruning_method)
    os.makedirs(folder, exist_ok=True)
    out["pruned_checkpoint"] = os.path.join(folder, job_id + ".pth")
    torch.save(model.state_dict(), out["pruned_checkpoint"])
    if sparsity_dict is not None and isinstance(sparsity_dict, dict):
        folder = os.path.join(root, "sparsity_dict")
        os.makedirs(folder, exist_ok=True)
        out["sparsity_dict"] = os.path.join(folder, job_id + ".yaml")
        with open(out["sparsity_dict"], "w") as f:
            yaml.dump(sparsity_dict, f)
    peak_memory = (torch.cuda.max_memory_allocated() / 1024 ** 2) / 1000 if torch.cuda.is_available() else 0.0
    stats = {"memory": peak_memory, "time": (time.time() - start_time) if start_time is not None else 0.0}
    folder = os.path.join(root, "training_statistics")
    os.makedirs(folder, exist_ok=True)
    out["training_statistics"] = os.path.join(folder, job_id + ".yaml")
    with open(out["training_statistics"], "w") as f:
        yaml.dump(stats, f)
    folder = os.path.join(root, "importance_scores")
    os.makedirs(folder, exist_ok=True)
    out["importance_scores"] = os.path.join(folder, job_id + ".pth")
    torch.save({k: v.importance_score for k, v in model.named_parameters()
                if getattr(v, "importance_score", None) is not None}, out["importance_scores"])
    return out


def load_pruned_language_model(model, checkpoint):
    """evaluate_old.py:246-265: the first of t5_model / opt_model / llm_model the model has receives the keys that start
    with its name, with the name stripped.  Returns the attribute name that was loaded (None if the model has none)."""
    for prefix in LANGUAGE_PREFIXES:
        sub = getattr(model, prefix, None)
        if sub is None:
            continue
        state = torch.load(checkpoint, map_location="cpu")
        state = {k: v for k, v in state.items() if k.startswith(prefix)}
        state = {k.replace(prefix + ".", ""): v for k, v in state.items()}
        sub.load_state_dict(state)
        return prefix
    return None


def load_pruned_vision_model(model, checkpoint, interpolate_pos_embed=None):
    """evaluate_old.py:268-290: keys under "visual." or "visual_encoder." replace the matching entries of the current
    visual_encoder state; everything else keeps its value.  interpolate_pos_embed(visual_encoder, state) is the
    reference's EVA position-embedding resize hook (lavis.models.eva_vit), optional here."""
    state = torch.load(checkpoint, map_location="cpu")
    prefix = next((p for p in VISION_PREFIXES if any(k.startswith(p) for k in state)), None)
    assert prefix is not None
    state = {k.replace(prefix, ""): v for k, v in state.items() if k.startswith(prefix)}
    merged = model.visual_encoder.state_dict()
    for k, v in state.items():
        if k in merged:
            merged[k] = v
    if interpolate_pos_embed is not None:
        interpolate_pos_embed(model.visual_encoder, merged)
    model.visual_encoder.load_state_dict(merged)
    return prefix


def save_compressed_checkpoint(model, path):
    """Writes the state of a model whose 2:4 linears are Sparse24Linear (vlmc.sparse24.compress_model) to `path`."""
    layers = {name: mod.in_features for name, mod in model.named_modules() if isinstance(mod, Sparse24Linear)}
    state = {k: v.contiguous() for k, v in model.state_dict().items()}
    torch.save({"format": COMPRESSED_FORMAT, "state_dict": state, "sparse24": layers}, path)


def load_compressed_checkpoint(model, path, dense=False, sparse_mma=False):
    """Loads a file of save_compressed_checkpoint into `model` (dense or already compressed, same architecture).
    dense=False: the compressed linears become Sparse24Linear (nn.Linears at those names are replaced, on their device).
    dense=True: the weights are expanded (K25, +0 at pruned positions) into the model's nn.Linears, which stay dense, so
    the result is an ordinary dense state that the reference's loaders take.  sparse_mma sets the routing flag of every
    Sparse24Linear loaded (vlmc.sparse24); the file format does not depend on it.  Returns the compressed linears'
    names."""
    ckpt = torch.load(path, map_location="cpu")
    if not isinstance(ckpt, dict) or ckpt.get("format") != COMPRESSED_FORMAT:
        raise ValueError(f"{path} is not a {COMPRESSED_FORMAT} checkpoint")
    state, layers = dict(ckpt["state_dict"]), ckpt["sparse24"]
    for name, C in layers.items():
        mod = model.get_submodule(name)
        values, meta = state.pop(name + ".values"), state.pop(name + ".meta")
        bias = state.get(name + ".bias")
        ref = mod.weight if isinstance(mod, nn.Linear) else mod.values
        dev = ref.device if ref.is_cuda else torch.device("cuda")
        if dense:
            if not isinstance(mod, nn.Linear):
                raise TypeError(f"dense=True needs an nn.Linear at {name}, found {type(mod).__name__}")
            state[name + ".weight"] = native.sparse24_decompress(values.to(dev), meta.to(dev), C)
            continue
        if isinstance(mod, nn.Linear):
            new = Sparse24Linear(values.to(dev), meta.to(dev), C, None if bias is None else bias.to(dev), sparse_mma)
            parent_name, _, child = name.rpartition(".")
            setattr(model.get_submodule(parent_name) if parent_name else model, child, new)
        else:
            mod.sparse_mma = bool(sparse_mma)
        state[name + ".values"], state[name + ".meta"] = values, meta
    model.load_state_dict(state)
    return list(layers)
