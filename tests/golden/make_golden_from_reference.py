"""Generates golden vectors from a checkout of the reference project (alibaba/TorchEasyRec @ 54cac316).

The reference package cannot be imported as a whole (torchrec / fbgemm_gpu / pyfg are absent), but
tzrec/modules/fm.py, interaction.py, mlp.py, mmoe.py, task_tower.py and sequence.py are plain PyTorch: they are loaded file by file
through stub parent packages, executed on seeded inputs, and their outputs (and autograd gradients) are
stored as small .npz fixtures.  `configs` stores what this project's config loader makes of every examples/*.config.
The tests read only the fixtures, so they run without the reference checkout.

    python tests/golden/make_golden_from_reference.py <reference checkout> [dense|blocks|configs]
"""
import glob
import gzip
import json
import os
import sys
import types

import numpy as np
import torch

REF = ""     # the reference checkout, set from the command line
HERE = os.path.dirname(os.path.abspath(__file__))


def _stub_packages():
    for name in ["tzrec", "tzrec.modules", "tzrec.utils", "tzrec.models", "tzrec.protos"]:
        m = types.ModuleType(name)
        m.__path__ = [os.path.join(REF, name.replace(".", "/"))]
        sys.modules[name] = m
    # tzrec/modules/sequence.py imports three things that cannot be loaded here: the generated proto module (only used
    # in type annotations), config_util (unused by DINEncoder) and fx_util (imports torchrec) of which it needs
    # fx_arange(len, device) == torch.arange(len, device=device) (tzrec/utils/fx_util.py:50-52)
    pb = types.ModuleType("tzrec.protos.seq_encoder_pb2")
    pb.SeqEncoderConfig = type("SeqEncoderConfig", (), {})
    sys.modules[pb.__name__] = pb
    sys.modules["tzrec.utils.config_util"] = types.ModuleType("tzrec.utils.config_util")
    fx = types.ModuleType("tzrec.utils.fx_util")
    fx.fx_arange = lambda len, device: torch.arange(len, device=device)
    sys.modules[fx.__name__] = fx


def _dump_module(out, tag, mod):
    for k, v in mod.state_dict().items():
        out[f"{tag}_sd__{k}"] = v.numpy()
    for k, p in mod.named_parameters():
        out[f"{tag}_grad__{k}"] = p.grad.numpy()


def model_blocks():
    """DIN attention, MMoE and TaskTower of the reference (tzrec/modules/sequence.py:65-128, mmoe.py:21-77,
    task_tower.py:21-52) at the shapes of cfg4 / cfg5 -> tests/golden/ref_model_blocks.npz."""
    from tzrec.modules.mmoe import MMoE
    from tzrec.modules.sequence import DINEncoder
    from tzrec.modules.task_tower import TaskTower

    torch.manual_seed(20260924)
    out = {}
    # DIN (structure of multi_tower_din_taobao.config: query dim == sequence dim, two-layer attn_mlp; widths reduced
    # to keep the fixture small); lengths incl. 0, 1 and T
    B, T, D = 12, 9, 24
    enc = DINEncoder(sequence_dim=D, query_dim=D, input="seq", attn_mlp={"hidden_units": [48, 16]})
    q = torch.randn(B, D, requires_grad=True)
    seq = torch.randn(B, T, D, requires_grad=True)
    lens = torch.tensor([0, 1, 9, 5, 3, 9, 2, 7, 1, 4, 8, 6])
    y = enc({"seq.query": q, "seq.sequence": seq, "seq.sequence_length": lens})
    dy = torch.randn_like(y)
    y.backward(dy)
    out.update(din_q=q.detach().numpy(), din_seq=seq.detach().numpy(), din_len=lens.numpy(), din_y=y.detach().numpy(),
               din_dy=dy.numpy(), din_dq=q.grad.numpy(), din_dseq=seq.grad.numpy())
    _dump_module(out, "din", enc)
    # DIN with a narrower query (padding branch) and max_seq_length clamp
    enc2 = DINEncoder(sequence_dim=16, query_dim=8, input="s", attn_mlp={"hidden_units": [32]}, max_seq_length=4)
    q2, s2 = torch.randn(5, 8, requires_grad=True), torch.randn(5, 6, 16, requires_grad=True)
    l2 = torch.tensor([6, 0, 4, 2, 5])
    y2 = enc2({"s.query": q2, "s.sequence": s2, "s.sequence_length": l2})
    y2.sum().backward()
    out.update(din2_q=q2.detach().numpy(), din2_seq=s2.detach().numpy(), din2_len=l2.numpy(), din2_y=y2.detach().numpy(),
               din2_dq=q2.grad.numpy(), din2_dseq=s2.grad.numpy())
    _dump_module(out, "din2", enc2)
    # MMoE (structure of mmoe_taobao.config: 3 experts with three-layer MLPs, 2 tasks, no gate_mlp; widths reduced)
    mm = MMoE(in_features=40, expert_mlp={"hidden_units": [64, 32, 16]}, num_expert=3, num_task=2)
    x = torch.randn(10, 40, requires_grad=True)
    ys = mm(x)
    dys = [torch.randn_like(t) for t in ys]
    torch.autograd.backward(ys, dys)
    out.update(mmoe_x=x.detach().numpy(), mmoe_dx=x.grad.numpy())
    for i, (t, d) in enumerate(zip(ys, dys)):
        out[f"mmoe_y{i}"], out[f"mmoe_dy{i}"] = t.detach().numpy(), d.numpy()
    _dump_module(out, "mmoe", mm)
    # TaskTower (three-layer MLP + Linear(., 1) as in mmoe_taobao.config; widths reduced)
    tt = TaskTower(16, 1, mlp={"hidden_units": [32, 16, 8]})
    xt = torch.randn(10, 16, requires_grad=True)
    yt = tt(xt)
    yt.sum().backward()
    out.update(tower_x=xt.detach().numpy(), tower_y=yt.detach().numpy(), tower_dx=xt.grad.numpy())
    _dump_module(out, "tower", tt)
    np.savez_compressed(os.path.join(HERE, "ref_model_blocks.npz"), **out)
    print("wrote", os.path.join(HERE, "ref_model_blocks.npz"), len(out), "arrays")


def main():
    _stub_packages()
    from tzrec.modules.fm import FactorizationMachine  # tzrec/modules/fm.py:16
    from tzrec.modules.interaction import InteractionArch  # tzrec/modules/interaction.py:57
    from tzrec.modules.mlp import MLP  # tzrec/modules/mlp.py:86

    torch.manual_seed(20260923)
    out = {}
    # FM: [B, N, D] (deepfm_criteo: N=26, D=16) + odd shapes
    for tag, (B, N, D) in {"fm_criteo": (64, 26, 16), "fm_small": (5, 3, 4), "fm_wide": (7, 9, 32)}.items():
        x = torch.randn(B, N, D, requires_grad=True)
        y = FactorizationMachine()(x)
        dy = torch.randn_like(y)
        y.backward(dy)
        out[f"{tag}_x"], out[f"{tag}_y"], out[f"{tag}_dy"], out[f"{tag}_dx"] = (
            x.detach().numpy(), y.detach().numpy(), dy.numpy(), x.grad.numpy())
    # InteractionArch: DLRM-Criteo N=27, D=16 and edge shapes (N=2, N not multiple of 4, D=4/64)
    for tag, (B, N, D) in {"ia_criteo": (48, 27, 16), "ia_min": (3, 2, 4), "ia_odd": (9, 13, 8),
                           "ia_wide": (4, 33, 64)}.items():
        x = torch.randn(B, N, D, requires_grad=True)
        z = InteractionArch(N)(x)
        dz = torch.randn_like(z)
        z.backward(dz)
        out[f"{tag}_x"], out[f"{tag}_z"], out[f"{tag}_dz"], out[f"{tag}_dx"] = (
            x.detach().numpy(), z.detach().numpy(), dz.numpy(), x.grad.numpy())
    # DLRM predict glue (tzrec/models/dlrm.py:113-131) re-enacted with the reference modules, forward only
    B, Ns, D = 32, 26, 16
    dense_mlp = MLP(13, [64, 16])
    final_mlp = MLP(351 + 16 + Ns * D, [64, 32])
    head = torch.nn.Linear(32, 1)
    dense_in = torch.rand(B, 13)
    sparse = torch.randn(B, Ns * D)
    with torch.no_grad():
        dense_feat = dense_mlp(dense_in)
        feat = torch.cat([dense_feat.unsqueeze(1), sparse.reshape(-1, Ns, D)], dim=1)
        inter = InteractionArch(Ns + 1)(feat)
        all_feat = torch.cat([inter, dense_feat, sparse], dim=-1)
        logits = head(final_mlp(all_feat)).squeeze(1)
        labels = (torch.rand(B) < 0.25).float()
        loss = torch.nn.functional.binary_cross_entropy_with_logits(logits, labels)
    out["dlrm_dense_in"], out["dlrm_sparse"], out["dlrm_labels"] = dense_in.numpy(), sparse.numpy(), labels.numpy()
    out["dlrm_all_feat"], out["dlrm_logits"], out["dlrm_loss"] = all_feat.numpy(), logits.numpy(), loss.numpy()
    for prefix, mod in [("dense_mlp", dense_mlp), ("final_mlp", final_mlp), ("output_mlp", head)]:
        for k, v in mod.state_dict().items():
            out[f"dlrm_sd__{prefix}.{k}"] = v.numpy()
    np.savez_compressed(os.path.join(HERE, "ref_dense_modules.npz"), **out)
    print("wrote", os.path.join(HERE, "ref_dense_modules.npz"), len(out), "arrays")


def example_configs():
    """Every examples/*.config of the reference as this project's loader parses it (`Message.to_dict()`), keyed by
    file name -> tests/golden/reference_example_configs.json.gz."""
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    from torcheasyrec_b200.config import load_pipeline_config

    out = {os.path.basename(p)[:-len(".config")]: load_pipeline_config(p).to_dict()
           for p in sorted(glob.glob(os.path.join(REF, "examples", "*.config")))}
    path = os.path.join(HERE, "reference_example_configs.json.gz")
    with gzip.GzipFile(path, "wb", mtime=0) as fh:
        fh.write(json.dumps(out, indent=1, sort_keys=True).encode())
    print("wrote", path, len(out), "configs")


if __name__ == "__main__":
    REF = os.path.abspath(sys.argv[1])
    which = sys.argv[2] if len(sys.argv) > 2 else "all"
    if which in ("all", "dense"):
        main()
    if which in ("all", "blocks"):
        _stub_packages()
        model_blocks()
    if which in ("all", "configs"):
        example_configs()
