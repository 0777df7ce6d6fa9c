"""Fused corpus-side encoder (SURVEY section 8 f1): DLDKD.encode_context (method/model.py:215-243) on hand-written kernels.

Per branch the reference runs  LN -> Linear(Dv -> H) -> ReLU -> + position table -> LN -> 4-head self-attention
(additive -10000 key mask) -> dense + residual -> LN -> out_mapping_linear  as ~25 PyTorch / cuBLAS (fp32 SIMT sgemm)
calls.  Here every Linear is one tcgen05 kind::tf32 x 3 GEMM (fp32 grade: ops.linear_exact) and the rest is three small
kernels:

  row_stats(x)                                   LayerNorm statistics of the raw features; the normalised features are
                                                 never written — the projection's A-operand stager applies (scale, shift)
  linear_exact(x, W1', b1', relu, row stats)     LN gamma / beta folded into W1' = W1 diag(gamma), b1' = b1 + W1 beta;
                                                 BOTH branches in one GEMM (N = 2H): the raw features are read once
  layernorm_rows(P_b + pos)                      position table + LN
  linear_exact(X2, [Wq; Wk; Wv])                 fused QKV projection (N = 3H)
  mha_small                                      scores, mask, softmax, weighted sum per (video, head)
  linear_exact(ctx, Wd) ; layernorm_rows(. + X2) dense + residual + LN
  linear_exact(X3, Wo)                           out_mapping_linear
  [linear_exact(out, [Wk'; Wv'])]                key / value projections of the key-clip attention (two-scale head)

Inference only (eval mode: dropout is the identity).  Weights are packed once per model (pack()); call pack() again
after the parameters change."""
import torch

from . import ops

MHA_HEAD_DIMS = (16, 32, 64, 96, 128)   # dkd_mha_small instantiations
MHA_MAX_L = 128                         # dkd_mha_small: frames per video
LN_MAX_D = 512                          # dkd_layernorm_rows: features per row


class FusedContextEncoder:
    def __init__(self, model):
        self.model = model
        self.packed = None

    @staticmethod
    def _branch_modules(model, b):
        if b == 0:
            return (model.visual_input_proj, model.visual_pos_embed, model.visual_encoder, model.out_mapping_linear,
                    model.inher_key_mapping, model.inher_val_mapping)
        return (model.exp_visual_input_proj, model.exp_visual_pos_embed, model.exp_visual_encoder,
                model.exp_out_mapping_linear, model.exp_key_mapping, model.exp_val_mapping)

    @torch.no_grad()
    def pack(self):
        m = self.model
        nb = 2 if m.double_branch else 1
        for b in range(nb):                           # shapes the kernels cannot run are refused before any launch
            att = getattr(self._branch_modules(m, b)[2], "self")
            H = att.heads * att.dh
            if att.dh not in MHA_HEAD_DIMS:
                raise ValueError(f"FusedContextEncoder: head size {att.dh} is not one of the attention kernel's "
                                 f"{MHA_HEAD_DIMS}")
            if H > LN_MAX_D or H % 32:
                raise ValueError(f"FusedContextEncoder: hidden size {H} must be a multiple of 32 (linear layers: "
                                 f"K % 32 == 0) and at most {LN_MAX_D} (LayerNorm kernel)")
        w1, b1, branches = [], [], []
        for b in range(nb):
            proj, pos, enc, outm, km, vm = self._branch_modules(m, b)
            ln, lin = proj.LayerNorm, proj.net[1]
            W = lin.weight.detach().float()
            w1.append(W * ln.weight.detach().float()[None, :])                       # W diag(gamma)
            b1.append(lin.bias.detach().float() + W @ ln.bias.detach().float())     # b + W beta
            att, so = getattr(enc, "self"), enc.output
            wqkv = torch.cat([att.query.weight, att.key.weight, att.value.weight]).detach().float().contiguous()
            bqkv = torch.cat([att.query.bias, att.key.bias, att.value.bias]).detach().float().contiguous()
            wkv = torch.cat([km.weight, vm.weight]).detach().float().contiguous()
            bkv = torch.cat([km.bias, vm.bias]).detach().float().contiguous()
            H = lin.weight.shape[0]
            branches.append(dict(
                H=H, heads=att.heads, dh=att.dh, eps1=ln.eps,
                pos=pos.position_embeddings.weight.detach().float().contiguous(),
                ln2=(pos.LayerNorm.weight.detach().float().contiguous(), pos.LayerNorm.bias.detach().float().contiguous(),
                     pos.LayerNorm.eps),
                wqkv=ops.pack_weight(wqkv), bqkv=bqkv,
                wd=ops.pack_weight(so.dense.weight.detach().float().contiguous()), bd=so.dense.bias.detach().float().contiguous(),
                ln3=(so.LayerNorm.weight.detach().float().contiguous(), so.LayerNorm.bias.detach().float().contiguous(),
                     so.LayerNorm.eps),
                wo=ops.pack_weight(outm.weight.detach().float().contiguous()), bo=outm.bias.detach().float().contiguous(),
                wkv=ops.pack_weight(wkv), bkv=bkv))
        if len({br["H"] for br in branches}) != 1 or len({br["eps1"] for br in branches}) != 1:
            raise ValueError("FusedContextEncoder: the branches must share the hidden size and the input LayerNorm eps")
        W1 = torch.cat(w1)
        Dv = W1.shape[1]
        Kp = ops.round_up(Dv, 32)                     # the GEMM's K is a multiple of 32: zero weight columns are exact
        if Kp != Dv:
            W1 = torch.nn.functional.pad(W1, (0, Kp - Dv))
        self.packed = dict(w1=ops.pack_weight(W1.contiguous()), b1=torch.cat(b1).contiguous(), branches=branches,
                           H=branches[0]["H"], eps1=branches[0]["eps1"], Dv=Dv, Kp=Kp)
        return self

    @torch.no_grad()
    def encode_context(self, frame_video_feat, video_mask=None, want_key_val=False):
        """(B, L, Dv) [+ (B, L) mask] -> (inheritance (B, L, H), exploration (B, L, H) | None)
        [+ per branch (key, val) (B, L, H) pairs of the key-clip attention when want_key_val]."""
        if self.model.training:
            raise RuntimeError("FusedContextEncoder is inference only (eval mode: dropout must be the identity)")
        if self.packed is None:
            self.pack()
        pk = self.packed
        x = frame_video_feat.contiguous().float()
        B, L, Dv = x.shape
        rows = B * L
        x2d = x.view(rows, Dv)
        H = pk["H"]
        m8 = None if video_mask is None else (video_mask > 0).to(torch.uint8).contiguous()
        if Dv != pk["Dv"]:
            raise ValueError(f"encode_context: feature size {Dv} does not match the packed projection ({pk['Dv']})")
        max_l = min([MHA_MAX_L] + [br["pos"].shape[0] for br in pk["branches"]])
        if L > max_l:
            raise ValueError(f"encode_context: {L} frames per video; the position table and the attention kernel "
                             f"hold at most {max_l}")
        ss = ops.row_stats(x2d, pk["eps1"])
        if pk["Kp"] != Dv:
            x2d = torch.nn.functional.pad(x2d, (0, pk["Kp"] - Dv)).contiguous()
        P = ops.linear_exact(x2d, pk["w1"], H * len(pk["branches"]), bias=pk["b1"], relu=True, row_scale_shift=ss)
        outs, kvs = [], []
        for b, br in enumerate(pk["branches"]):
            g2, be2, e2 = br["ln2"]
            X2 = ops.layernorm_rows(P[:, b * H:(b + 1) * H], g2, be2, e2, pos=br["pos"][:L].contiguous(), L=L)
            qkv = ops.linear_exact(X2, br["wqkv"], 3 * H, bias=br["bqkv"])
            ctx = ops.mha_small(qkv, B, L, br["heads"], br["dh"], m8)
            dn = ops.linear_exact(ctx, br["wd"], H, bias=br["bd"])
            g3, be3, e3 = br["ln3"]
            X3 = ops.layernorm_rows(dn, g3, be3, e3, residual=X2)
            out = ops.linear_exact(X3, br["wo"], H, bias=br["bo"])
            outs.append(out.view(B, L, H))
            if want_key_val:
                kv = ops.linear_exact(out, br["wkv"], 2 * H, bias=br["bkv"])
                kvs.append((kv[:, :H].contiguous().view(B, L, H), kv[:, H:].contiguous().view(B, L, H)))
        res = (outs[0], outs[1] if len(outs) > 1 else None)
        return res + (kvs,) if want_key_val else res
