"""Drop-in mirror of the reference model's entry points for the retrieval scoring path.

Mirrors `DLDKD` of the reference (method/model.py:13): same constructor arguments, same parameter
names (a reference checkpoint's state_dict loads with strict=False; only the key-clip attention
projections are new), same method names and argument meaning:

    encode_context(frame_video_feat, video_mask=None)       method/model.py:215-227
    encode_query(query_feat, query_mask)                    method/model.py:199-211
    get_sim_scores(query, context_feat, mask=None)          method/model.py:307-329  (CUDA kernels)
    get_pred_from_raw_query(...)                            two-scale head, SURVEY §8 N6 (CUDA kernels)
    key_clip_guided_attention[_in_inference](...)           SURVEY §8 N4 (CUDA kernels)

The encoders stay PyTorch (SURVEY §8 R1/R2: query independent or <1% of eval); everything from the
encoded vectors onward runs in the hand-written kernels behind include/dkd_b200.h.  The retrieval
kernels are inference only; the training step (forward(batch), method/model.py:100-162) goes through
train.py, whose similarity and KL kernels have hand-written backward passes.
"""
import math

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import engine, ops


class PositionalEncoding(nn.Module):
    """Learned position table added to the features, then LayerNorm (+dropout).
    Parameter names follow the reference's TrainablePositionalEncoding (method/model_components.py:269)."""

    def __init__(self, max_position_embeddings, hidden_size, dropout=0.1):
        super().__init__()
        self.position_embeddings = nn.Embedding(max_position_embeddings, hidden_size)
        self.LayerNorm = nn.LayerNorm(hidden_size)
        self.dropout = nn.Dropout(dropout)

    def forward(self, x):
        L = x.shape[1]
        pos = self.position_embeddings.weight[:L].unsqueeze(0)
        return self.dropout(self.LayerNorm(x + pos))


class InputProjection(nn.Module):
    """LayerNorm -> dropout -> Linear -> ReLU (reference LinearLayer, method/model_components.py:294)."""

    def __init__(self, in_hsz, out_hsz, dropout=0.1):
        super().__init__()
        self.LayerNorm = nn.LayerNorm(in_hsz)
        self.net = nn.Sequential(nn.Dropout(dropout), nn.Linear(in_hsz, out_hsz))

    def forward(self, x):
        return F.relu(self.net(self.LayerNorm(x)))


class _SelfAttention(nn.Module):
    def __init__(self, hidden, heads, dropout):
        super().__init__()
        if hidden % heads:
            raise ValueError(f"hidden size {hidden} is not a multiple of the number of heads {heads}")
        self.heads, self.dh = heads, hidden // heads
        self.query = nn.Linear(hidden, hidden)
        self.key = nn.Linear(hidden, hidden)
        self.value = nn.Linear(hidden, hidden)
        self.dropout = nn.Dropout(dropout)

    def forward(self, x, mask):
        N, L, _ = x.shape
        split = lambda t: t.view(N, L, self.heads, self.dh).transpose(1, 2)  # noqa: E731
        q, k, v = split(self.query(x)), split(self.key(x)), split(self.value(x))
        att = q @ k.transpose(-1, -2) / math.sqrt(self.dh)
        if mask is not None:  # additive -10000 on masked keys (method/model_components.py:420-422)
            att = att + (1 - mask.unsqueeze(1)) * -10000.0
        att = self.dropout(torch.softmax(att, dim=-1))
        return (att @ v).transpose(1, 2).reshape(N, L, self.heads * self.dh)


class _SelfOutput(nn.Module):
    def __init__(self, hidden, dropout):
        super().__init__()
        self.dense = nn.Linear(hidden, hidden)
        self.LayerNorm = nn.LayerNorm(hidden)
        self.dropout = nn.Dropout(dropout)

    def forward(self, h, residual):
        return self.LayerNorm(self.dropout(self.dense(h)) + residual)


class AttentionBlock(nn.Module):
    """One post-LN self-attention block (reference BertAttention, method/model_components.py:339);
    sub-module names `self` / `output` keep checkpoint compatibility."""

    def __init__(self, hidden, heads, dropout):
        super().__init__()
        setattr(self, "self", _SelfAttention(hidden, heads, dropout))
        self.output = _SelfOutput(hidden, dropout)

    def forward(self, x, mask=None):
        return self.output(getattr(self, "self")(x, mask), x)


def _cfg(config, key, default=None):
    try:
        return getattr(config, key)
    except AttributeError:
        if isinstance(config, dict) and key in config:
            return config[key]
        return default


class DLDKD(nn.Module):
    """Two-branch (inheritance / exploration) DL-DKD++ model, retrieval entry points only."""

    def __init__(self, config, opt):
        super().__init__()
        self.config = config
        self.double_branch = bool(_cfg(opt, "double_branch", True))
        H, E = config.inheritance_hidden, config.exploration_hidden
        drop, idrop, heads = config.drop, config.input_drop, config.n_heads
        self.map_size = int(_cfg(config, "map_size", ops.T_CLIPS))
        self.clip_scale_w = float(_cfg(config, "clip_scale_w", 0.7))
        self.frame_scale_w = float(_cfg(config, "frame_scale_w", 0.3))

        self.query_pos_embed = PositionalEncoding(config.max_desc_l, H, idrop)
        self.query_input_proj = InputProjection(config.query_input_size, H, idrop)
        self.query_encoder = AttentionBlock(H, heads, drop)
        self.modular_vector_mapping = nn.Linear(H, 1, bias=False)
        self.visual_pos_embed = PositionalEncoding(config.max_ctx_l, H, idrop)
        self.visual_input_proj = InputProjection(config.visual_input_size, H, idrop)
        self.visual_encoder = AttentionBlock(H, heads, drop)
        self.out_mapping_linear = nn.Linear(H, H)
        # key-clip-guided attention projections (two-scale head; not in the reference checkpoint)
        self.inher_key_mapping = nn.Linear(H, H)
        self.inher_val_mapping = nn.Linear(H, H)
        if self.double_branch:
            self.exp_query_pos_embed = PositionalEncoding(config.max_desc_l, E, idrop)
            self.exp_query_input_proj = InputProjection(config.query_input_size, E, idrop)
            self.exp_query_encoder = AttentionBlock(E, heads, drop)
            self.exp_modular_vector_mapping = nn.Linear(E, 1, bias=False)
            self.exp_visual_pos_embed = PositionalEncoding(config.max_ctx_l, E, idrop)
            self.exp_visual_input_proj = InputProjection(config.visual_input_size, E, idrop)
            self.exp_visual_encoder = AttentionBlock(E, heads, drop)
            self.exp_out_mapping_linear = nn.Linear(E, E)
            self.exp_key_mapping = nn.Linear(E, E)
            self.exp_val_mapping = nn.Linear(E, E)
        # loss weights read by forward() (method/model.py:67-75)
        self.weight = 1
        self.kl_intra_weight = _cfg(opt, "kl_intra_weight", 0.1)
        self.inher_nce_weight = _cfg(opt, "inher_nce_weight", 0.04)
        self.explore_nce_weight = _cfg(opt, "explore_nce_weight", 0.04)
        self.collection = _cfg(opt, "collection", None)
        self.alpha = _cfg(opt, "alpha", 0.8)
        self.belta = _cfg(opt, "belta", 0.8)
        self.reset_parameters()

    def set_hard_negative(self, use_hard_negative, hard_pool_size):
        """method/model.py:95-98."""
        self.config.use_hard_negative = use_hard_negative
        self.config.hard_pool_size = hard_pool_size

    def forward(self, batch):
        """Training step losses (method/model.py:100-162): same batch keys, returns (loss, dict of terms).
        Similarity forward/backward and the KL term run in the kernels of csrc/dkd_train.cu (train.py)."""
        from . import train
        return train.forward_losses(self, batch)

    def reset_parameters(self):
        """N(0, initializer_range) linears/embeddings, LayerNorm = (1, 0), zero biases (method/model.py:80-93)."""
        std = self.config.initializer_range
        for m in self.modules():
            if isinstance(m, (nn.Linear, nn.Embedding)):
                m.weight.data.normal_(mean=0.0, std=std)
            elif isinstance(m, nn.LayerNorm):
                m.bias.data.zero_()
                m.weight.data.fill_(1.0)
            if isinstance(m, nn.Linear) and m.bias is not None:
                m.bias.data.zero_()

    # ------------------------------------------------------------------ encoders (PyTorch)
    @staticmethod
    def encode_input(feat, mask, input_proj_layer, encoder_layer, pos_embed_layer):
        """method/model.py:229-243."""
        x = pos_embed_layer(input_proj_layer(feat))
        return encoder_layer(x, None if mask is None else mask.unsqueeze(1))

    def enable_fused_encoder(self, on=True):
        """Route encode_context (eval mode, CUDA, no autograd) through the hand-written encoder kernels
        (encoder.FusedContextEncoder: tcgen05 kind::tf32 x 3 linears, fused LayerNorm / attention kernels).  Call again
        after the parameters change (the weights are packed once)."""
        from .encoder import FusedContextEncoder
        self._fused_encoder = FusedContextEncoder(self).pack() if on else None
        return self

    def encode_context(self, frame_video_feat, video_mask=None):
        """(B, L, Dv) [+ (B, L) mask] -> (inheritance (B, L, H), exploration (B, L, E) | None)."""
        fe = getattr(self, "_fused_encoder", None)
        if fe is not None and not self.training and frame_video_feat.is_cuda and not torch.is_grad_enabled():
            return fe.encode_context(frame_video_feat, video_mask)
        inher = self.out_mapping_linear(self.encode_input(
            frame_video_feat, video_mask, self.visual_input_proj, self.visual_encoder, self.visual_pos_embed))
        if not self.double_branch:
            return inher, None
        expl = self.exp_out_mapping_linear(self.encode_input(
            frame_video_feat, video_mask, self.exp_visual_input_proj, self.exp_visual_encoder,
            self.exp_visual_pos_embed))
        return inher, expl

    def get_modularized_queries(self, encoded_query, query_mask, inheritance=False):
        """Softmax-pooled query vector (method/model.py:245-258).  Always returns (N, D) — the reference's
        bare .squeeze() additionally drops the batch dimension when N == 1."""
        proj = self.modular_vector_mapping if inheritance else self.exp_modular_vector_mapping
        logits = proj(encoded_query)
        m = query_mask.unsqueeze(2)
        att = torch.softmax(logits * m + (1 - m) * -1e10, dim=1)
        return torch.einsum("blm,bld->bmd", att, encoded_query).squeeze(1)

    def encode_query(self, query_feat, query_mask):
        """(M, Lq, Dq), (M, Lq) -> (inheritance (M, H), exploration (M, E) | None)."""
        q = self.encode_input(query_feat, query_mask, self.query_input_proj, self.query_encoder, self.query_pos_embed)
        inher = self.get_modularized_queries(q, query_mask, True)
        if not self.double_branch:
            return inher, None
        q = self.encode_input(query_feat, query_mask, self.exp_query_input_proj, self.exp_query_encoder,
                              self.exp_query_pos_embed)
        return inher, self.get_modularized_queries(q, query_mask)

    # ------------------------------------------------------------------ scoring (CUDA kernels)
    @staticmethod
    def get_sim_scores(modularied_query, context_feat, mask=None, want_rows=True):
        """Cosine max-over-frames scores (method/model.py:307-329) on the exact fp32-grade kernels.
        Returns (scores (M, N), per_frame (M, L, N) | None).

        want_rows=True reproduces the reference's second return value (the SIMT kernel writes the (M, L, N) tensor);
        want_rows=False skips it and runs the tcgen05 kind::tf32 x 3 kernel (dkd_score_max_exact).
        INFERENCE ONLY: the kernels build no autograd graph, so a call that would need gradients raises instead of
        silently returning constants — the training step goes through DLDKD.forward (train.py)."""
        if torch.is_grad_enabled() and (modularied_query.requires_grad or context_feat.requires_grad):
            raise RuntimeError("DLDKD.get_sim_scores runs inference-only CUDA kernels (no autograd graph); call it under "
                               "torch.no_grad(), or use DLDKD.forward / train.in_batch_similarity for the training step")
        q = modularied_query.contiguous().float()
        ctx = context_feat.contiguous().float()
        N, L, D = ctx.shape
        qn, _ = ops.normalize_rows(q)
        xn, _ = ops.normalize_rows(ctx)
        m8 = None if mask is None else (mask > 0).to(torch.uint8).contiguous()
        if not want_rows and D % 32 == 0 and D <= 512 and L <= 128:
            s, _ = ops.score_max_exact(qn, ops.pack_rows(xn.view(N, L, D)), L, m8)
            return s, None
        s, _, rows = ops.score_max_f32(qn, xn.view(N, L, D), m8, want_rows=want_rows)
        return s, rows

    def attention_params(self):
        ps = [(self.inher_key_mapping.weight, self.inher_key_mapping.bias,
               self.inher_val_mapping.weight, self.inher_val_mapping.bias)]
        if self.double_branch:
            ps.append((self.exp_key_mapping.weight, self.exp_key_mapping.bias,
                       self.exp_val_mapping.weight, self.exp_val_mapping.bias))
        return ps

    def prepare_context(self, inher_frame_feat, explore_frame_feat, video_mask, heads=("frame", "two_scale"),
                        precisions=("exact", "bf16"), id_base=0):
        """Build the HBM-resident prepared corpus (engine.PreparedCorpus) from encode_context outputs."""
        frames = [inher_frame_feat] + ([explore_frame_feat] if self.double_branch else [])
        return engine.prepare_corpus(frames, video_mask, self.attention_params() if "two_scale" in heads else None,
                                     T=self.map_size, heads=heads, precisions=precisions, id_base=id_base)

    def get_pred_from_raw_query(self, query_feat, query_mask, query_labels=None, video_proposal_feat=None,
                                video_feat=None, video_feat_mask=None, precision="exact", return_fused=False,
                                return_key_clip=False):
        """Two-scale prediction for raw query features against a prepared corpus (SURVEY §8 N6).

        video_proposal_feat: the engine.PreparedCorpus from prepare_context (it owns the clip proposals,
        the frame features and their mask, so video_feat / video_feat_mask are accepted for signature
        compatibility and ignored).  Returns (clip_scale_scores, frame_scale_scores): (M, Nv) tensors for
        a single-branch model, (inheritance, exploration) pairs for the double-branch model; with
        return_fused also the 0.7/0.3-fused branch-weighted score; with return_key_clip also the key clips
        ((M, Nv) int32 proposal indices, same per-branch form), last.
        """
        if not isinstance(video_proposal_feat, engine.PreparedCorpus):
            raise TypeError("video_proposal_feat must be the PreparedCorpus returned by prepare_context")
        qi, qe = self.encode_query(query_feat, query_mask)
        pq = engine.prepare_queries([qi] + ([qe] if self.double_branch else []), want_bf16=precision == "bf16")
        fused, per = engine.score_two_scale_head(video_proposal_feat, pq, precision, self.clip_scale_w,
                                                 self.frame_scale_w, want_frame=True)
        clip = tuple(p["clip"] for p in per)
        frame = tuple(p["frame"] for p in per)
        key_clip = tuple(p["key_clip"] for p in per)
        if not self.double_branch:
            clip, frame, key_clip = clip[0], frame[0], key_clip[0]
        out = (clip, frame, fused) if return_fused else (clip, frame)
        return out + (key_clip,) if return_key_clip else out

    def _attn_table(self, frame_feat, feat_mask, branch):
        kw, kb, vw, vb = self.attention_params()[branch]
        fr = frame_feat.contiguous().float()
        lengths = (feat_mask > 0).sum(dim=1).to(torch.int32).contiguous()
        clips = ops.downsample_clips(fr, lengths, self.map_size)
        tf, _ = ops.frame_attn_table(F.linear(fr, kw, kb).contiguous(), F.linear(fr, vw, vb).contiguous(), clips,
                                     lengths, want_f32=True, want_f16=False)
        return tf

    def key_clip_guided_attention_in_inference(self, frame_feat, proposal_feat, feat_mask, max_index, branch=0):
        """All (query, video) pairs: L2-normalised attention output g[m, n] guided by proposal max_index[m, n]
        (SURVEY §8 N4).  proposal_feat is accepted for signature compatibility (proposals are rebuilt from
        frame_feat on the device).  Returns (M, Nv, D) — small problems only; the hot path never
        materialises this tensor (engine.score_two_scale_head gathers inside the kernel)."""
        tf = self._attn_table(frame_feat, feat_mask, branch)
        idx = max_index.long().clamp_(0, tf.shape[1] - 1)                       # (M, Nv)
        n = torch.arange(tf.shape[0], device=tf.device).unsqueeze(0).expand_as(idx)
        return tf[n, idx]

    def key_clip_guided_attention(self, frame_feat, proposal_feat, feat_mask, max_index, query_labels, branch=0):
        """Training-style call: query m attends only to its own video query_labels[m]; max_index (M,).
        Returns (M, D) L2-normalised attention outputs."""
        tf = self._attn_table(frame_feat, feat_mask, branch)
        labels = torch.as_tensor(query_labels, device=tf.device).long()
        return tf[labels, max_index.long().to(tf.device).clamp_(0, tf.shape[1] - 1)]
