"""
Step engine: owns the HBM workspaces of one (batch, length) shape and issues the kernel sequence of the
ECG-ViT forward / backward / clip+AdamW through the C ABI (include/ecgvit_b200.h).

Data layout in HBM (T = bf16 in performance mode, fp32 in parity mode; M = B * (n_patch + 1) token rows):
  parameters / gradients / AdamW moments : three flat fp32 buffers, tensors at 256-byte aligned offsets
  weight shadow                          : flat bf16 copy of the parameters (GEMM operands), written by AdamW
  a_patch  [B*n_patch, P*C]  T           : gathered patches, time-major / lead-minor features
  per layer: x_in [M,d], ln1 [M,d], qkv [M,3*inner], lse [B,H,N] f32, o [M,inner], y [M,d], ln2 [M,d],
             u [M,mlp] (pre-GELU), h [M,mlp] (post-GELU), row statistics (mean, rstd) f32.  x_in / y are fp32 when the
             residual stream is fp32 (config.residual_dtype; models deeper than 12 layers).  With
             config.activation_checkpointing only x_in is kept per layer; two rotating sets hold the rest and backward
             re-runs the block forward (same dropout masks: they are functions of the step's seed)
  backward scratch, double-buffered by layer parity (the weight-gradient GEMMs of layer l read it on the side stream while
             the main stream already writes layer l-1's): dz[2], dy[2] [M,d], dln [M,d], d_o [M,inner], dqkv[2]
             [M,3*inner], du[2] [M,mlp], dzm[site][2] [M,d] (dropout-masked LayerNorm gradients)
Everything is row-major with the feature dimension contiguous, so every GEMM operand is either K-major or
MN-major for TMA without a transposed copy.

Reference semantics: forward = vit_pytorch.ViT.forward via ecg_vit.py:140-149; backward = autograd of it
(train.py:280); optimizer = train.py:281-282.
"""
import ctypes
import os

import torch

from . import _lib
from .config import drop_path_rates
from ._lib import (GemmArgs, F32, BF16, EPI_STORE, EPI_BIAS_RES, EPI_BIAS_GELU, EPI_DGELU, EPI_ATOMIC_F32,
                   EPI_BIAS_RES_F32, EPI_BIAS_SUB_ROWSQ)

LN_EPS = 1e-5  # nn.LayerNorm default


class _Workspace:
    pass


class StepEngine:
    def __init__(self, model):
        self.model = model
        self.lib = _lib.load()
        self.ws = {}
        self._cur = None
        # device scalar holding this step's dropout seed (refreshed by the host before every training forward)
        self.device = model._flat_p.device
        self._lw_key = self._lw_table = None
        self._spans = {}
        self.rng = torch.zeros(2, device=self.device, dtype=torch.int32)
        # Weight-gradient GEMMs do not feed the backward chain: issued on a side stream they become a parallel branch of
        # the step graph and fill the SMs that the chain's kernels leave idle (partial last waves, launch ramps,
        # memory-bound kernels).  ECGVIT_WGRAD_STREAM=0 keeps everything on one stream.
        self.side_stream = torch.cuda.Stream(device=model._flat_p.device) \
            if os.environ.get('ECGVIT_WGRAD_STREAM', '1') != '0' else None
        self._seed_counter = 0
        self._seed_ring = None
        self.base_seed = 0x5EED     # rank-independent (saved in trainer state); replicas add `rank_offset`
        self.rank_offset = 0
        self._fwd_id = 0            # generation of the last forward (the autograd bridge checks it at backward)
        self.last_seed = None       # (seed, counter) uploaded last

    def new_dropout_seed(self, seed=None):
        """draw the seed of the next training forward (its backward regenerates the same masks from it)"""
        self._seed_counter += 1
        if seed is None:
            seed = ((self.base_seed + self.rank_offset) * 0x9E3779B1 + self._seed_counter * 0x85EBCA6B) & 0x7FFFFFFF
        self.upload_seed(seed, self._seed_counter & 0x7FFFFFFF)
        return seed

    def upload_seed(self, seed, counter):
        if self._seed_ring is None:
            self._seed_ring = _lib.PinnedRing(2, torch.int32)
        self._seed_ring.upload(self.rng, [seed, counter])  # asynchronous: no host stall
        self.last_seed = (seed, counter)

    def _dropout_probs(self):
        """(p_embedding, p_block) as the reference wires them (ecg_vit.py:113-114); zero in eval mode"""
        m = self.model
        if not m.training:
            return 0.0, 0.0
        return float(m.config.attention_probs_dropout_prob), float(m.config.hidden_dropout_prob)

    def _drop_path_rates(self):
        """per-block drop-path rates of the encoder (config.drop_path_rate); zero in eval mode"""
        m = self.model
        depth = m.config.num_hidden_layers
        return drop_path_rates(m.config) if m.training else [0.0] * depth

    # ---- helpers ---------------------------------------------------------------------------------
    @property
    def _stream(self):
        return torch.cuda.current_stream().cuda_stream

    def _gemm(self, M, N, K, A, lda, a_k, B, ldb, b_k, epi, out, ldo, out2=None, aux=None, bias=None, split_k=1,
              drop=None, path=None):
        """path: (rate, site, rows per record) of a drop-path residual epilogue, or None"""
        p, stream = drop if drop is not None else (0.0, 0)
        r = path[0] if path is not None else 0.0
        g = GemmArgs(M, N, K, A.data_ptr(), lda, a_k, B.data_ptr(), ldb, b_k, epi, out.data_ptr(), ldo,
                     _lib.ptr(out2), _lib.ptr(aux), _lib.ptr(bias), self.model._dtype_code, split_k,
                     stream, p, self.rng.data_ptr() if p > 0 or r > 0 else None)
        if _lib.profile[0] is not None:
            keep = GemmArgs.from_buffer_copy(g)  # lets bench.py re-launch exactly this call when timing the kernel
            _lib.profile_meta[0] = (M, N, K, epi, a_k, b_k, keep)
        if r > 0:
            _lib.check(self.lib.ecgvit_gemm_drop_path(ctypes.byref(g), r, path[1], path[2], self._stream), 'gemm')
        else:
            _lib.check(self.lib.ecgvit_gemm(ctypes.byref(g), self._stream), 'gemm')

    def workspace(self, B, L, n_vis=None):
        """activations of one (batch, length) shape; n_vis: the patches the encoder sees per record (all when None)"""
        key = (B, L, n_vis)
        w = self.ws.get(key)
        if w is not None:
            return w
        m = self.model
        c = m.config
        dev = m._flat_p.device
        T = m._act_dtype
        P, C, d, mlp = c.patch_size, c.num_channels, c.hidden_size, c.intermediate_size
        H = c.num_attention_heads
        assert L % P == 0, f'signal length {L} must be a multiple of patch_size {P}'
        per_lead = bool(getattr(c, 'per_lead_tokens', False))
        n = L // P * (C if per_lead else 1)
        K = P if per_lead else P * C            # features of one patch
        Kp = (K + 7) // 8 * 8 if per_lead else K  # row length of the patch matrix (16-byte aligned rows for TMA)
        assert n + 1 <= m.vit.pos_embedding.shape[1], \
            f'{n} patches exceed the positional table ({m.vit.pos_embedding.shape[1] - 1})'
        nv = n if n_vis is None else n_vis
        N = nv + 1
        M = B * N
        depth = c.num_hidden_layers
        w = _Workspace()
        w.B, w.L, w.n, w.N, w.M = B, L, n, N, M
        w.n_vis = nv
        w.per_lead, w.K, w.Kp = per_lead, K, Kp

        def buf(*shape, dtype=T):
            return torch.empty(*shape, device=dev, dtype=dtype)

        w.a_patch = buf(B * n, Kp)
        w.a_emb = w.a_patch    # the embedding GEMM's operand: the rows of the patches the encoder sees
        # per-lead tokens with P % 8 != 0: zero-padded copies of the embedding weight and of its gradient
        w.embed_wpad = buf(d, Kp) if Kp != K else None
        w.embed_gpad = buf(d, Kp, dtype=torch.float32) if Kp != K else None
        w.e = buf(B * nv, d)
        # Activation checkpointing (config.activation_checkpointing; BASELINE.json configs[4]): only the block inputs x[l]
        # are kept per layer; everything inside a block lives in TWO buffer sets used alternately (layer l -> set l % 2)
        # and is recomputed from x[l] in backward.  Two sets, so that the weight-gradient GEMMs of layer l (side stream)
        # can still read their operands while layer l - 1 is being recomputed into the other set.
        ckpt = bool(getattr(c, 'activation_checkpointing', False)) and depth > 2
        self._alloc_stack(w, 'l', B, N, d, mlp, H, depth, ckpt)
        # head
        n_class = m.num_class
        w.xn = buf(B, d, dtype=torch.float32)
        w.hstat = buf(2, B, dtype=torch.float32)
        w.logits = buf(B, n_class, dtype=torch.float32)
        w.loss = buf(1, dtype=torch.float32)
        w.loss_none = buf(B, n_class, dtype=torch.float32)
        w.head_scratch = buf(B * d + B * n_class, dtype=torch.float32)
        w.labels = buf(B, n_class, dtype=torch.float32)
        # pool='mean': the pooled rows and their gradient, fp32 [B, d] (the head kernels read them as N = 1 tokens)
        w.pooled = buf(B, d, dtype=torch.float32) if m._mean_pool else None
        w.dpool = buf(B, d, dtype=torch.float32) if m._mean_pool else None
        w.de = buf(B * nv, d)
        self.ws[key] = w
        return w

    def _alloc_stack(self, s, prefix, B, N, d, mlp, H, depth, ckpt):
        """a block stack on the object s: `depth` blocks of width d over B sequences of N tokens, parameters keyed
        `{prefix}{l}.`, its dims, activations and backward scratch.  Only the encoder stack (prefix 'l') calls the layer
        hooks; p_blk is its block dropout probability and r_path its per-block drop-path rates, both set by the forward
        pass (the encoder's; a decoder keeps zeros).  Drop-path site of branch j (0 attention, 1 feed-forward) of block l:
        path_site + 2 * l + j, after the dropout sites 0 .. 4 * depth and the mask site 4 * depth + 1."""
        m = self.model
        dev = m._flat_p.device
        T = m._act_dtype
        M = B * N
        inner = d  # dim_head = d // heads (ecg_vit.py:100)
        s.prefix, s.d, s.mlp, s.H, s.depth, s.ckpt, s.hooks = prefix, d, mlp, H, depth, ckpt, prefix == 'l'
        s.B, s.N, s.M = B, N, M
        s.p_blk = 0.0
        s.r_path = [0.0] * depth
        s.path_site = 4 * depth + 2

        def buf(*shape, dtype=T):
            return torch.empty(*shape, device=dev, dtype=dtype)

        RT = m._res_dtype  # residual stream: fp32 for deep models in bf16 mode (config.residual_dtype)
        s.x = [buf(M, d, dtype=RT) for _ in range(depth + 1)]  # x[l] = input of block l; x[depth] = stack output
        n_sets = 2 if ckpt else depth

        def per_layer(make):
            sets = [make() for _ in range(n_sets)]
            return [sets[l % n_sets] for l in range(depth)]

        s.ln1 = per_layer(lambda: buf(M, d))
        s.ln2 = per_layer(lambda: buf(M, d))
        s.stat1 = per_layer(lambda: buf(2, M, dtype=torch.float32))
        s.stat2 = per_layer(lambda: buf(2, M, dtype=torch.float32))
        s.qkv = per_layer(lambda: buf(M, 3 * inner))
        s.lse = per_layer(lambda: buf(B, H, N, dtype=torch.float32))
        s.o = per_layer(lambda: buf(M, inner))
        s.y = per_layer(lambda: buf(M, d, dtype=RT))
        s.u = per_layer(lambda: buf(M, mlp))
        s.h = per_layer(lambda: buf(M, mlp))
        # backward scratch
        # Every scratch buffer that a side-stream weight-gradient GEMM reads exists TWICE, indexed by layer parity: the main
        # chain of layer l - 1 then never has to wait for the weight gradients of layer l (it waits for those of layer
        # l + 1, a whole layer old), so the side stream is free to lag and fill whatever the chain leaves idle
        s.dz = [buf(M, d), buf(M, d)]          # gradient w.r.t. a block's output (input of its backward)
        s.dy = [buf(M, d), buf(M, d)]          # gradient w.r.t. the block's middle residual sum y
        s.dln = buf(M, d)
        s.d_o = buf(M, inner)
        s.dqkv = [buf(M, 3 * inner), buf(M, 3 * inner)]
        s.du = [buf(M, mlp), buf(M, mlp)]
        # dropout-masked copies of the residual-stream gradients (only used when p > 0): one per site of a block
        s.dzm = [[buf(M, d), buf(M, d)], [buf(M, d), buf(M, d)]]   # [site 0 = after net[3], 1 = after to_out][parity]
        # two partial-row scratch buffers (one per LayerNorm of a block): their fold runs off the critical chain
        s.ln_scratch = [buf(int(self.lib.ecgvit_layernorm_bwd_scratch_floats(d)), dtype=torch.float32) for _ in range(2)]
        n_attn = int(self.lib.ecgvit_attention_bwd_scratch_floats(B, N, H, d // H, m._dtype_code))
        s.attn_scratch = buf(n_attn, dtype=torch.float32) if n_attn > 0 else None

    # ---- forward ---------------------------------------------------------------------------------
    def forward(self, sample_values, labels=None, reduction='mean', record_attention=False):
        """sample_values: fp32 cuda [B, C, L]; returns (loss | None, logits) as views of workspace buffers.
        record_attention: also materialise every layer's softmax probabilities (slow path for `Recorder`); they are
        left in `self.recorded_attention`, fp32 [B, layers, heads, N, N]."""
        m, lib, st = self.model, self.lib, self._stream
        c = m.config
        dt = m._dtype_code
        rdt = m._res_code                                        # dtype code of calls whose operand is the residual stream
        epi_res = EPI_BIAS_RES_F32 if m._res_f32 else EPI_BIAS_RES
        x = sample_values
        assert x.is_cuda and x.dtype == torch.float32 and x.dim() == 3, 'sample_values must be fp32 cuda [B, C, L]'
        assert x.shape[1] == c.num_channels
        if x.stride(2) != 1 or x.stride(0) != x.shape[1] * x.stride(1):
            x = x.contiguous()
        B, C, L_in = x.shape
        pipe = m.input_pipeline
        L = L_in if pipe is None else pipe.padded_length(L_in)  # TimeEndPad happens inside the gather
        w = self.workspace(B, L)
        self._cur = w
        self._fwd_id += 1
        w.fwd_id = self._fwd_id   # a later forward through the same workspace invalidates this one's backward
        P, d, mlp, H = c.patch_size, c.hidden_size, c.intermediate_size, c.num_attention_heads
        inner, dh = d, d // H
        n, N, M = w.n, w.N, w.M
        wt = m._weights()  # GEMM operand views (bf16 shadow or fp32 master)
        pf = m._params_f32()  # fp32 master views (biases, LayerNorm, cls, pos, head)

        mean = std = spans = None
        if pipe is not None:
            # raw records in: Normalize -> TimeEndPad -> TimeOut (training only) fused into the gather
            mean, std = pipe.device_stats(x.device)
            spans = self.span_buffer(B) if (pipe.timeout is not None and m.training) else None
        K, Kp = w.K, w.Kp
        if w.per_lead:
            _lib.check(lib.ecgvit_patchify_leads(x.data_ptr(), _lib.ptr(mean), _lib.ptr(std), _lib.ptr(spans),
                                                 w.a_patch.data_ptr(), B, C, x.stride(1), L_in, L // P, P, Kp, dt, st),
                       'patchify_leads')
        elif pipe is None:
            _lib.check(lib.ecgvit_patchify(x.data_ptr(), w.a_patch.data_ptr(), B, C, x.stride(1), n, P, dt, st),
                       'patchify')
        else:
            _lib.check(lib.ecgvit_patchify_transform(x.data_ptr(), _lib.ptr(mean), _lib.ptr(std), _lib.ptr(spans),
                                                     w.a_patch.data_ptr(), B, C, x.stride(1), L_in, n, P, dt, st),
                       'patchify_transform')
        self._select_patches(w)
        hook = m._before_layer_forward
        if hook is not None:
            hook(-1)   # embedding weights, cls, pos
        # e = a_emb @ We^T + be
        w_embed = wt['embed.w']
        if Kp != K:
            _lib.check(lib.ecgvit_pad_cols(w_embed.data_ptr(), w.embed_wpad.data_ptr(), d, K, Kp, dt, st), 'pad_cols')
            w_embed = w.embed_wpad
        self._gemm(B * w.n_vis, d, Kp, w.a_emb, Kp, 1, w_embed, Kp, 1, EPI_STORE, w.e, d, bias=pf['embed.b'])
        p_emb, p_blk = self._dropout_probs()
        w.p_emb, w.p_blk = p_emb, p_blk
        w.r_path = self._drop_path_rates()
        self._assemble(w)
        for l in range(c.num_hidden_layers):
            if hook is not None:
                hook(l)
            self._block_forward(l, w, record_attention=record_attention)
        if hook is not None:
            hook(c.num_hidden_layers)   # head
        return self._head_forward(w, labels, reduction)

    def _select_patches(self, w):
        """the rows of the patch matrix the encoder embeds (`w.a_emb`, `w.n_vis` per record): all of them here"""

    def _assemble(self, w):
        """token matrix x[0] = [cls | e] + pos (embedding dropout)"""
        m, lib, st = self.model, self.lib, self._stream
        pf = m._params_f32()
        seed_ptr = self.rng.data_ptr()
        _lib.check(lib.ecgvit_embed_assemble(w.e.data_ptr(), pf['cls'].data_ptr(), pf['pos'].data_ptr(),
                                             w.x[0].data_ptr(), w.B, w.n, m.config.hidden_size, w.p_emb, 0,
                                             seed_ptr if w.p_emb > 0 else None, m._res_code, st), 'embed_assemble')

    def _head_forward(self, w, labels, reduction):
        """CLS (or mean) pool + mlp_head + BCE: (loss | None, logits)"""
        m, lib, st = self.model, self.lib, self._stream
        c = m.config
        rdt = m._res_code
        pf = m._params_f32()
        B, N, d = w.B, w.N, c.hidden_size
        tok = w.x[c.num_hidden_layers]
        if m._mean_pool:
            # pool='mean': fp32 token means, then the CLS head over them as one fp32 token per record
            _lib.check(lib.ecgvit_token_mean(tok.data_ptr(), w.pooled.data_ptr(), B, N, d, rdt, st), 'token_mean')
            tok, N, rdt = w.pooled, 1, F32
        red = _lib.REDUCTION[reduction]
        loss_buf = None
        if labels is not None:
            assert labels.shape == (B, m.num_class)
            w.labels.copy_(labels, non_blocking=True)  # also casts (the reference passes float multi-hot)
            loss_buf = w.loss_none if reduction == 'none' else w.loss
        _lib.check(lib.ecgvit_head_fwd(
            tok.data_ptr(), pf['head.ln.w'].data_ptr(), pf['head.ln.b'].data_ptr(),
            pf['head.w'].data_ptr(), pf['head.b'].data_ptr(), w.labels.data_ptr() if labels is not None else None,
            *self._loss_weight_table(), w.xn.data_ptr(), w.hstat[0].data_ptr(), w.hstat[1].data_ptr(), w.logits.data_ptr(),
            _lib.ptr(loss_buf), B, N, d, m.num_class, red, LN_EPS, rdt, st), 'head_fwd')
        w.reduction = reduction
        loss = None
        if labels is not None:
            loss = w.loss_none if reduction == 'none' else w.loss[0]
        return loss, w.logits

    def _block_forward(self, l, s, record_attention=False, recompute=False):
        """block l of the stack s (the encoder's is the workspace itself): x[l] -> x[l + 1] (PreNorm attention +
        residual, PreNorm feed-forward + residual).
        recompute=True (activation checkpointing, from backward): rebuild what backward reads of the block -- ln1, qkv,
        lse, o, y, ln2, u, h -- from x[l]; the last Linear (whose output x[l + 1] is kept) is skipped.  Dropout masks are
        a function of (seed, site, element), so the recomputed tensors are bit-identical to the forward pass's."""
        m, lib, st = self.model, self.lib, self._stream
        dt, rdt = m._dtype_code, m._res_code
        epi_res = EPI_BIAS_RES_F32 if m._res_f32 else EPI_BIAS_RES
        d, mlp, H = s.d, s.mlp, s.H
        inner, dh = d, d // H
        B, N, M = s.B, s.N, s.M
        wt, pf = m._weights(), m._params_f32()
        p_blk = s.p_blk
        scale = float(dh) ** -0.5
        blk_seed = self.rng.data_ptr() if p_blk > 0 else None
        p = f'{s.prefix}{l}.'
        # dropout sites of block l: 1+4l attention probabilities, 2+4l after to_out, 3+4l after GELU, 4+4l after net[3]
        s_att, s_out, s_act, s_ff2 = 1 + 4 * l, 2 + 4 * l, 3 + 4 * l, 4 + 4 * l
        _lib.check(lib.ecgvit_layernorm_fwd(s.x[l].data_ptr(), pf[p + 'ln1.w'].data_ptr(), pf[p + 'ln1.b'].data_ptr(),
                                            s.ln1[l].data_ptr(), s.stat1[l][0].data_ptr(), s.stat1[l][1].data_ptr(),
                                            M, d, LN_EPS, rdt, st), 'layernorm_fwd')
        self._gemm(M, 3 * inner, d, s.ln1[l], d, 1, wt[p + 'qkv.w'], d, 1, EPI_STORE, s.qkv[l], 3 * inner)
        if record_attention:
            if l == 0:
                self.recorded_attention = torch.empty(B, s.depth, H, N, N, device=self.device, dtype=torch.float32)
            rec = self.recorded_attention
            _lib.check(lib.ecgvit_attention_probs(s.qkv[l].data_ptr(), rec[:, l].data_ptr(), B, N, H, dh, scale,
                                                  rec.stride(0), dt, st), 'attention_probs')
        _lib.check(lib.ecgvit_attention_fwd(s.qkv[l].data_ptr(), s.o[l].data_ptr(), s.lse[l].data_ptr(), B, N, H, dh,
                                            scale, p_blk, s_att, blk_seed, dt, st), 'attention_fwd')
        self._gemm(M, d, inner, s.o[l], inner, 1, wt[p + 'out.w'], inner, 1, epi_res, s.y[l], d,
                   aux=s.x[l], bias=pf[p + 'out.b'], drop=(p_blk, s_out), path=(s.r_path[l], s.path_site + 2 * l, N))
        _lib.check(lib.ecgvit_layernorm_fwd(s.y[l].data_ptr(), pf[p + 'ln2.w'].data_ptr(), pf[p + 'ln2.b'].data_ptr(),
                                            s.ln2[l].data_ptr(), s.stat2[l][0].data_ptr(), s.stat2[l][1].data_ptr(),
                                            M, d, LN_EPS, rdt, st), 'layernorm_fwd')
        self._gemm(M, mlp, d, s.ln2[l], d, 1, wt[p + 'ff1.w'], d, 1, EPI_BIAS_GELU, s.u[l], mlp,
                   out2=s.h[l], bias=pf[p + 'ff1.b'], drop=(p_blk, s_act))
        if not recompute:
            self._gemm(M, d, mlp, s.h[l], mlp, 1, wt[p + 'ff2.w'], mlp, 1, epi_res, s.x[l + 1], d,
                       aux=s.y[l], bias=pf[p + 'ff2.b'], drop=(p_blk, s_ff2),
                       path=(s.r_path[l], s.path_site + 2 * l + 1, N))

    def span_buffer(self, B):
        """device int32 [B, 2] (start, length) of the TimeOut span of every record; a persistent buffer, so a captured
        step reads whatever `set_spans` wrote last"""
        buf = self._spans.get(B)
        if buf is None:
            buf = self._spans[B] = torch.zeros(B, 2, device=self.device, dtype=torch.int32)
        return buf

    def set_spans(self, spans):
        """spans: int [B, 2] (host or device), see `InputPipeline.draw_spans`"""
        self.span_buffer(spans.shape[0]).copy_(spans.to(torch.int32), non_blocking=True)

    def _loss_weight_table(self):
        """(device pointer, length) of `EcgVit.loss_weight` (ecg_vit.py:144-147), or (None, 0) when unset; the table
        is re-uploaded only when the attribute changes (never inside a captured step)"""
        lw = self.model.loss_weight
        if not lw:
            return None, 0
        key = tuple(float(v) for v in lw)
        if self._lw_key != key:
            self._lw_table = torch.tensor(key, dtype=torch.float32, device=self.device)
            self._lw_key = key
        return self._lw_table.data_ptr(), len(key)

    # ---- backward --------------------------------------------------------------------------------
    def backward(self, grad_scale=1.0, zero_grads=True, grad_scale_dev=None):
        """Gradients of the last forward's loss w.r.t. every parameter, accumulated into the flat grad buffer.
        grad_scale_dev: optional fp32 CUDA scalar multiplied into the upstream gradient on the device (no host sync)."""
        m, lib, st = self.model, self.lib, self._stream
        c = m.config
        w = self._cur
        assert w is not None, 'backward before forward'
        assert w.reduction in ('mean', 'sum'), "backward needs loss_reduction 'mean' or 'sum'"
        B, d = w.B, c.hidden_size
        depth = c.num_hidden_layers
        gr = m._grads_f32()
        if zero_grads:
            m._flat_g.zero_()
        last = f'l{depth - 1}.'
        top = (depth - 1) & 1
        # with dropout or drop path between net[3] / to_out[0] and the residual add, the Linear sees s * mask * dz / (1 - p):
        # its operand and its bias gradient come from the masked copy, so the producers must not pre-sum the unmasked
        # gradient
        self._head_backward(w, w.dz[top], None if self._masked(w, depth - 1) else gr[last + 'ff2.b'], grad_scale,
                            grad_scale_dev)
        self._stack_backward(w)
        dz = w.dz[(-1) & 1]   # gradient w.r.t. the token matrix (input of block 0)
        # ---- embedding: tok = [cls | a_emb We^T + be] + pos
        self._assemble_backward(w, dz)
        rows = B * w.n_vis
        if w.Kp == w.K:
            self._gemm(d, w.K, rows, w.de, d, 0, w.a_emb, w.K, 0, EPI_ATOMIC_F32, gr['embed.w'], w.K, split_k=0)
        else:
            w.embed_gpad.zero_()
            self._gemm(d, w.Kp, rows, w.de, d, 0, w.a_emb, w.Kp, 0, EPI_ATOMIC_F32, w.embed_gpad, w.Kp, split_k=0)
            _lib.check(lib.ecgvit_unpad_add_f32(w.embed_gpad.data_ptr(), gr['embed.w'].data_ptr(), d, w.K, w.Kp, st),
                       'unpad_add')
        if m._after_layer_backward is not None:
            m._after_layer_backward(-1)

    @staticmethod
    def _masked(s, l):
        """whether the residual branches of block l of stack s are masked (element dropout or drop path): their
        Linears then read a masked copy of the residual-stream gradient"""
        return s.p_blk > 0 or s.r_path[l] > 0

    def _stack_backward(self, s):
        """backward through the blocks of the stack s, from the gradient of its output in s.dz[(depth - 1) & 1] (its
        column sum already added to the top ff2 bias gradient when the top block is not masked) to that of its input in
        s.dz[1]; the weight gradients run on the side stream, which is joined at the end"""
        m, lib, st = self.model, self.lib, self._stream
        dt = m._dtype_code
        rdt = m._res_code
        M, d, mlp, H = s.M, s.d, s.mlp, s.H
        B, N = s.B, s.N
        inner, dh = d, d // H
        depth = s.depth
        wt, pf, gr = m._weights(), m._params_f32(), m._grads_f32()
        p_blk = s.p_blk
        seed_ptr = self.rng.data_ptr()
        blk_seed = seed_ptr if p_blk > 0 else None
        last = f'{s.prefix}{depth - 1}.'
        top = (depth - 1) & 1
        scale = float(dh) ** -0.5

        main, side = torch.cuda.current_stream(), self.side_stream

        def wgrad(*args, **kw):
            """weight-gradient GEMM on the side stream, ordered after everything issued so far on the main stream;
            returns the event that marks its completion (None when there is no side stream)"""
            if side is None:
                self._gemm(*args, **kw)
                return None
            ready = torch.cuda.Event()
            ready.record(main)
            side.wait_event(ready)
            with torch.cuda.stream(side):
                self._gemm(*args, **kw)
                done = torch.cuda.Event()
                done.record(side)
            return done

        def before_overwrite(ev):
            """the main stream may not overwrite a scratch buffer that a side-stream GEMM is still reading"""
            if ev is not None:
                main.wait_event(ev)

        ev_fold = [None, None]

        def layernorm_bwd(which, dln, x_in, gamma, stat, dres, dx, dgamma, dbeta, dcol, dxm, p_drop, site,
                          r_path=0.0, path_site=0):
            """dx = dres + LN'(dln) (+ the masked copy dxm: dropout p_drop at `site`, drop path r_path at `path_site`) on
            the main stream; the fold of the per-CTA partial rows into dgamma / dbeta / dcol feeds nothing in the chain and
            runs on the side stream"""
            scr = s.ln_scratch[which]
            before_overwrite(ev_fold[which])  # the fold of this scratch's previous user
            seed = seed_ptr if (dxm is not None and (p_drop > 0 or r_path > 0)) else None
            args = (dln.data_ptr(), x_in.data_ptr(), gamma.data_ptr(), stat[0].data_ptr(), stat[1].data_ptr(),
                    dres.data_ptr(), dx.data_ptr(), dgamma.data_ptr(), dbeta.data_ptr(), _lib.ptr(dcol), scr.data_ptr(),
                    _lib.ptr(dxm), p_drop, site, seed, M, d, 0 if side is None else 1, rdt)
            what = 'layernorm_bwd' if side is None else 'layernorm_bwd_partial'
            if r_path > 0:
                _lib.check(lib.ecgvit_layernorm_bwd_drop_path(*args, r_path, path_site, N, st), what)
            else:
                _lib.check(lib.ecgvit_layernorm_bwd(*args, st), what)
            if side is not None:
                ready = torch.cuda.Event()
                ready.record(main)
                side.wait_event(ready)
                with torch.cuda.stream(side):
                    _lib.check(lib.ecgvit_layernorm_bwd_finalize(scr.data_ptr(), dgamma.data_ptr(), dbeta.data_ptr(),
                                                                 _lib.ptr(dcol), M, d, side.cuda_stream),
                               'layernorm_bwd_finalize')
                    ev_fold[which] = torch.cuda.Event()
                    ev_fold[which].record(side)

        # side-stream events per layer: ev[l] = {'ff2', 'ff1', 'out', 'qkv'} -> completion of that weight gradient
        evs = {}
        if self._masked(s, depth - 1):
            # the top block's input gradient comes from the head, not from a LayerNorm': mask it here
            args = (s.dz[top].data_ptr(), s.dzm[0][top].data_ptr(), gr[last + 'ff2.b'].data_ptr(), M, d, d, p_blk,
                    4 * depth, seed_ptr, dt)
            r_top = s.r_path[depth - 1]
            if r_top > 0:
                _lib.check(lib.ecgvit_dropout_bwd_copy_drop_path(*args, r_top, s.path_site + 2 * (depth - 1) + 1, N, st),
                           'dropout_bwd_copy')
            else:
                _lib.check(lib.ecgvit_dropout_bwd_copy(*args, st), 'dropout_bwd_copy')
        for l in range(depth - 1, -1, -1):
            p = f'{s.prefix}{l}.'
            q, qn = l & 1, (l - 1) & 1      # buffer parity of this layer / of the layer below
            s_att, s_out, s_act, s_ff2 = 1 + 4 * l, 2 + 4 * l, 3 + 4 * l, 4 + 4 * l
            old = evs.pop(l + 2, {})        # the previous users of this parity's buffers (a whole layer ago)
            if s.ckpt and l < depth - 2:
                # the activation set of layer l was last used by layer l + 2: its weight gradients must have read it
                for ev in old.values():
                    before_overwrite(ev)
                self._block_forward(l, s, recompute=True)
            e = evs.setdefault(l, {})
            dz, dy, du, dqkv = s.dz[q], s.dy[q], s.du[q], s.dqkv[q]
            masked, r_l = self._masked(s, l), s.r_path[l]
            dzl = s.dzm[0][q] if masked else dz      # what net[3] saw: s * mask * dz / (1 - p)
            # ---- feed-forward branch: x[l+1] = y + drop(W2 drop(gelu(W1 ln2(y) + b1)) + b2)
            e['ff2'] = wgrad(d, mlp, M, dzl, d, 0, s.h[l], mlp, 0, EPI_ATOMIC_F32, gr[p + 'ff2.w'], mlp, split_k=0)
            before_overwrite(old.get('ff1'))   # du of this parity
            self._gemm(M, mlp, d, dzl, d, 1, wt[p + 'ff2.w'], mlp, 0, EPI_DGELU, du, mlp, aux=s.u[l], drop=(p_blk, s_act))
            # FF1's bias gradient (column sums of du) feeds nothing in the chain: it rides on the side stream in front of
            # FF1's weight gradient (same operand, so the event that guards `du` covers both)
            if side is None:
                _lib.check(lib.ecgvit_colsum(du.data_ptr(), gr[p + 'ff1.b'].data_ptr(), M, mlp, mlp, dt, st), 'colsum')
            else:
                ready = torch.cuda.Event()
                ready.record(main)
                side.wait_event(ready)
                with torch.cuda.stream(side):
                    _lib.check(lib.ecgvit_colsum(du.data_ptr(), gr[p + 'ff1.b'].data_ptr(), M, mlp, mlp, dt,
                                                 side.cuda_stream), 'colsum')
            e['ff1'] = wgrad(mlp, d, M, du, mlp, 0, s.ln2[l], d, 0, EPI_ATOMIC_F32, gr[p + 'ff1.w'], d, split_k=0)
            self._gemm(M, d, mlp, du, mlp, 1, wt[p + 'ff1.w'], d, 0, EPI_STORE, s.dln, d)
            before_overwrite(old.get('out'))   # dy / its masked copy of this parity
            dyl = s.dzm[1][q] if masked else dy
            layernorm_bwd(0, s.dln, s.y[l], pf[p + 'ln2.w'], s.stat2[l], dz, dy, gr[p + 'ln2.w'], gr[p + 'ln2.b'],
                          gr[p + 'out.b'], dyl if masked else None, p_blk, s_out, r_l, s.path_site + 2 * l)
            # ---- attention branch: y = x + s * drop(Wo attn(Wqkv ln1(x)) + bo); dyl = s * mask * dy / (1 - p)
            e['out'] = wgrad(d, inner, M, dyl, d, 0, s.o[l], inner, 0, EPI_ATOMIC_F32, gr[p + 'out.w'], inner, split_k=0)
            self._gemm(M, inner, d, dyl, d, 1, wt[p + 'out.w'], inner, 0, EPI_STORE, s.d_o, inner)
            before_overwrite(old.get('qkv'))   # dqkv of this parity
            _lib.check(lib.ecgvit_attention_bwd(s.qkv[l].data_ptr(), s.o[l].data_ptr(), s.d_o.data_ptr(),
                                                s.lse[l].data_ptr(), dqkv.data_ptr(), _lib.ptr(s.attn_scratch), B, N,
                                                H, dh, scale, p_blk, s_att, blk_seed, dt, st),
                       'attention_bwd' if s.attn_scratch is None else 'attention_bwd_flash')
            e['qkv'] = wgrad(3 * inner, d, M, dqkv, 3 * inner, 0, s.ln1[l], d, 0, EPI_ATOMIC_F32, gr[p + 'qkv.w'], d,
                             split_k=0)
            self._gemm(M, d, 3 * inner, dqkv, 3 * inner, 1, wt[p + 'qkv.w'], d, 0, EPI_STORE, s.dln, d)
            below_bias = gr[f'{s.prefix}{l - 1}.ff2.b'] if l > 0 else None
            drop_below = l > 0 and self._masked(s, l - 1)
            r_below = s.r_path[l - 1] if l > 0 else 0.0
            # LayerNorm' writes the input gradient of layer l - 1 into the OTHER parity, last read by the ff2 weight
            # gradient of layer l + 1
            before_overwrite(evs.get(l + 1, {}).get('ff2'))
            layernorm_bwd(1, s.dln, s.x[l], pf[p + 'ln1.w'], s.stat1[l], dy, s.dz[qn], gr[p + 'ln1.w'], gr[p + 'ln1.b'],
                          below_bias, s.dzm[0][qn] if drop_below else None, p_blk if drop_below else 0.0, s_ff2 - 4,
                          r_below if drop_below else 0.0, s.path_site + 2 * (l - 1) + 1)
            if s.hooks and m._after_layer_backward is not None:
                # the gradient bucket of layer l is complete once its side-stream wgrads AND everything the main stream
                # has issued so far (LayerNorm / bias gradients) are done.  The collective is therefore issued from the
                # side stream after it has waited for the main stream's current point: c10d orders the NCCL kernel
                # after the issuing stream, and the main chain never waits for the weight-gradient GEMMs.
                if side is None:
                    m._after_layer_backward(l)
                else:
                    here = torch.cuda.Event()
                    here.record(main)
                    side.wait_event(here)
                    with torch.cuda.stream(side):
                        m._after_layer_backward(l)
        for e in evs.values():
            for ev in e.values():
                before_overwrite(ev)  # join the side stream
        for ev in ev_fold:
            before_overwrite(ev)

    def _head_backward(self, w, dtok, dcolsum, grad_scale, grad_scale_dev):
        """backward of `_head_forward`: writes the whole token-shaped gradient `dtok` of the encoder output and adds its
        column sum into `dcolsum` (the top block's ff2 bias gradient, when not None)"""
        m, lib, st = self.model, self.lib, self._stream
        c = m.config
        pf, gr = m._params_f32(), m._grads_f32()
        tok, dhead, N, rdt = w.x[c.num_hidden_layers], dtok, w.N, m._res_code
        if m._mean_pool:
            # the head's backward over the pooled rows writes the fp32 pooled gradient, and its dcolsum
            # sum_b dpool[b] is already the column sum of the broadcast gradient below
            tok, dhead, N, rdt = w.pooled, w.dpool, 1, F32
        _lib.check(lib.ecgvit_head_bwd(
            tok.data_ptr(), pf['head.ln.w'].data_ptr(), pf['head.w'].data_ptr(), w.labels.data_ptr(),
            *self._loss_weight_table(), w.xn.data_ptr(), w.hstat[0].data_ptr(), w.hstat[1].data_ptr(), w.logits.data_ptr(),
            dhead.data_ptr(),
            gr['head.w'].data_ptr(), gr['head.b'].data_ptr(), gr['head.ln.w'].data_ptr(), gr['head.ln.b'].data_ptr(),
            _lib.ptr(dcolsum), w.head_scratch.data_ptr(), w.B, N, c.hidden_size, m.num_class,
            _lib.REDUCTION[w.reduction], float(grad_scale), _lib.ptr(grad_scale_dev), rdt, st), 'head_bwd')
        if m._mean_pool:
            _lib.check(lib.ecgvit_token_mean_bwd(w.dpool.data_ptr(), dtok.data_ptr(), w.B, w.N, c.hidden_size,
                                                 m._dtype_code, st), 'token_mean_bwd')

    def _assemble_backward(self, w, dz):
        """backward of `_assemble`: de, and the cls / pos / embedding-bias gradients"""
        m, lib, st = self.model, self.lib, self._stream
        gr = m._grads_f32()
        p_emb = w.p_emb
        _lib.check(lib.ecgvit_embed_assemble_bwd(dz.data_ptr(), w.de.data_ptr(), gr['cls'].data_ptr(),
                                                 gr['pos'].data_ptr(), gr['embed.b'].data_ptr(), w.B, w.n,
                                                 m.config.hidden_size, p_emb, 0,
                                                 self.rng.data_ptr() if p_emb > 0 else None, m._dtype_code, st),
                   'embed_assemble_bwd')


class MaskedPatchEngine(StepEngine):
    """StepEngine of `EcgVitForMaskedPatchModeling`: the same encoder sequence; the token assembly puts the learned
    mask token on the masked patches and the head is the reconstruction objective

        pred = LN_r(z[:, 1:]) Wr^T + br;  loss = sum over masked patches of (pred - a_patch)^2 / (n_masked * K)

    Forward: mask draw (or count of the caller's mask) -> masked assembly -> blocks -> patch-row LayerNorm -> one GEMM
    whose epilogue writes r = pred - a_patch and fp32 row partials of r^2 -> one-CTA loss fold.  Backward: dpred =
    upstream * 2 * mask * r / (count * K) -> recon weight / bias gradients -> dgrad -> patch-row LayerNorm' into the
    top block's gradient.  With per-lead tokens (K = P not a multiple of 8) the recon weight rows and bias are padded
    to Kp like the embedding weight; the padded target columns are zero, so they add nothing to the loss."""

    EVAL_SEED = 0x5EED5   # mask seed in eval mode: the same batch always gets the same mask

    def __init__(self, model):
        super().__init__(model)
        self._eval_seed = torch.tensor([self.EVAL_SEED, 0], device=self.device, dtype=torch.int32)
        self._user_mask = None

    @property
    def mask_site(self):
        """counter-hash site of the mask keys: the dropout sites are 0 .. 4 * depth"""
        return 4 * self.model.config.num_hidden_layers + 1

    def workspace(self, B, L, n_vis=None):
        w = super().workspace(B, L, n_vis)
        if hasattr(w, 'mask'):
            return w
        m = self.model
        d = m.recon_head[0].normalized_shape[0]   # width of the token matrix the head reads
        T = m._act_dtype
        rows, K, Kp = B * w.n, w.K, w.Kp
        dev = self.device
        w.mask = torch.zeros(rows, device=dev, dtype=torch.uint8)
        w.counts = torch.zeros(B, device=dev, dtype=torch.int32)
        w.ln_r = torch.empty(rows, d, device=dev, dtype=T)
        w.rstat = torch.empty(2, rows, device=dev, dtype=torch.float32)
        w.r = torch.empty(rows, Kp, device=dev, dtype=T)        # pred - target
        w.dpred = torch.empty(rows, Kp, device=dev, dtype=T)
        w.n_groups = (Kp + 63) // 64
        w.rowsq = torch.empty(w.n_groups, rows, device=dev, dtype=torch.float32)
        w.mloss = torch.zeros(1, device=dev, dtype=torch.float32)
        w.mcount = torch.zeros(1, device=dev, dtype=torch.float32)
        w.dln_r = torch.empty(rows, d, device=dev, dtype=T)
        if Kp != K:
            w.recon_wpad = torch.zeros(Kp, d, device=dev, dtype=T)
            w.recon_bpad = torch.zeros(Kp, device=dev, dtype=torch.float32)
            w.recon_gpad = torch.zeros(Kp * d + Kp, device=dev, dtype=torch.float32)
        return w

    def forward(self, sample_values, labels=None, reduction='mean', record_attention=False, bool_masked_pos=None):
        """(loss, None); the loss is a view of a workspace buffer.  bool_masked_pos: optional bool [B, n_patch] (any
        number of masked patches per record); drawn on the device when None (see `_assemble`)."""
        assert labels is None, 'masked-patch pre-training takes no labels'
        assert reduction == 'mean', "the masked-patch loss is a mean ('mean' reduction only)"
        self._user_mask = bool_masked_pos
        try:
            return super().forward(sample_values, None, reduction, record_attention)
        finally:
            self._user_mask = None

    def _draw_mask(self, w):
        """w.mask / w.counts: the caller's mask, or round(mask_ratio * n) patches per record drawn on the device"""
        m, lib, st = self.model, self.lib, self._stream
        B, n = w.B, w.n
        user = self._user_mask
        if user is not None:
            assert tuple(user.shape) == (B, n), f'bool_masked_pos must be [{B}, {n}], got {tuple(user.shape)}'
            w.mask.view(B, n).copy_(user, non_blocking=True)
            seed = None
        else:
            k = int(round(m.mask_ratio * n))
            # training: the step's device seed (refreshed per forward, read at replay by a captured graph); eval: fixed
            seed = (self.rng if m.training else self._eval_seed).data_ptr()
        _lib.check(lib.ecgvit_mpm_mask(seed, B, n, k if user is None else 0, self.mask_site, w.mask.data_ptr(),
                                       w.counts.data_ptr(), st), 'mpm_mask')

    def _assemble(self, w):
        m, lib, st = self.model, self.lib, self._stream
        pf = m._params_f32()
        B, n = w.B, w.n
        self._draw_mask(w)
        _lib.check(lib.ecgvit_embed_assemble_masked(
            w.e.data_ptr(), pf['cls'].data_ptr(), pf['pos'].data_ptr(), pf['mask'].data_ptr(), w.mask.data_ptr(),
            w.x[0].data_ptr(), B, n, m.config.hidden_size, w.p_emb, 0, self.rng.data_ptr() if w.p_emb > 0 else None,
            m._res_code, st), 'embed_assemble_masked')

    def _recon_params(self, w):
        """(weight, bias) operands of the recon GEMM: padded to Kp rows in per-lead mode"""
        m = self.model
        wt, pf = m._weights(), m._params_f32()
        if w.Kp == w.K:
            return wt['recon.w'], pf['recon.b']
        return w.recon_wpad, w.recon_bpad

    def _head_stack(self, w):
        """the block stack whose output the reconstruction head reads: the encoder"""
        return w

    def _head_forward(self, w, labels, reduction):
        m, lib, st = self.model, self.lib, self._stream
        hs = self._head_stack(w)
        d = hs.d
        pf, wt = m._params_f32(), m._weights()
        B, n, K, Kp = w.B, w.n, w.K, w.Kp
        rows = B * n
        if Kp != K:
            # rows K..Kp-1 of the padded copies stay zero (allocation)
            _lib.check(lib.ecgvit_pad_cols(wt['recon.w'].data_ptr(), w.recon_wpad.data_ptr(), 1, K * d, Kp * d,
                                           m._dtype_code, st), 'pad_cols')
            _lib.check(lib.ecgvit_pad_cols(pf['recon.b'].data_ptr(), w.recon_bpad.data_ptr(), 1, K, Kp, _lib.F32, st),
                       'pad_cols')
        w_r, b_r = self._recon_params(w)
        _lib.check(lib.ecgvit_layernorm_patch_fwd(
            hs.x[hs.depth].data_ptr(), pf['recon.ln.w'].data_ptr(), pf['recon.ln.b'].data_ptr(),
            w.ln_r.data_ptr(), w.rstat[0].data_ptr(), w.rstat[1].data_ptr(), B, n, d, LN_EPS, m._res_code, st),
            'layernorm_patch_fwd')
        self._gemm(rows, Kp, d, w.ln_r, d, 1, w_r, d, 1, EPI_BIAS_SUB_ROWSQ, w.r, Kp, out2=w.rowsq, aux=w.a_patch,
                   bias=b_r)
        _lib.check(lib.ecgvit_mpm_loss(w.rowsq.data_ptr(), w.n_groups, w.mask.data_ptr(), w.counts.data_ptr(), B, n, K,
                                       w.mloss.data_ptr(), w.mcount.data_ptr(), st), 'mpm_loss')
        w.reduction = reduction
        return w.mloss[0], None

    def reconstruction(self):
        """fp32 [B, n_patch, K] prediction of the last forward (patch-matrix feature order)"""
        w = self._cur
        out = torch.empty(w.B, w.n, w.K, device=self.device, dtype=torch.float32)
        _lib.check(self.lib.ecgvit_mpm_reconstruction(w.r.data_ptr(), w.a_patch.data_ptr(), out.data_ptr(), w.B * w.n,
                                                      w.Kp, w.K, self.model._dtype_code, self._stream),
                   'mpm_reconstruction')
        return out

    def mask(self):
        """bool [B, n_patch] mask of the last forward (a copy)"""
        w = self._cur
        return w.mask.view(w.B, w.n).bool()

    def _head_backward(self, w, dtok, dcolsum, grad_scale, grad_scale_dev):
        m, lib, st = self.model, self.lib, self._stream
        hs = self._head_stack(w)
        d = hs.d
        dt = m._dtype_code
        pf, gr = m._params_f32(), m._grads_f32()
        B, n, K, Kp = w.B, w.n, w.K, w.Kp
        rows = B * n
        _lib.check(lib.ecgvit_mpm_dpred(w.r.data_ptr(), w.mask.data_ptr(), w.mcount.data_ptr(), rows, Kp, K,
                                        float(grad_scale), _lib.ptr(grad_scale_dev), w.dpred.data_ptr(), dt, st),
                   'mpm_dpred')
        # recon weight gradient dWr = dpred^T ln_r (split-K) and bias gradient colsum(dpred)
        if Kp == K:
            self._gemm(Kp, d, rows, w.dpred, Kp, 0, w.ln_r, d, 0, EPI_ATOMIC_F32, gr['recon.w'], d, split_k=0)
            _lib.check(lib.ecgvit_colsum(w.dpred.data_ptr(), gr['recon.b'].data_ptr(), rows, K, Kp, dt, st), 'colsum')
        else:
            w.recon_gpad.zero_()
            gw, gb = w.recon_gpad[:Kp * d], w.recon_gpad[Kp * d:]
            self._gemm(Kp, d, rows, w.dpred, Kp, 0, w.ln_r, d, 0, EPI_ATOMIC_F32, gw, d, split_k=0)
            _lib.check(lib.ecgvit_colsum(w.dpred.data_ptr(), gb.data_ptr(), rows, Kp, Kp, dt, st), 'colsum')
            _lib.check(lib.ecgvit_unpad_add_f32(gw.data_ptr(), gr['recon.w'].data_ptr(), 1, K * d, Kp * d, st),
                       'unpad_add')
            _lib.check(lib.ecgvit_unpad_add_f32(gb.data_ptr(), gr['recon.b'].data_ptr(), 1, K, Kp, st), 'unpad_add')
        w_r, _ = self._recon_params(w)
        self._gemm(rows, d, Kp, w.dpred, Kp, 1, w_r, d, 0, EPI_STORE, w.dln_r, d)
        _lib.check(lib.ecgvit_layernorm_patch_bwd(
            w.dln_r.data_ptr(), hs.x[hs.depth].data_ptr(), pf['recon.ln.w'].data_ptr(), w.rstat[0].data_ptr(),
            w.rstat[1].data_ptr(), dtok.data_ptr(), gr['recon.ln.w'].data_ptr(), gr['recon.ln.b'].data_ptr(),
            _lib.ptr(dcolsum), hs.ln_scratch[0].data_ptr(), B, n, d, m._res_code, st), 'layernorm_patch_bwd')

    def _assemble_backward(self, w, dz):
        m, lib, st = self.model, self.lib, self._stream
        gr = m._grads_f32()
        p_emb = w.p_emb
        _lib.check(lib.ecgvit_embed_assemble_masked_bwd(
            dz.data_ptr(), w.mask.data_ptr(), w.de.data_ptr(), gr['cls'].data_ptr(), gr['pos'].data_ptr(),
            gr['embed.b'].data_ptr(), gr['mask'].data_ptr(), w.B, w.n, m.config.hidden_size, p_emb, 0,
            self.rng.data_ptr() if p_emb > 0 else None, m._dtype_code, st), 'embed_assemble_masked_bwd')


class MaskedAutoencoderEngine(MaskedPatchEngine):
    """StepEngine of `EcgVitForMaskedAutoencoding` (MAE): the encoder sees only the n_vis visible patches of every
    record; a second, narrower block stack (the decoder, keys `dec{i}.`) runs over all n + 1 positions and the head and
    loss are `MaskedPatchEngine`'s, at the decoder's width.

    Forward: patchify -> mask draw -> index build (vis_idx [B, n_vis], slot [B, n]) -> row gather of the visible patch
    rows -> embedding GEMM on B * n_vis rows -> visible assemble (pos at the patches' positions) -> encoder blocks over
    n_vis + 1 tokens -> LayerNorm + decoder embedding GEMM -> unshuffle (mask token at the masked positions, + decoder pos)
    -> decoder blocks over n + 1 tokens -> reconstruction head.  Backward runs the same path in reverse."""

    def workspace(self, B, L, n_vis=None):
        m = self.model
        c = m.config
        if n_vis is None:
            n = L // c.patch_size * (c.num_channels if getattr(c, 'per_lead_tokens', False) else 1)
            k = self._user_k if self._user_mask is not None else int(round(m.mask_ratio * n))
            n_vis = n - k
        w = super().workspace(B, L, n_vis)
        if hasattr(w, 'dec'):
            return w
        dev, T = self.device, m._act_dtype
        d, dd = c.hidden_size, m.decoder_hidden_size
        n, nv, Kp, M = w.n, w.n_vis, w.Kp, w.M
        w.vis_idx = torch.empty(B, nv, device=dev, dtype=torch.int32)
        w.slot = torch.empty(B, n, device=dev, dtype=torch.int32)
        w.a_vis = torch.empty(B * nv, Kp, device=dev, dtype=T)
        w.a_emb = w.a_vis
        w.ln_t = torch.empty(M, d, device=dev, dtype=T)            # decoder.norm(encoder output)
        w.stat_t = torch.empty(2, M, device=dev, dtype=torch.float32)
        w.t = torch.empty(M, dd, device=dev, dtype=T)              # decoder.embed(ln_t)
        w.dt = torch.empty(M, dd, device=dev, dtype=T)
        w.dln_t = torch.empty(M, d, device=dev, dtype=T)
        # per-position partial sums of the two deterministic backward folds (used one after the other)
        w.pos_scratch = torch.empty(n * max(d, dd), device=dev, dtype=torch.float32)
        w.dec = _Workspace()
        self._alloc_stack(w.dec, 'dec', B, n + 1, dd, m.decoder_intermediate_size, m.decoder_num_attention_heads,
                          m.decoder_num_hidden_layers, False)
        return w

    def forward(self, sample_values, labels=None, reduction='mean', record_attention=False, bool_masked_pos=None):
        # the caller's mask sets the encoder's token count: its per-record count (equal in every record, checked by the
        # model) is read on the host
        self._user_k = None if bool_masked_pos is None else int(bool_masked_pos[0].sum())
        return super().forward(sample_values, labels, reduction, record_attention, bool_masked_pos)

    def _select_patches(self, w):
        lib, st = self.lib, self._stream
        self._draw_mask(w)
        _lib.check(lib.ecgvit_mae_index(w.mask.data_ptr(), w.B, w.n, w.n_vis, w.vis_idx.data_ptr(), w.slot.data_ptr(),
                                        st), 'mae_index')
        _lib.check(lib.ecgvit_row_gather(w.a_patch.data_ptr(), w.a_vis.data_ptr(), w.vis_idx.data_ptr(), w.B, w.n,
                                         w.n_vis, w.Kp, self.model._dtype_code, st), 'row_gather')

    def _assemble(self, w):
        m, lib, st = self.model, self.lib, self._stream
        pf = m._params_f32()
        _lib.check(lib.ecgvit_embed_assemble_visible(
            w.e.data_ptr(), pf['cls'].data_ptr(), pf['pos'].data_ptr(), w.vis_idx.data_ptr(), w.x[0].data_ptr(), w.B,
            w.n_vis, m.config.hidden_size, w.p_emb, 0, self.rng.data_ptr() if w.p_emb > 0 else None, m._res_code, st),
            'embed_assemble_visible')

    def _head_stack(self, w):
        return w.dec

    def _head_forward(self, w, labels, reduction):
        m, lib, st = self.model, self.lib, self._stream
        c = m.config
        pf, wt = m._params_f32(), m._weights()
        d, dec = c.hidden_size, w.dec
        _lib.check(lib.ecgvit_layernorm_fwd(w.x[c.num_hidden_layers].data_ptr(), pf['dec.ln.w'].data_ptr(),
                                            pf['dec.ln.b'].data_ptr(), w.ln_t.data_ptr(), w.stat_t[0].data_ptr(),
                                            w.stat_t[1].data_ptr(), w.M, d, LN_EPS, m._res_code, st), 'layernorm_fwd')
        self._gemm(w.M, dec.d, d, w.ln_t, d, 1, wt['dec.embed.w'], d, 1, EPI_STORE, w.t, dec.d, bias=pf['dec.embed.b'])
        _lib.check(lib.ecgvit_mae_unshuffle(w.t.data_ptr(), pf['dec.mask'].data_ptr(), pf['dec.pos'].data_ptr(),
                                            w.slot.data_ptr(), dec.x[0].data_ptr(), w.B, w.n, w.n_vis, dec.d,
                                            m._res_code, st), 'mae_unshuffle')
        for l in range(dec.depth):
            self._block_forward(l, dec)
        return super()._head_forward(w, labels, reduction)

    def _head_backward(self, w, dtok, dcolsum, grad_scale, grad_scale_dev):
        m, lib, st = self.model, self.lib, self._stream
        c = m.config
        dt = m._dtype_code
        wt, pf, gr = m._weights(), m._params_f32(), m._grads_f32()
        d, dec, M = c.hidden_size, w.dec, w.M
        super()._head_backward(w, dec.dz[(dec.depth - 1) & 1], gr[f'dec{dec.depth - 1}.ff2.b'], grad_scale,
                               grad_scale_dev)
        self._stack_backward(dec)
        _lib.check(lib.ecgvit_mae_unshuffle_bwd(dec.dz[1].data_ptr(), w.slot.data_ptr(), w.dt.data_ptr(),
                                                gr['dec.pos'].data_ptr(), gr['dec.mask'].data_ptr(),
                                                w.pos_scratch.data_ptr(), w.B, w.n, w.n_vis, dec.d, dt, st),
                   'mae_unshuffle_bwd')
        # decoder.embed: weight gradient dt^T ln_t, bias gradient colsum(dt), input gradient dt We
        self._gemm(dec.d, d, M, w.dt, dec.d, 0, w.ln_t, d, 0, EPI_ATOMIC_F32, gr['dec.embed.w'], d, split_k=0)
        _lib.check(lib.ecgvit_colsum(w.dt.data_ptr(), gr['dec.embed.b'].data_ptr(), M, dec.d, dec.d, dt, st), 'colsum')
        self._gemm(M, d, dec.d, w.dt, dec.d, 1, wt['dec.embed.w'], d, 0, EPI_STORE, w.dln_t, d)
        # decoder.norm': the whole gradient of the encoder output (no residual term), its column sum into the top block's
        # ff2 bias gradient when that block has no dropout
        _lib.check(lib.ecgvit_layernorm_bwd(
            w.dln_t.data_ptr(), w.x[c.num_hidden_layers].data_ptr(), pf['dec.ln.w'].data_ptr(), w.stat_t[0].data_ptr(),
            w.stat_t[1].data_ptr(), None, dtok.data_ptr(), gr['dec.ln.w'].data_ptr(), gr['dec.ln.b'].data_ptr(),
            _lib.ptr(dcolsum), w.ln_scratch[0].data_ptr(), None, 0.0, 0, None, M, d, 0, m._res_code, st),
            'layernorm_bwd')

    def _assemble_backward(self, w, dz):
        m, lib, st = self.model, self.lib, self._stream
        gr = m._grads_f32()
        _lib.check(lib.ecgvit_embed_assemble_visible_bwd(
            dz.data_ptr(), w.slot.data_ptr(), w.de.data_ptr(), gr['cls'].data_ptr(), gr['pos'].data_ptr(),
            gr['embed.b'].data_ptr(), w.pos_scratch.data_ptr(), w.B, w.n, w.n_vis, m.config.hidden_size, w.p_emb, 0,
            self.rng.data_ptr() if w.p_emb > 0 else None, m._dtype_code, st), 'embed_assemble_visible_bwd')
